"""Deterministic synthetic inputs for the distillation-loss hot path (SURVEY.md §8d).

Everything is drawn on the CPU from `torch.Generator().manual_seed(...)` so the
same tensors can be rebuilt on any box of this image; callers move them to the
GPU.  Shapes follow the reference's DeiT-Tiny student / DeiT-Small-distilled
teacher: student block MLP outputs [B,197,192] (CLS at 0), teacher [B,198,384]
(CLS, DIST at 0,1) — /root/reference/model/models.py:181-199.
"""
from __future__ import annotations

import torch
import torch.nn as nn

STUDENT_TOKENS, STUDENT_DIM = 197, 192
TEACHER_TOKENS, TEACHER_DIM = 198, 384
NUM_LAYERS = 12


def default_args(**kw):
    """Loss-relevant argparse defaults of the reference CLI (tools/train.py:103-136,157-186)."""
    from types import SimpleNamespace
    d = dict(lrkd_rank=32, lrkd_alpha=0.1, lrkd_beta=0.1, lrkd_gamma=0.1, saliency_method=1,
             saliency_mask_ratio=0.5, wasskd_type="l1", mgd_alpha=7e-5, mgd_mask_ratio=0.5,
             mixup=0.8, cutmix=1.0, cutmix_minmax=None, smoothing=0.1, current_epoch=0,
             distillation_type="none")
    d.update(kw)
    return SimpleNamespace(**d)


def _gen(seed: int) -> torch.Generator:
    return torch.Generator().manual_seed(seed)


def make_logits(B: int, C: int, seed: int = 1234, int_labels: bool = False):
    """(outputs, outputs_kd, teacher_logits, labels): N(0,1) logits; labels = softmax(N(0,1)) rows
    (mixup-like, sum to 1) or int64 class ids."""
    g = _gen(seed)
    outputs = torch.randn(B, C, generator=g)
    outputs_kd = torch.randn(B, C, generator=g)
    teacher_logits = torch.randn(B, C, generator=g)
    if int_labels:
        labels = torch.randint(0, C, (B,), generator=g)
    else:
        labels = torch.softmax(torch.randn(B, C, generator=g), dim=-1)
    return outputs, outputs_kd, teacher_logits, labels


def make_features(B: int, seed: int = 1234, layers=range(NUM_LAYERS), scale: float = 1.0, t_shift: float = 0.0,
                  teacher_dim: int = TEACHER_DIM, n_tok: int = STUDENT_TOKENS - 1):
    """12-entry lists (None where the layer is not requested) of student [B,1+n_tok,192] and
    teacher [B,2+n_tok,teacher_dim] fp32 tensors (384: DeiT-Small, 768: DeiT-Base).  `n_tok` is the patch-token count:
    196 for 224-px inputs, 576 for 384-px inputs.  `scale`/`t_shift` give the Sinkhorn variant of §8d."""
    layers = set(int(i) % NUM_LAYERS for i in layers)
    s_feats, t_feats = [None] * NUM_LAYERS, [None] * NUM_LAYERS
    for i in range(NUM_LAYERS):
        if i not in layers:
            continue
        g = _gen(seed * 1000 + i)
        s_feats[i] = torch.randn(B, 1 + n_tok, STUDENT_DIM, generator=g) * scale
        t_feats[i] = torch.randn(B, 2 + n_tok, teacher_dim, generator=g) * scale + t_shift
    return s_feats, t_feats


def make_noise(B: int, L: int = 196, seed: int = 99) -> torch.Tensor:
    """Stand-in for the reference's torch.rand(N, L) draw (misc.py:14)."""
    return torch.rand(B, L, generator=_gen(seed))


class _Mlp(nn.Module):
    """`.mlp` of a stand-in block: emits a preset feature tensor so the reference's
    forward hooks (models.py:185-193) capture it."""

    def __init__(self):
        super().__init__()
        self.value = None

    def forward(self, x):
        return self.value


class _Block(nn.Module):
    def __init__(self):
        super().__init__()
        self.mlp = _Mlp()


class FeatureReplayModel(nn.Module):
    """Stand-in for a timm DeiT exposing what the hot path touches: `.embed_dim`,
    `.blocks[i].mlp`, and a forward that replays preset block outputs and logits.
    Used as the frozen teacher in tests / bench (teacher outputs are *inputs* to the
    loss path) and as the bare student that the KD heads are attached to."""

    def __init__(self, embed_dim: int, depth: int = NUM_LAYERS):
        super().__init__()
        self.embed_dim = embed_dim
        self.blocks = nn.ModuleList([_Block() for _ in range(depth)])
        self.logits = None

    def set_outputs(self, logits, feats):
        # plain attributes, set past nn.Module.__setattr__ (its parameter / buffer / module checks cost ~4 us per
        # assignment — this runs once per step inside the end-to-end timed region of bench.py)
        object.__setattr__(self, "logits", logits)
        object.__setattr__(self, "_has_feats", feats is not None)
        if feats is None and not getattr(self, "_feats_set", False):
            return                                  # logits-only replay: nothing to reset
        self._feats_set = feats is not None
        for blk, f in zip(self.blocks, feats if feats is not None else [None] * len(self.blocks)):
            blk.mlp.value = f

    def set_distilled_training(self, enable=True):  # models.py:97
        self.distilled_training = enable

    def forward(self, x):
        if getattr(self, "_has_feats", True):       # the hooks only matter when block outputs are replayed
            for blk in self.blocks:
                blk.mlp(x)
        return self.logits
