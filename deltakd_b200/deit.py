"""Minimal DeiT (timm-compatible attribute surface) — BENCH / TEST HARNESS ONLY.

The reference builds its student and teacher with `timm.create_model` (model/models.py:59-75); timm is not in this
image and the models are outside the hot path (SURVEY.md §8: plain PyTorch is fine; `row_ops="dkd"` swaps the
HBM-bound LayerNorm / bias-gradient / head-relayout passes for libdeltakd_sm100 kernels, §8f rank 1).  This file
provides random-init stand-ins of `deit_tiny[_distilled]_patch16_224` (192-d, 3 heads),
`deit_small[_distilled]_patch16_224` (384-d, 6 heads) and `deit_base[_distilled]_patch16_224` (768-d, 12 heads; the
wider teacher of the 192 -> 768 feature losses) exposing exactly what the loss path touches:
`.embed_dim`, `.blocks[i].mlp` (hooked by forward_with_features, models.py:185-193), `.head` / `.head_dist`,
`set_distilled_training` (models.py:97), and timm's output convention (distilled + training + distilled_training
-> (cls_logits, dist_logits); otherwise their mean / the single head).
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F


class LayerNorm(nn.LayerNorm):
    """nn.LayerNorm parameters / state_dict, computed by dkd_layernorm_fwd / _bwd (deltakd_b200/csrc/rowops.cu); under
    autocast the output is written directly in the autocast dtype.  CUDA tensors only (`row_ops="dkd"` models)."""

    def forward(self, x):
        from . import functional as Fn
        out_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
        return Fn.layer_norm(x, self.weight, self.bias, self.eps, out_dtype)


class Linear(nn.Linear):
    """nn.Linear parameters: cuBLAS GEMMs both ways; when a gradient is needed the bias gradient is reduced by dkd_colsum."""

    def forward(self, x):
        if not torch.is_grad_enabled() or not self.weight.requires_grad:
            return super().forward(x)          # frozen / inference: no backward, nothing to replace
        from . import functional as Fn
        return Fn.linear_tokens(x, self.weight, self.bias)


# row_ops = "aten": plain torch modules (the timm-like model the reference runs; CPU-capable — used by the CPU tests and
#                   by the oracle-side step of bench.py's cpu_baseline);
# row_ops = "dkd" : the same parameters on libdeltakd_sm100's row ops (CUDA only, no fallback: CPU tensors raise).
_ROW_OPS = {"aten": (nn.LayerNorm, nn.Linear), "dkd": (LayerNorm, Linear)}


class Mlp(nn.Module):
    def __init__(self, dim: int, hidden: int, row_ops: str = "aten"):
        super().__init__()
        _, Lin = _ROW_OPS[row_ops]
        self.fc1 = Lin(dim, hidden)
        self.act = nn.GELU()
        self.fc2 = Lin(hidden, dim)

    def forward(self, x):
        return self.fc2(self.act(self.fc1(x)))


class Attention(nn.Module):
    def __init__(self, dim: int, num_heads: int, row_ops: str = "aten"):
        super().__init__()
        _, Lin = _ROW_OPS[row_ops]
        self.num_heads = num_heads
        self.dkd = row_ops == "dkd"
        self.qkv = Lin(dim, dim * 3)
        self.proj = Lin(dim, dim)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x)
        if self.dkd:   # head relayouts by dkd_head_copy (ATen: strided copies, and select-backward fills / cat in backward)
            from . import functional as Fn
            q, k, v = Fn.split_qkv(qkv, self.num_heads)
            return self.proj(Fn.merge_heads(F.scaled_dot_product_attention(q, k, v)))
        q, k, v = qkv.reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4).unbind(0)
        x = F.scaled_dot_product_attention(q, k, v)
        return self.proj(x.transpose(1, 2).reshape(B, N, C))


class Block(nn.Module):
    def __init__(self, dim: int, num_heads: int, mlp_ratio: float = 4.0, row_ops: str = "aten"):
        super().__init__()
        Norm, _ = _ROW_OPS[row_ops]
        self.norm1 = Norm(dim, eps=1e-6)
        self.attn = Attention(dim, num_heads, row_ops)
        self.norm2 = Norm(dim, eps=1e-6)
        self.mlp = Mlp(dim, int(dim * mlp_ratio), row_ops)

    def forward(self, x):
        x = x + self.attn(self.norm1(x))
        return x + self.mlp(self.norm2(x))


class DeiT(nn.Module):
    def __init__(self, embed_dim: int, depth: int, num_heads: int, num_classes: int = 1000, distilled: bool = False,
                 img_size: int = 224, patch: int = 16, row_ops: str = "aten"):
        super().__init__()
        Norm, Lin = _ROW_OPS[row_ops]
        self.row_ops = row_ops
        self.embed_dim = embed_dim
        self.distilled = distilled
        self.distilled_training = False
        n = (img_size // patch) ** 2
        self.patch = patch
        # non-overlapping 16x16 patches: the stride-16 convolution is a GEMM over unfolded patches (same parameters,
        # [D, 3*16*16] weight) — cuDNN's strided-conv kernel is ~5x slower than the GEMM at these shapes
        self.patch_embed = Lin(3 * patch * patch, embed_dim)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.dist_token = nn.Parameter(torch.zeros(1, 1, embed_dim)) if distilled else None
        self.pos_embed = nn.Parameter(torch.randn(1, n + (2 if distilled else 1), embed_dim) * 0.02)
        self.blocks = nn.ModuleList([Block(embed_dim, num_heads, row_ops=row_ops) for _ in range(depth)])
        self.norm = Norm(embed_dim, eps=1e-6)
        self.head = nn.Linear(embed_dim, num_classes)
        self.head_dist = nn.Linear(embed_dim, num_classes) if distilled else None

    def set_distilled_training(self, enable: bool = True):
        self.distilled_training = enable

    def forward(self, x):
        B, C, H, W = x.shape
        pz = self.patch
        x = x.reshape(B, C, H // pz, pz, W // pz, pz).permute(0, 2, 4, 1, 3, 5).reshape(B, (H // pz) * (W // pz), C * pz * pz)
        x = self.patch_embed(x)
        toks = [self.cls_token.expand(x.shape[0], -1, -1)]
        if self.distilled:
            toks.append(self.dist_token.expand(x.shape[0], -1, -1))
        x = torch.cat(toks + [x], dim=1) + self.pos_embed
        for blk in self.blocks:
            x = blk(x)
        x = self.norm(x)
        if not self.distilled:
            return self.head(x[:, 0])
        a, b = self.head(x[:, 0]), self.head_dist(x[:, 1])
        if self.distilled_training and self.training and not torch.jit.is_scripting():
            return a, b
        return (a + b) / 2


_ZOO = {
    "deit_tiny_patch16_224": dict(embed_dim=192, depth=12, num_heads=3, distilled=False),
    "deit_tiny_distilled_patch16_224": dict(embed_dim=192, depth=12, num_heads=3, distilled=True),
    "deit_small_patch16_224": dict(embed_dim=384, depth=12, num_heads=6, distilled=False),
    "deit_small_distilled_patch16_224": dict(embed_dim=384, depth=12, num_heads=6, distilled=True),
    "deit_base_patch16_224": dict(embed_dim=768, depth=12, num_heads=12, distilled=False),
    "deit_base_distilled_patch16_224": dict(embed_dim=768, depth=12, num_heads=12, distilled=True),
}


def create_model(name: str, num_classes: int = 1000, row_ops: str = "aten", img_size: int = 224, **_) -> DeiT:
    """Stand-in for timm.create_model(name, pretrained=False, num_classes=..., img_size=...) restricted to the DeiT variants the
    reference's exp/*.sh scripts use, plus the DeiT-Base teacher.  `img_size` is timm's keyword: 384 gives the 24 x 24 patch
    grid of the DeiT "384" recipe (577 tokens, 578 distilled).  `row_ops="dkd"` builds the same model (same state_dict) on libdeltakd_sm100's
    LayerNorm / bias-gradient / head-relayout kernels — CUDA only."""
    if name not in _ZOO:
        raise ValueError(f"unknown model {name}; available: {sorted(_ZOO)}")
    if row_ops not in _ROW_OPS:
        raise ValueError(f"row_ops must be one of {sorted(_ROW_OPS)}, got {row_ops!r}")
    return DeiT(num_classes=num_classes, row_ops=row_ops, img_size=img_size, **_ZOO[name])
