"""GPU: masked generation at 384-px inputs — the 24 x 24 patch grid (576 patch tokens; 577 student / 578 teacher tokens
with the special tokens) — against the fp64 oracle: the functional at both precisions, a persistent-loop case, MGD,
ViTKD and the whole CurKD curriculum through DistillationLoss, deterministic mode, clear errors for the grids and losses
that stay 224-px only, and one CurKD step of DeiT models built at img_size=384.  The mask noise is injected so that
mask selection is bit-identical; gradients are compared given the ReLU gate the kernel used (tests/gate_search.py)."""
from types import SimpleNamespace
from unittest import mock

import pytest
import torch

from oracle import losses as O
from oracle.util import rel_err
from tests.cases import A
from tests.gate_search import kernel_gate_oracle
from tests.test_deterministic_gpu import deterministic
from deltakd_b200 import heads as H
from deltakd_b200 import synth

pytestmark = pytest.mark.gpu

HW = 24
N = HW * HW


def _gate(hidden):
    """ReLU gate [B, Dt, 24, 24] (the oracle's NCHW layout) from the kernel's hidden planes [P, B, 576, Dt]."""
    live = (hidden.float() != 0).any(dim=0)
    B, n, D = live.shape
    return live.reshape(B, HW, HW, D).permute(0, 3, 1, 2).contiguous().cpu()


def _mgd_student(seed):
    teacher, student = synth.FeatureReplayModel(384), synth.FeatureReplayModel(192)
    torch.manual_seed(seed)
    H.attach_distillation_heads(student, teacher, SimpleNamespace(distillation_type="mgd"))
    with torch.no_grad():
        student.mask_token.normal_(0, 0.1)
    return student


# ----------------------------------------------------------------------------- the functional
@pytest.mark.parametrize("B,ratio", [(1, 0.5), (3, 0.25)])
@pytest.mark.parametrize("mode", ["bf16x3", "bf16"])
def test_masked_generation_576_matches_oracle(B, ratio, mode):
    """B * 24 image rows = 24 / 72: partial 5-row tiles in the forward / dgrad convolutions.  Loss, g_s, align W / b,
    mask_token and both convolutions' W / b against the fp64 oracle, given the kernel's ReLU gate."""
    from deltakd_b200 import functional as Fn
    Fn.set_matmul_precision(mode)
    try:
        student = _mgd_student(1)
        s_feats, t_feats = synth.make_features(B, 3, layers=[11], n_tok=N)
        noise = synth.make_noise(B, L=N, seed=B)
        host_heads = {k: v.detach().double() for k, v in H.head_tensors(student).items()}
        student = student.cuda()
        sc = s_feats[11].cuda().requires_grad_(True)
        probe = {}
        loss = Fn.masked_generation_loss(sc, t_feats[11].cuda(), student.align, student.mask_token, student.generation,
                                         mask_ratio=ratio, noise=noise.cuda(), scale=7e-5 / (B * N * 384), probe=probe)
        loss.backward()
        assert probe["mask"].shape == (B, N) and int(probe["mask"].sum()) == B * (N - int(N * (1 - ratio)))
        ours = {k: p.grad.detach().cpu().double() for k, p in H.head_tensors(student).items()}
        ours["s"] = sc.grad.detach().cpu().double()

        def eval_fn(pr):
            heads64 = {k: v.clone().requires_grad_(True) for k, v in host_heads.items()}
            s64 = s_feats[11].double().requires_grad_(True)
            l = O.mgd([s64], [t_feats[11].double()], heads64, 7e-5, ratio, noise, probe=pr)
            l.backward()
            g = {k: v.grad for k, v in heads64.items()}
            g["s"] = s64.grad
            return l, g

        tau = 3e-5 if mode == "bf16x3" else 3e-2
        ref, grads, n_amb, n_diff = kernel_gate_oracle(eval_fn, _gate(probe["hidden"]), tau=tau)
        print(f"[B={B} {mode}] ReLU gates: {n_amb} ambiguous, {n_diff} differ from the fp64 oracle's")
        lt, gt = (1e-5, 1e-4) if mode == "bf16x3" else (5e-3, 6e-2)   # as tests/test_mgd_gpu.py
        assert abs(loss.item() - ref.item()) <= lt * abs(ref.item()), (loss.item(), ref.item())
        assert len(ours) == 8   # g_s, align W / b, mask_token, 2 x (conv W, b)
        for k in ours:
            assert float(grads[k].abs().sum()) > 0, k
            assert rel_err(ours[k], grads[k]) < gt, (k, n_amb, n_diff)
        assert float(sc.grad[:, 0].abs().max()) == 0.0
    finally:
        Fn.set_matmul_precision(None)


def test_persistent_multi_tile_576():
    """B = 64: 308 forward tiles of 5 image rows on 148 CTAs, so every persistent loop wraps.  Splitting the batch gives
    the same loss, the same per-sample g_s, and convolution weight gradients that add up."""
    from deltakd_b200 import functional as Fn
    B = 64
    student = _mgd_student(2).cuda()
    s_feats, t_feats = synth.make_features(B, 5, layers=[11], n_tok=N)
    s, t = s_feats[11].cuda(), t_feats[11].cuda()
    noise = synth.make_noise(B, L=N, seed=8).cuda()

    def run(sl):
        x = s[sl].clone().requires_grad_(True)
        for p in student.parameters():
            p.grad = None
        l = Fn.masked_generation_loss(x, t[sl], student.align, student.mask_token, student.generation,
                                      mask_ratio=0.5, noise=noise[sl], scale=1e-6)
        l.backward()
        return l.item(), x.grad, student.generation[0].weight.grad.clone(), student.generation[2].weight.grad.clone()

    full = run(slice(0, B))
    parts = [run(slice(i, i + 16)) for i in range(0, B, 16)]
    assert abs(sum(p[0] for p in parts) - full[0]) <= 2e-5 * abs(full[0])
    assert rel_err(torch.cat([p[1] for p in parts]), full[1]) < 1e-4
    assert rel_err(sum(p[2] for p in parts), full[2]) < 1e-4
    assert rel_err(sum(p[3] for p in parts), full[3]) < 1e-4


# ----------------------------------------------------------------------------- DistillationLoss end to end
def _case(kind, B=2, dtype=torch.float32, device="cuda", **args):
    """The tests/cases.py construction at 577 / 578 tokens; `noise` is the [B, 576] mask noise torch.rand would draw."""
    a = A(**args)
    a.distillation_type = kind
    teacher = synth.FeatureReplayModel(384)
    student = synth.FeatureReplayModel(192)
    torch.manual_seed(0)
    H.attach_distillation_heads(student, teacher, a, "deit_tiny_patch16_224")
    if hasattr(student, "mask_token"):
        with torch.no_grad():
            student.mask_token.copy_(torch.randn(student.mask_token.shape, generator=torch.Generator().manual_seed(7)) * 0.1)
    student = student.to(dtype).to(device)
    outputs, _, t_logits, labels = synth.make_logits(B, 100, 1234)
    outputs, t_logits, labels = (x.to(dtype).to(device) for x in (outputs, t_logits, labels))
    s_feats, t_feats = synth.make_features(B, 1234, n_tok=N)
    s_feats = [f.to(dtype).to(device).requires_grad_(True) for f in s_feats]
    t_feats = [f.to(dtype).to(device) for f in t_feats]
    teacher.set_outputs(t_logits, t_feats)
    outputs.requires_grad_(True)
    noise = synth.make_noise(B, L=N, seed=4321).to(device)
    return SimpleNamespace(kind=kind, args=a, B=B, teacher=teacher, student=student, outputs=outputs, labels=labels,
                           teacher_logits=t_logits, s_feats=s_feats, t_feats=t_feats, noise=noise)


def _criterion_loss(c, probe=None):
    from deltakd_b200 import DistillationLoss, call_base_loss
    from deltakd_b200 import functional as Fn
    crit = DistillationLoss(call_base_loss(c.args), c.teacher, c.kind, 0.1, 3.0)
    real = Fn.masked_generation_loss
    spy = (lambda *a, **k: real(*a, probe=probe, **k)) if probe is not None else real
    with mock.patch("torch.rand", side_effect=lambda *a, **k: c.noise.clone()), \
            mock.patch.object(Fn, "masked_generation_loss", spy):
        return crit(torch.zeros(c.B, 3, 2, 2, device="cuda"), c.outputs, c.student, c.s_feats, c.labels, c.args)


# n_grads: parameter and feature gradients the type produces.  Masked generation: g_s, align W / b, mask_token and
# 2 x (conv W, b); ViTKD adds two mimicking heads and their two student layers; CurKD early / mid: 3 / 4 heads and layers.
@pytest.mark.parametrize("kind,args,n_grads", [("mgd", {}, 8), ("vitkd", {}, 14), ("curkd", dict(current_epoch=0), 9),
                                               ("curkd", dict(current_epoch=120), 12), ("curkd", dict(current_epoch=200), 8)],
                         ids=["mgd", "vitkd", "curkd_ep0", "curkd_ep120", "curkd_ep200"])
def test_distillation_loss_576_matches_oracle(kind, args, n_grads):
    c = _case(kind, **args)
    probe = {}
    loss = _criterion_loss(c, probe)
    loss.backward()
    heads = H.head_tensors(c.student)
    ours = {k: p.grad.detach().double().cpu() for k, p in heads.items() if p.grad is not None}
    for i, f in enumerate(c.s_feats):
        if f.grad is not None:
            ours[f"s{i}"] = f.grad.detach().double().cpu()
            assert float(f.grad[:, 0].abs().max()) == 0.0, i

    def eval_fn(pr):
        o = _case(kind, dtype=torch.float64, device="cpu", **args)
        oh = H.head_tensors(o.student)
        l = O.distillation_loss(o.kind, o.outputs, o.labels, o.teacher_logits, o.s_feats, o.t_feats, oh, o.args, 0.1, 3.0,
                                noise=o.noise, probe=pr)
        l.backward()
        g = {k: v.grad for k, v in oh.items() if v.grad is not None}
        for i, f in enumerate(o.s_feats):
            if f.grad is not None:
                g[f"s{i}"] = f.grad
        return l, g

    generation = kind != "curkd" or args["current_epoch"] >= 151
    assert ("hidden" in probe) == generation
    if generation:
        ol, grads, n_amb, n_diff = kernel_gate_oracle(eval_fn, _gate(probe["hidden"]))
        print(f"[{kind} {args}] ReLU gates: {n_amb} ambiguous, {n_diff} differ from the fp64 oracle's")
    else:
        ol, grads = eval_fn(None)
    assert abs(loss.item() - ol.item()) <= 1e-5 * abs(ol.item()), (loss.item(), ol.item())
    assert set(ours) == set(grads), (sorted(ours), sorted(grads))
    assert len(grads) == n_grads, sorted(grads)
    for k in grads:
        assert rel_err(ours[k], grads[k]) < 1e-4, k


# ----------------------------------------------------------------------------- deterministic mode
def _mgd_call(B, dtype, seed=5):
    """masked_generation_loss at 576 tokens with seeded heads, inputs and mask: a closure giving [loss, g_s, head grads]."""
    from deltakd_b200 import functional as Fn
    g = torch.Generator().manual_seed(seed)
    s = torch.randn(B, 1 + N, 192, generator=g).to(dtype).cuda()
    t = torch.randn(B, 2 + N, 384, generator=g).to(dtype).cuda()
    mask = (torch.rand(B, N, generator=g) < 0.5).float().cuda()
    student = _mgd_student(seed).cuda()
    params = list(H.head_tensors(student).values())

    def run():
        sc = s.clone().requires_grad_(True)
        for p in params:
            p.grad = None
        loss = Fn.masked_generation_loss(sc, t, student.align, student.mask_token, student.generation,
                                         scale=7e-5 / (B * N * 384), mask=mask)
        loss.backward()
        torch.cuda.synchronize()
        return [loss.detach().clone(), sc.grad] + [p.grad for p in params]
    return run


def _equal(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), (i, float((x.double() - y.double()).abs().max()))


@pytest.mark.parametrize("B,dtype", [(5, torch.float32), (5, torch.bfloat16), (64, torch.float32)])
def test_deterministic_repeated_calls_576(B, dtype):
    run = _mgd_call(B, dtype)
    with deterministic("cudnn"):
        first = [x.clone() for x in run()]
        _equal(first, run())


def test_deterministic_graph_replay_576():
    run = _mgd_call(5, torch.float32)
    with deterministic("cudnn"):
        eager = [x.clone() for x in run()]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run()   # warm-up outside the capture (scratch allocation, lazy module loads)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with mock.patch("torch.cuda.synchronize"), torch.cuda.graph(graph, stream=side):
            outs = run()
        for _ in range(2):
            graph.replay()
            torch.cuda.synchronize()
            _equal(eager, outs)


# ----------------------------------------------------------------------------- clear errors
@pytest.mark.parametrize("n_tok", [225, 200])
def test_other_grids_raise_clearly(n_tok):
    from deltakd_b200 import _lib
    from deltakd_b200 import functional as Fn
    student = _mgd_student(0).cuda()
    s, t = torch.randn(2, 1 + n_tok, 192, device="cuda"), torch.randn(2, 2 + n_tok, 384, device="cuda")
    with pytest.raises(ValueError, match=r"built for 196 patch tokens .* or 576 patch tokens .*got %d" % n_tok):
        Fn.masked_generation_loss(s, t, student.align, student.mask_token, student.generation, scale=1.0, mask_ratio=0.5)
    # the C ABI checks the grid itself (before it reads any pointer), including a student / teacher mismatch
    fn = _lib.lib.dkd_masked_generation_fwdbwd
    for Ts, Tt in ((1 + n_tok, 2 + n_tok), (1 + N, 2 + 196)):
        rc = fn(*([None] * 10), 2, Ts, 1, Tt, 2, 192, 384, _lib.F32, _lib.PREC_BF16X3, 1.0, *([None] * 10), 0, None)
        assert rc == -1 and "196 (14x14 grid) or 576 (24x24 grid)" in _lib.last_error(), _lib.last_error()


@pytest.mark.parametrize("kind,args,match", [
    ("wasskd", dict(wasskd_type="l1"), r"n_tok <= 256"),
    ("saliency_mgd", dict(saliency_method=1), r"built for 196 patch tokens"),
    ("saliency_mgd", dict(saliency_method=2), r"n_keys < 256"),
    ("saliency_mgd", dict(saliency_method=3), r"n_keys < 256"),
], ids=["wasskd_l1", "saliency_mgd_m1", "saliency_mgd_m2", "saliency_mgd_m3"])
def test_224_only_losses_raise_at_first_call(kind, args, match):
    c = _case(kind, **args)
    with pytest.raises(RuntimeError, match=match):
        _criterion_loss(c)


@pytest.mark.parametrize("kind", ["lrkd", "diffkd"])
def test_lrkd_and_diffkd_run_at_576(kind):
    """Their kernels take any token count: at 384 px the first call gives a finite loss and finite gradients on every
    student feature it reads.  (Not compared with the oracle at this size.)"""
    c = _case(kind)
    loss = _criterion_loss(c)
    loss.backward()
    assert torch.isfinite(loss).item()
    fed = [f for f in c.s_feats if f.grad is not None]
    assert fed and all(torch.isfinite(f.grad).all().item() for f in fed)


def test_deit_384_curkd_late_step():
    """A FrozenTeacher DeiT-Small at img_size=384 feeds one CurKD epoch-200 step (masked generation on block 11) of a
    DeiT-Tiny student at img_size=384: finite loss, and the generator convolutions get finite, non-zero gradients."""
    from deltakd_b200 import DistillationLoss, FrozenTeacher, attach_distillation_heads, deit, forward_with_features
    from deltakd_b200.loss import LabelSmoothingCrossEntropy
    args = A(current_epoch=200)
    args.distillation_type = "curkd"
    torch.manual_seed(0)
    teacher = FrozenTeacher(deit.create_model("deit_small_distilled_patch16_224", num_classes=100, img_size=384).cuda())
    student = deit.create_model("deit_tiny_patch16_224", num_classes=100, img_size=384)
    attach_distillation_heads(student, teacher, args, "deit_tiny_patch16_224")
    student = student.cuda().train()
    x = torch.randn(2, 3, 384, 384, device="cuda")
    labels = torch.tensor([3, 7], device="cuda")
    outputs, s_feats = forward_with_features(student, x, layers=(11,))
    assert s_feats[11].shape == (2, 577, 192)
    crit = DistillationLoss(LabelSmoothingCrossEntropy(0.1), teacher, "curkd", 0.1, 3.0)
    loss = crit(x, outputs, student, s_feats, labels, args)
    loss.backward()
    assert torch.isfinite(loss).item()
    for conv in (student.generation[0], student.generation[2]):
        assert conv.weight.grad is not None and torch.isfinite(conv.weight.grad).all().item()
        assert float(conv.weight.grad.abs().sum()) > 0
