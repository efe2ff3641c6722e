"""GPU: the DeiT-Tiny <- DeiT-Base pair (student 192, teacher 768) — hidden-state matching (CurKD early / mid, ViTKD
mimicking) and WassKD-l1 against the fp64 oracle, end to end through DistillationLoss, repeatability and CUDA-graph
replay, and the losses that stay built for 192 -> 384 only raising a clear error at their first call."""
from types import SimpleNamespace

import pytest
import torch

from oracle import losses as O
from oracle.util import rel_err
from tests.cases import A
from tests.test_wass_gpu import _close, _flip_budget
from deltakd_b200 import heads as H
from deltakd_b200 import synth

pytestmark = pytest.mark.gpu

DT = 768
TOL = {"f32": (1e-5, 1e-4), "bf16": (2e-2, 5e-2)}     # (loss, gradients): bf16x3 on fp32 data | one bf16 pass on bf16 data


def _curkd_heads(n_layers, seed=0):
    torch.manual_seed(seed)
    return [torch.nn.Linear(192, DT).cuda() for _ in range(n_layers)]


def _feats(B, layers, dtype):
    s_feats, t_feats = synth.make_features(B, 17, layers=layers, teacher_dim=DT)
    s = [s_feats[i].to(dtype).cuda() for i in layers]
    t = [t_feats[i].to(dtype).cuda() for i in layers]
    return s, t


def _oracle_curkd(s, t, lins, epoch):
    """fp64 oracle of curkd_loss early (3 layers) / mid (4 layers) on the GPU, on the same (rounded) inputs."""
    n = len(lins)
    off = 0 if epoch < 100 else 3
    name = "curkd_align_early" if epoch < 100 else "curkd_align_mid"
    sd = [None] * 12
    td = [None] * 12
    heads = {}
    for j in range(n):
        sd[off + j] = s[j].detach().double().requires_grad_(True)
        td[off + j] = t[j].double()
        heads[f"{name}.{j}.weight"] = lins[j].weight.detach().double().requires_grad_(True)
        heads[f"{name}.{j}.bias"] = lins[j].bias.detach().double().requires_grad_(True)
    loss = O.curkd_hidden(sd, td, heads, epoch)
    loss.backward()
    return loss.item(), [sd[off + j].grad for j in range(n)], [heads[f"{name}.{j}.weight"].grad for j in range(n)], \
        [heads[f"{name}.{j}.bias"].grad for j in range(n)]


def _ours_curkd(s, t, lins, B):
    from deltakd_b200 import functional as Fn
    sc = [x.detach().clone().requires_grad_(True) for x in s]
    for lin in lins:
        lin.zero_grad(set_to_none=True)
    loss = Fn.align_mse_layers_loss(sc, t, lins, scale=4e-5 / len(lins) / B)
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), [x.grad for x in sc], [lin.weight.grad.clone() for lin in lins], [lin.bias.grad.clone() for lin in lins]


@pytest.mark.parametrize("B", [1, 3, 37, 512])
@pytest.mark.parametrize("mode", ["f32", "bf16"])
def test_align_mse_768_matches_oracle(B, mode):
    """3 layers (CurKD early): loss, g_s, g_W and g_b at B*196 rows, 37 leaving a partial last 128-row tile."""
    dtype = torch.float32 if mode == "f32" else torch.bfloat16
    s, t = _feats(B, [0, 1, 2], dtype)
    lins = _curkd_heads(3)
    l, gs, gw, gb = _ours_curkd(s, t, lins, B)
    ol, ogs, ogw, ogb = _oracle_curkd(s, t, lins, 0)
    lt, gt = TOL[mode]
    assert abs(l - ol) <= lt * abs(ol), (l, ol)
    for j in range(3):
        assert gs[j].dtype == dtype
        assert float(gs[j][:, 0].abs().max()) == 0.0          # CLS rows get exactly zero gradient
        assert rel_err(gs[j].double(), ogs[j]) < gt, ("g_s", j)
        assert rel_err(gw[j].double(), ogw[j]) < gt, ("g_W", j)
        assert rel_err(gb[j].double(), ogb[j]) < gt, ("g_b", j)


@pytest.mark.parametrize("epoch,n_layers", [(0, 3), (120, 4)])
def test_align_mse_768_layer_streams(monkeypatch, epoch, n_layers):
    """CurKD early (3 layers) and mid (4 layers): every layer on its own stream gives the single-stream result (g_s
    bit-identical), and both match the oracle."""
    from deltakd_b200 import functional as Fn
    B = 37
    s, t = _feats(B, list(range(n_layers)), torch.float32)
    lins = _curkd_heads(n_layers, seed=epoch)
    monkeypatch.setattr(Fn, "_LAYER_STREAMS", True)
    l1, gs1, gw1, gb1 = _ours_curkd(s, t, lins, B)
    monkeypatch.setattr(Fn, "_LAYER_STREAMS", False)
    l0, gs0, gw0, gb0 = _ours_curkd(s, t, lins, B)
    assert abs(l1 - l0) <= 1e-6 * abs(l0)
    for a, b in zip(gs1, gs0):
        assert torch.equal(a, b)
    for a, b in zip(gw1 + gb1, gw0 + gb0):   # split-K weight gradients: fp32 atomics, equal up to the order of the adds
        assert rel_err(a, b) < 1e-5
    ol, ogs, ogw, ogb = _oracle_curkd(s, t, lins, epoch)
    assert abs(l1 - ol) <= 1e-5 * abs(ol)
    for j in range(n_layers):
        assert rel_err(gs1[j].double(), ogs[j]) < 1e-4
        assert rel_err(gw1[j].double(), ogw[j]) < 1e-4
        assert rel_err(gb1[j].double(), ogb[j]) < 1e-4


@pytest.mark.parametrize("B", [2, 37])
def test_wass_l1_768_matches_oracle(B):
    """WassKD-l1 over 3 layers at 768 channels (48 sort CTAs per sample, 4 N tiles in the align GEMM, 12 K blocks in
    dgrad, two 3-CTA tile groups in wgrad), with the ambiguous-sign budget of test_wass_gpu.py."""
    from deltakd_b200 import functional as Fn
    s, t = _feats(B, [0, 1, 2], torch.float32)
    torch.manual_seed(3)
    lins = [torch.nn.Linear(192, DT).cuda() for _ in range(3)]
    sc = [x.clone().requires_grad_(True) for x in s]
    loss = Fn.wass_l1_loss(sc, t, lins, weight=5.0)
    loss.backward()
    heads64 = {}
    for i, lin in enumerate(lins):
        heads64[f"align_wasskd.{i}.weight"] = lin.weight.detach().double().requires_grad_(True)
        heads64[f"align_wasskd.{i}.bias"] = lin.bias.detach().double().requires_grad_(True)
    o = SimpleNamespace(s_feats=[x.detach().double().requires_grad_(True) for x in s], t_feats=[x.double() for x in t])
    ol = O.wass_l1(o.s_feats, o.t_feats, heads64) * 5.0
    ol.backward()
    assert abs(loss.item() - ol.item()) <= 1e-5 * abs(ol.item())
    budget = _flip_budget(o, heads64)
    # The ambiguous elements are a property of the fp64 inputs, and their number grows with B * 196 * Dt.  Bound
    # their density at test_wass_gpu.py's (64 in its 2 * 196 * 384 elements), so that the budget stays a few
    # isolated sign flips: B = 37 at Dt = 768 has 37x as many elements.
    numel = B * 196 * DT
    for i in range(3):
        nb, gs, gw, gb = budget[i]
        assert nb <= 64 * numel / (2 * 196 * 384), f"layer {i}: {nb} ambiguous elements in {numel}"
        _close(sc[i].grad, o.s_feats[i].grad, gs, f"g_s{i} ({nb} ambiguous)")
        assert float(sc[i].grad[:, 0].abs().max()) == 0.0
        _close(lins[i].weight.grad, heads64[f"align_wasskd.{i}.weight"].grad, gw, f"g_W{i}")
        _close(lins[i].bias.grad, heads64[f"align_wasskd.{i}.bias"].grad, gb, f"g_b{i}")


def test_wass_l1_768_bf16_permutation_invariant():
    """bf16 I/O (one plane, the bf16 G plane path): the loss does not see a permutation of each sample's tokens."""
    from deltakd_b200 import functional as Fn
    s, t = _feats(3, [0], torch.bfloat16)
    torch.manual_seed(5)
    lin = torch.nn.Linear(192, DT).cuda()
    base = Fn.wass_l1_loss(s, t, [lin], weight=1.0).item()
    g = torch.Generator().manual_seed(3)
    ps = torch.cat([torch.zeros(1, dtype=torch.long), 1 + torch.randperm(196, generator=g)]).cuda()
    pt = torch.cat([torch.arange(2), 2 + torch.randperm(196, generator=g)]).cuda()
    perm = Fn.wass_l1_loss([s[0][:, ps].contiguous()], [t[0][:, pt].contiguous()], [lin], weight=1.0).item()
    assert abs(perm - base) <= 2e-6 * abs(base)


# ----------------------------------------------------------------------------- DistillationLoss end to end
def _case(kind, B=2, dtype=torch.float32, device="cuda", **args):
    """The tests/cases.py construction with a 768-wide teacher stand-in (heads built by attach_distillation_heads)."""
    a = A(**args)
    a.distillation_type = kind
    teacher = synth.FeatureReplayModel(DT)
    student = synth.FeatureReplayModel(192)
    torch.manual_seed(0)
    H.attach_distillation_heads(student, teacher, a, "deit_tiny_patch16_224")
    student = student.to(dtype).to(device)
    outputs, outputs_kd, t_logits, labels = synth.make_logits(B, 100, 1234)
    outputs, t_logits, labels = (x.to(dtype).to(device) for x in (outputs, t_logits, labels))
    s_feats, t_feats = synth.make_features(B, 1234, teacher_dim=DT)
    s_feats = [f.to(dtype).to(device).requires_grad_(True) for f in s_feats]
    t_feats = [f.to(dtype).to(device) for f in t_feats]
    teacher.set_outputs(t_logits, t_feats)
    outputs.requires_grad_(True)
    return SimpleNamespace(kind=kind, args=a, B=B, teacher=teacher, student=student, outputs=outputs, labels=labels,
                           teacher_logits=t_logits, s_feats=s_feats, t_feats=t_feats)


def _criterion_loss(c):
    from deltakd_b200 import DistillationLoss, call_base_loss
    crit = DistillationLoss(call_base_loss(c.args), c.teacher, c.kind, 0.1, 3.0)
    torch.manual_seed(4321)
    return crit(torch.zeros(c.B, 3, 2, 2, device="cuda"), c.outputs, c.student, c.s_feats, c.labels, c.args)


@pytest.mark.parametrize("kind,args", [("curkd", dict(current_epoch=0)), ("curkd", dict(current_epoch=120)),
                                       ("wasskd", dict(wasskd_type="l1"))])
def test_distillation_loss_768_matches_oracle(kind, args):
    c = _case(kind, **args)
    loss = _criterion_loss(c)
    loss.backward()
    o = _case(kind, dtype=torch.float64, device="cpu", **args)
    oh = H.head_tensors(o.student)
    ol = O.distillation_loss(o.kind, o.outputs, o.labels, o.teacher_logits, o.s_feats, o.t_feats, oh, o.args, 0.1, 3.0)
    ol.backward()
    assert abs(loss.item() - ol.item()) <= 1e-5 * abs(ol.item()), (loss.item(), ol.item())
    heads = H.head_tensors(c.student)
    budget = _flip_budget(o, oh) if kind == "wasskd" else None
    n_checked = 0
    for k in oh:
        if oh[k].grad is None:
            assert heads[k].grad is None, k
            continue
        n_checked += 1
        if budget is None:
            assert rel_err(heads[k].grad.double().cpu(), oh[k].grad) < 1e-4, k
        else:
            i = int(k.split(".")[1])
            _close(heads[k].grad, oh[k].grad, budget[i][2 if k.endswith("weight") else 3], k)
    assert n_checked == (6 if kind == "wasskd" else 2 * (3 if args.get("current_epoch", 0) < 100 else 4))
    for i, (f, g) in enumerate(zip(c.s_feats, o.s_feats)):
        if g.grad is None:
            assert f.grad is None, i
            continue
        assert float(f.grad[:, 0].abs().max()) == 0.0
        if budget is None:
            assert rel_err(f.grad.double().cpu(), g.grad) < 1e-4, i
        else:
            _close(f.grad, g.grad, budget[i][1], f"g_s{i}")


@pytest.mark.parametrize("kind,args", [("curkd", dict(current_epoch=200)), ("mgd", {}), ("lrkd", {}), ("diffkd", {}),
                                       ("wasskd", dict(wasskd_type="sinkhorn"))])
def test_unsupported_at_768_raise_clearly(kind, args):
    """The losses still built for 192 -> 384 only reject the 768-wide teacher at their first call, naming the pairs."""
    c = _case(kind, **args)
    with pytest.raises(ValueError, match=r"built for student/teacher widths 192 -> 384 .*got 192 -> 768"):
        _criterion_loss(c)


# ----------------------------------------------------------------------------- repeatability
@pytest.mark.parametrize("entry", ["align_mse", "wass_l1"])
def test_768_repeatable_and_graph_replay(entry):
    """Two eager calls give bit-identical loss and g_s; a captured CUDA graph of forward + backward, replayed twice,
    gives the eager result bit for bit."""
    from deltakd_b200 import functional as Fn
    B = 37
    s, t = _feats(B, [0, 1, 2], torch.float32)
    lins = _curkd_heads(3, seed=9)
    fn = (lambda x: Fn.align_mse_layers_loss(x, t, lins, scale=1e-4)) if entry == "align_mse" \
        else (lambda x: Fn.wass_l1_loss(x, t, lins, weight=5.0))
    sc = [x.clone().requires_grad_(True) for x in s]

    def eager():
        for x in sc:
            x.grad = None
        loss = fn(sc)
        loss.backward()
        torch.cuda.synchronize()
        return loss.detach().clone(), [x.grad.clone() for x in sc]

    la, ga = eager()
    lb, gb = eager()
    assert torch.equal(la, lb)
    for a, b in zip(ga, gb):
        assert torch.equal(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):      # warm-up on the capture stream (its scratch)
        fn(sc).backward()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for x in sc:
        x.grad = None
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        loss = fn(sc)
        loss.backward()
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(loss, la)
        for x, a in zip(sc, ga):
            assert torch.equal(x.grad, a)


def test_frozen_deit_base_teacher_curkd_step():
    """A FrozenTeacher(DeiT-Base) forward feeds one CurKD-early step of a DeiT-Tiny student: no error, finite loss,
    gradients on the three alignment heads."""
    from deltakd_b200 import DistillationLoss, FrozenTeacher, attach_distillation_heads, deit, forward_with_features
    from deltakd_b200.loss import LabelSmoothingCrossEntropy
    args = A(current_epoch=0)
    args.distillation_type = "curkd"
    torch.manual_seed(0)
    teacher = FrozenTeacher(deit.create_model("deit_base_distilled_patch16_224", num_classes=100).cuda())
    student = deit.create_model("deit_tiny_patch16_224", num_classes=100)
    attach_distillation_heads(student, teacher, args, "deit_tiny_patch16_224")
    student = student.cuda().train()
    assert teacher.embed_dim == DT and student.curkd_align_early[0].out_features == DT
    x = torch.randn(2, 3, 224, 224, device="cuda")
    labels = torch.tensor([3, 7], device="cuda")
    outputs, s_feats = forward_with_features(student, x, layers=(0, 1, 2))
    crit = DistillationLoss(LabelSmoothingCrossEntropy(0.1), teacher, "curkd", 0.1, 3.0)
    loss = crit(x, outputs, student, s_feats, labels, args)
    loss.backward()
    assert torch.isfinite(loss).item()
    for lin in student.curkd_align_early:
        assert lin.weight.grad is not None and torch.isfinite(lin.weight.grad).all().item()
