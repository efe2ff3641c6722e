"""GPU: the deterministic mode of the feature losses (DKD_PREC_DETERMINISTIC, selected by
torch.use_deterministic_algorithms(True) or torch.backends.cudnn.deterministic).  Every gradient — g_s and the head,
generator-convolution and mask-token gradients — must be bit-identical across repeated calls, layer streams on and off,
concurrent work on another stream, CUDA-graph replay and a fresh process, and still meet the fp64 oracle at the
existing tests' tolerances (those tests are re-run here with the mode on)."""
import contextlib
import ctypes
import os
import subprocess
import sys
from unittest import mock

import pytest
import torch

import tests.test_curkd_gpu as curkd_t
import tests.test_diffkd_gpu as diffkd_t
import tests.test_lrkd_gpu as lrkd_t
import tests.test_mgd_gpu as mgd_t
import tests.test_sinkhorn_gpu as sinkhorn_t
import tests.test_teacher_width_768_gpu as w768_t
import tests.test_wass_gpu as wass_t
from tests.cases import build_case
from deltakd_b200 import heads as H
from deltakd_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def deterministic(flag="torch"):
    """The mode on through one of the two torch flags that select it; both flags restored afterwards."""
    was_alg, was_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    was_cudnn = torch.backends.cudnn.deterministic
    try:
        if flag == "torch":   # warn_only: the oracle's own torch ops need not have deterministic implementations
            torch.use_deterministic_algorithms(True, warn_only=True)
        else:
            torch.backends.cudnn.deterministic = True
        yield
    finally:
        torch.use_deterministic_algorithms(was_alg, warn_only=was_warn)
        torch.backends.cudnn.deterministic = was_cudnn


def _equal(a, b, what):
    assert len(a) == len(b), what
    for i, (x, y) in enumerate(zip(a, b)):
        if x is None or y is None:
            assert x is None and y is None, (what, i)
            continue
        assert torch.equal(x, y), (what, i, float((x.double() - y.double()).abs().max()))


# ----------------------------------------------------------------------------- the oracle gates with the mode on
@pytest.mark.parametrize("check", [
    lambda g: curkd_t.test_curkd_hidden_matches_reference(g, "curkd_ep0"),
    lambda g: w768_t.test_align_mse_768_matches_oracle(37, "f32"),
    lambda g: w768_t.test_align_mse_768_matches_oracle(512, "bf16"),
    lambda g: diffkd_t.test_diffkd_matches_reference(),
    lambda g: wass_t.test_wass_l1_matches_reference(g),
    lambda g: w768_t.test_wass_l1_768_matches_oracle(37),
    lambda g: sinkhorn_t.test_wass_sinkhorn_matches_reference(g),
    lambda g: mgd_t.test_masked_generation_matches_reference(g, "mgd_r05"),
    lambda g: mgd_t.test_masked_generation_matches_reference(g, "vitkd"),
    lambda g: mgd_t.test_generation_shapes_and_modes(7, 0.9, "bf16x3"),
    lambda g: mgd_t.test_generation_shapes_and_modes(4, 0.25, "bf16"),
    lambda g: lrkd_t.test_lrkd_matches_oracle_sign_aligned(g, "lrkd_r32"),
], ids=["align_mse", "align_mse_768", "align_mse_768_b512_bf16", "align_nmse", "wass_l1", "wass_l1_768", "wass_sinkhorn",
        "mgd", "vitkd", "mgd_f32_b7", "mgd_bf16", "lrkd"])
def test_oracle_with_mode_on(golden, check):
    with deterministic():
        check(golden)


# ----------------------------------------------------------------------------- repeated calls
def _align_call(entry, Dt, dtype, B=37, layers=(0, 1)):
    from deltakd_b200 import functional as Fn
    s_feats, t_feats = synth.make_features(B, 29, layers=layers, teacher_dim=Dt,
                                           **(dict(scale=0.5, t_shift=0.1) if entry == "sinkhorn" else {}))
    torch.manual_seed(1)
    lins = [torch.nn.Linear(192, Dt).cuda() for _ in layers]
    s_dev = [s_feats[i].to(dtype).cuda() for i in layers]
    t = [t_feats[i].to(dtype).cuda() for i in layers]

    def run():   # device work only, so that it can be captured in a CUDA graph
        s = [x.clone().requires_grad_(True) for x in s_dev]
        for lin in lins:
            lin.zero_grad(set_to_none=True)
        if entry == "mse":
            loss = Fn.align_mse_layers_loss(s, t, lins, scale=1e-3)
        elif entry == "nmse":
            loss = Fn.align_normalized_mse_loss(s, t, lins)
        elif entry == "l1":
            loss = Fn.wass_l1_loss(s, t, lins)
        else:
            loss = Fn.wass_sinkhorn_loss(s, t, lins)
        loss.backward()
        torch.cuda.synchronize()
        return [loss.detach().clone()] + [x.grad for x in s] + [p.grad for lin in lins for p in (lin.weight, lin.bias)]
    return run


def _mgd_call(B, dtype, seed=5):
    """masked_generation_loss with seeded heads, inputs and mask; returns a closure giving [loss, g_s, every head grad]."""
    from deltakd_b200 import functional as Fn
    g = torch.Generator().manual_seed(seed)
    s = (torch.randn(B, 197, 192, generator=g)).to(dtype).cuda()
    t = (torch.randn(B, 198, 384, generator=g)).to(dtype).cuda()
    mask = (torch.rand(B, 196, generator=g) < 0.5).float().cuda()
    torch.manual_seed(seed)
    align = torch.nn.Linear(192, 384).cuda()
    gen = torch.nn.Sequential(torch.nn.Conv2d(384, 384, 3, padding=1), torch.nn.ReLU(),
                              torch.nn.Conv2d(384, 384, 3, padding=1)).cuda()
    mask_token = torch.nn.Parameter(torch.randn(1, 1, 384, device="cuda") * 0.1)
    params = [align.weight, align.bias, mask_token, gen[0].weight, gen[0].bias, gen[2].weight, gen[2].bias]

    def run():
        sc = s.clone().requires_grad_(True)
        for p in params:
            p.grad = None
        loss = Fn.masked_generation_loss(sc, t, align, mask_token, gen, scale=7e-5 / (B * 196 * 384), mask=mask)
        loss.backward()
        torch.cuda.synchronize()
        return [loss.detach().clone(), sc.grad] + [p.grad for p in params]
    return run


def _lrkd_call(B=3, dtype=torch.float32, rank=32):
    from deltakd_b200 import functional as Fn
    s_feats, t_feats = synth.make_features(B, 31, layers=(0, 1, 11))
    torch.manual_seed(2)
    lins = [torch.nn.Linear(192, rank).cuda() for _ in range(3)]
    s_dev = [s_feats[i].to(dtype).cuda() for i in (0, 1, 11)]
    t = [t_feats[i].to(dtype).cuda() for i in (0, 1, 11)]

    def run():
        s = [x.clone().requires_grad_(True) for x in s_dev]
        for lin in lins:
            lin.zero_grad(set_to_none=True)
        loss = Fn.lrkd_layers_loss(s, t, lins, rank, (0.1, 0.2, 0.3))
        loss.backward()
        torch.cuda.synchronize()
        return [loss.detach().clone()] + [x.grad for x in s] + [p.grad for lin in lins for p in (lin.weight, lin.bias)]
    return run


CALLS = {
    "align_mse_384": lambda: _align_call("mse", 384, torch.float32),
    "align_mse_768": lambda: _align_call("mse", 768, torch.float32),
    "align_mse_384_bf16": lambda: _align_call("mse", 384, torch.bfloat16),
    "align_nmse": lambda: _align_call("nmse", 384, torch.float32),
    "wass_l1_384": lambda: _align_call("l1", 384, torch.float32),
    "wass_l1_768": lambda: _align_call("l1", 768, torch.float32),
    "wass_sinkhorn": lambda: _align_call("sinkhorn", 384, torch.float32, B=5),
    "mgd_f32": lambda: _mgd_call(6, torch.float32),
    "mgd_bf16": lambda: _mgd_call(6, torch.bfloat16),
    "mgd_f32_b512": lambda: _mgd_call(512, torch.float32),
    "lrkd": lambda: _lrkd_call(),
    # ranks that are not a multiple of 4: the per-split slots of rank * (Ds + 1) floats are padded to 128-byte boundaries
    "lrkd_rank10": lambda: _lrkd_call(B=37, rank=10),
    "lrkd_rank30_bf16": lambda: _lrkd_call(B=37, dtype=torch.bfloat16, rank=30),
}


@pytest.mark.parametrize("name", list(CALLS))
def test_repeated_calls_are_bit_identical(name):
    run = CALLS[name]()
    with deterministic():
        first = [x.clone() for x in run()]
        second = run()
    _equal(first, second, name)


@pytest.mark.parametrize("rank", [7, 10, 30, 33])
def test_lrkd_any_rank_matches_default_mode(rank):
    """Deterministic LRKD head gradients at ranks whose slots are not a whole number of 16-byte vectors equal the default
    (atomic) mode up to the order of the adds; loss and g_s are computed identically in both modes."""
    from oracle.util import rel_err
    run = _lrkd_call(B=37, rank=rank)
    default = [x.clone() for x in run()]
    with deterministic():
        det = run()
    _equal(default[:4], det[:4], "loss and g_s")
    for a, b in zip(default[4:], det[4:]):
        assert rel_err(b.double(), a.double()) < 1e-5


# ----------------------------------------------------------------------------- layer streams, concurrent load, graphs
@pytest.mark.parametrize("entry,Dt", [("mse", 384), ("mse", 768), ("l1", 384), ("nmse", 384)])
def test_layer_streams_give_identical_weight_gradients(entry, Dt, monkeypatch):
    from deltakd_b200 import functional as Fn
    run = _align_call(entry, Dt, torch.float32, B=21, layers=(0, 1, 2))
    with deterministic():
        monkeypatch.setattr(Fn, "_LAYER_STREAMS", True)
        multi = [x.clone() for x in run()]
        monkeypatch.setattr(Fn, "_LAYER_STREAMS", False)
        single = run()
    _equal(multi[4:], single[4:], "head gradients")   # [loss, 3 x g_s, 3 x (g_W, g_b)]
    _equal(multi[1:4], single[1:4], "g_s")


@pytest.mark.parametrize("name", ["mgd_f32", "align_mse_384", "lrkd"])
def test_concurrent_load_on_another_stream(name):
    """A call made while another stream runs a large masked-generation call equals the isolated call bit for bit."""
    run = CALLS[name]()
    side = torch.cuda.Stream()
    with deterministic():
        alone = [x.clone() for x in run()]
        _enqueue_mgd(side)   # warm: the side stream's scratch allocated
        torch.cuda.synchronize()
        busy = _enqueue_mgd(side)
        loaded = run()       # on the calling stream while `side` runs
        torch.cuda.synchronize()
        del busy
    _equal(alone, loaded, name)


def _enqueue_mgd(stream):
    """Enqueue one B = 384 masked-generation forward + backward on `stream` without synchronising."""
    from deltakd_b200 import functional as Fn
    B = 384
    g = torch.Generator().manual_seed(11)
    s = torch.randn(B, 197, 192, generator=g).cuda().requires_grad_(True)
    t = torch.randn(B, 198, 384, generator=g).cuda()
    mask = (torch.rand(B, 196, generator=g) < 0.5).float().cuda()
    align = torch.nn.Linear(192, 384).cuda()
    gen = torch.nn.Sequential(torch.nn.Conv2d(384, 384, 3, padding=1), torch.nn.ReLU(),
                              torch.nn.Conv2d(384, 384, 3, padding=1)).cuda()
    mask_token = torch.nn.Parameter(torch.zeros(1, 1, 384, device="cuda"))
    torch.cuda.current_stream().synchronize()
    with torch.cuda.stream(stream):
        loss = Fn.masked_generation_loss(s, t, align, mask_token, gen, scale=1e-6, mask=mask)
        loss.backward()
    return loss, s, align, gen, mask_token


@pytest.mark.parametrize("name", ["mgd_f32", "align_mse_384", "wass_l1_768", "lrkd"])
def test_graph_replay_equals_eager(name):
    run = CALLS[name]()
    with deterministic():
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
            _equal(eager, outs, name)


# ----------------------------------------------------------------------------- fresh process
_CHILD = """
import sys, torch
sys.path.insert(0, {root!r})
from tests.test_deterministic_gpu import _mgd_call, deterministic
run = _mgd_call(6, torch.float32)
with deterministic("cudnn"):
    out = run()
torch.save([x.cpu() for x in out], {path!r})
"""


def test_fresh_process_gives_the_same_bits(tmp_path):
    path = str(tmp_path / "mgd.pt")
    r = subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT, path=path)], cwd=ROOT, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    child = torch.load(path)
    with deterministic("cudnn"):
        here = [x.cpu() for x in _mgd_call(6, torch.float32)()]
    _equal(here, child, "subprocess vs in-process")


# ----------------------------------------------------------------------------- DistillationLoss end to end
def _e2e_step(c):
    from deltakd_b200 import DistillationLoss, call_base_loss
    crit = DistillationLoss(call_base_loss(c.args), c.teacher, c.kind, c.alpha, c.tau)
    torch.manual_seed(4321)   # the same random masks in both steps
    loss = crit(torch.zeros(c.B, 3, 2, 2, device="cuda"), c.outputs, c.student, c.s_feats, c.labels, c.args)
    loss.backward()
    torch.cuda.synchronize()
    heads = H.head_tensors(c.student)
    out = {k: p.grad.clone() for k, p in heads.items() if p.grad is not None}
    out.update({f"s{i}": f.grad.clone() for i, f in enumerate(c.s_feats) if f is not None and f.grad is not None})
    for p in c.student.parameters():
        p.grad = None
    for f in c.s_feats:
        if f is not None:
            f.grad = None
    return loss.item(), out


@pytest.mark.parametrize("name", ["curkd_ep0", "curkd_ep120", "curkd_ep200", "mgd_r05", "mgd_b512", "salmgd_m1", "vitkd",
                                  "lrkd_r32", "wass_l1", "wass_sinkhorn"])
def test_distillation_loss_steps_are_bit_identical(name):
    from tests import cases
    extra = {"mgd_b512": ("mgd", cases.A(), 512, 100, {})}   # mgd_r05 at B = 512
    with mock.patch.dict(cases.CASES, extra):
        c = build_case(name, device="cuda")
    with deterministic("cudnn"):
        l1, g1 = _e2e_step(c)
        l2, g2 = _e2e_step(c)
    assert l1 == l2
    assert set(g1) == set(g2) and len(g1) >= 2
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


def test_diffkd_steps_are_bit_identical():
    """The alignment head of the DiffKD branch (its denoise_fn runs through torch, outside the library)."""
    from tests.test_oracle_diffkd import diffkd_case
    c = diffkd_case(torch.float32, "cuda")
    grads = []
    with deterministic("cudnn"):
        for _ in range(2):
            diffkd_t._run_ours(c)
            heads = H.head_tensors(c.student)
            grads.append({k: p.grad.clone() for k, p in heads.items() if k.startswith("align") and p.grad is not None})
            for p in c.student.parameters():
                p.grad = None
            for f in c.s_feats:
                if f is not None:
                    f.grad = None
    assert len(grads[0]) >= 2
    for k in grads[0]:
        assert torch.equal(grads[0][k], grads[1][k]), k


@pytest.mark.parametrize("kind,args", [("curkd", dict(current_epoch=0)), ("curkd", dict(current_epoch=120)),
                                       ("wasskd", dict(wasskd_type="l1"))])
def test_distillation_loss_768_steps_are_bit_identical(kind, args):
    c = w768_t._case(kind, **args)
    outs = []
    with deterministic("cudnn"):
        for _ in range(2):
            loss = w768_t._criterion_loss(c)
            loss.backward()
            torch.cuda.synchronize()
            heads = H.head_tensors(c.student)
            outs.append((loss.item(), {k: p.grad.clone() for k, p in heads.items() if p.grad is not None}))
            for p in c.student.parameters():
                p.grad = None
    assert outs[0][0] == outs[1][0] and len(outs[0][1]) >= 2
    for k in outs[0][1]:
        assert torch.equal(outs[0][1][k], outs[1][1][k]), k


# ----------------------------------------------------------------------------- flag selection (fold kernels in the trace)
def _kernel_names(run):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    return {e.key for e in prof.key_averages()}


@pytest.mark.parametrize("flag", ["torch", "cudnn", None])
def test_flags_select_the_fold_kernels(flag):
    mgd = _mgd_call(4, torch.float32)
    align = _align_call("mse", 384, torch.float32, B=3)
    mgd(), align()   # warm
    ctx = deterministic(flag) if flag else contextlib.nullcontext()
    with ctx:
        names = _kernel_names(lambda: (mgd(), align()))
    folds = [n for n in names if "fold_splits_kernel" in n or "fold_rows_kernel" in n]
    if flag:
        assert any("fold_splits_kernel" in n for n in folds) and any("fold_rows_kernel" in n for n in folds), sorted(names)
    else:
        assert not folds, folds
    assert any("conv_wgrad_transpose_kernel" in n for n in names)


# ----------------------------------------------------------------------------- C ABI
def test_abi_flag_bits():
    from deltakd_b200 import _lib
    lib = _lib.lib
    DET = _lib.PREC_DETERMINISTIC
    for base in (_lib.PREC_BF16, _lib.PREC_BF16X3):
        for B in (1, 37, 512):
            for fn in ("dkd_align_mse", "dkd_align_nmse", "dkd_wass_l1", "dkd_wass_sinkhorn", "dkd_masked_generation"):
                for Dt in ((384, 768) if fn in ("dkd_align_mse", "dkd_wass_l1") else (384,)):
                    ws = getattr(lib, fn + "_workspace_bytes")
                    assert ws(B, 196, 192, Dt, base | DET) >= ws(B, 196, 192, Dt, base), (fn, B, Dt)
            assert lib.dkd_lrkd_workspace_bytes(3, B, 196, 192, 384, 32, _lib.F32, base | DET) >= \
                lib.dkd_lrkd_workspace_bytes(3, B, 196, 192, 384, 32, _lib.F32, base)
            assert lib.dkd_masked_generation_hidden_offset(B, 196, 192, 384, base | DET) == \
                lib.dkd_masked_generation_hidden_offset(B, 196, 192, 384, base)

    # unknown bits are rejected before anything is launched
    B = 2
    s = torch.zeros(B, 197, 192, device="cuda")
    t = torch.zeros(B, 198, 384, device="cuda")
    W = torch.zeros(384, 192, device="cuda")
    loss = torch.zeros(1, device="cuda")
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    for prec in (0x200, 0x101 | 0x400, 2, 2 | DET):
        nbytes = lib.dkd_align_mse_workspace_bytes(B, 196, 192, 384, 1 | DET)
        ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device="cuda")
        wp = ctypes.c_void_p(ws.data_ptr() + (-ws.data_ptr()) % 1024)
        rc = lib.dkd_align_mse_fwdbwd(p(s), p(t), p(W), None, B, 197, 1, 198, 2, 196, 192, 384, _lib.F32, prec, 1.0,
                                      None, None, None, p(loss), wp, nbytes, None)
        assert rc == -7, (prec, rc)   # DKD_E_UNSUPPORTED
    for prec in (1, 1 | DET):
        rc = lib.dkd_align_mse_fwdbwd(p(s), p(t), p(W), None, B, 197, 1, 198, 2, 196, 192, 384, _lib.F32, prec, 1.0,
                                      None, None, None, p(loss), wp, nbytes, None)
        assert rc == 0, (prec, _lib.last_error())
    torch.cuda.synchronize()
