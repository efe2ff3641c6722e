"""GPU: every logit-KD kernel variant the dispatcher (`dispatch_vec` -> `launch_logit_kd` in logit_kd.cu) can reach,
each against the fp64 oracle.

Each case of the table names the kernel family it is meant to reach and the vector width, and the op runs once under
torch.profiler: the launched kernel's name (template arguments <T, VEC, NV, THREADS, LK, KK>) and block shape must
match.  If a dispatch threshold moves, the case fails instead of silently testing another kernel.

Families: row128/nv{1,2,4} and row128/stream (one 128-thread CTA per row, the row in 1, 2 or 4 register chunks or
re-read), row64/nv{1,2,4} (64-thread rows for B >= 1024), ring/8warp and ring/anywarp (the persistent bulk-copy ring,
B >= 1024 and 16-byte aligned 1-4 KB rows), fold128 / fold1024 (the one-CTA launch that folds the row partials).
bf16 has no 2-wide kernel: a bf16 row that is not 8-byte aligned runs at VEC = 1.

Gates (as in test_logit_gpu.py): fp32 loss 1e-5 relative, gradients 1e-4 (norm-wise); bf16 against the oracle fed the
same bf16-rounded inputs, loss 1e-5, gradients 6e-3.
"""
from __future__ import annotations

import dataclasses
import json
import math
import os
import re
import tempfile
import zlib

import pytest
import torch

from oracle import losses as O
from oracle.step import mixup_target
from oracle.util import rel_err

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-5
GRAD_RTOL = 1e-4
BF16_LOSS_RTOL = 1e-5
BF16_GRAD_RTOL = 6e-3

DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16}
LK = {"soft": 0, "int": 1, "mix": 1, None: -1}
KK = {"none": 0, "soft": 1, "hard": 2}
RUNTIME_MODE = (-2, -2)
MODES = [("soft", "none"), ("int", "none"), ("soft", "soft"), ("int", "soft"), ("soft", "hard"), ("int", "hard"),
         (None, "soft"), (None, "hard")]   # the six compiled (label_kind, kd_kind) modes, then KD-only soft / hard


@dataclasses.dataclass(frozen=True)
class Case:
    dt: str                 # "f32" | "bf16"
    B: int
    C: int
    labels: str | None      # "soft" (float targets) | "int" | "mix" (int + mix_lam) | None (KD-only)
    kd: str                 # "none" | "soft" | "hard"
    fam: str                # expected kernel family
    vec: int                # expected vector width
    off: tuple = ()         # ((operand, element offset), ...): operand is a view buf[k:k + B*C] of a larger buffer
    alpha: float = 0.3
    tau: float = 2.5
    smoothing: float = 0.1
    lam: float | None = None
    frozen: str | None = None   # "z" | "zk": that logit tensor does not require grad

    @property
    def id(self):
        s = f"{self.dt}-B{self.B}-C{self.C}-{self.labels}-{self.kd}-{self.fam}-v{self.vec}"
        for k, v in self.off:
            s += f"-{k}+{v}"
        if self.lam is not None:
            s += f"-lam{self.lam}"
        if self.frozen:
            s += f"-frozen_{self.frozen}"
        if (self.alpha, self.tau, self.smoothing) != (0.3, 2.5, 0.1):
            s += f"-a{self.alpha}-t{self.tau}-s{self.smoothing}"
        return s

    @property
    def fold(self):
        return {"row128": "fold128", "row64": "fold1024", "ring": None}[self.fam.split("/")[0]]

    @property
    def mode(self):
        """(LK, KK) template arguments: the six modes are compiled for 16-byte vectors of the register kernels and the
        ring; everything else runs the runtime-mode instantiation."""
        lk, kk = LK[self.labels], KK[self.kd]
        elt = 2 if self.dt == "bf16" else 4
        if self.fam.startswith("ring") or (lk >= 0 and "stream" not in self.fam and self.vec * elt == 16):
            return (lk, kk)
        return RUNTIME_MODE


# --------------------------------------------------------------------------- which kernel ran
_NAME = re.compile(r"(logit_kd_kernel|logit_ring_kernel|logit_fold_small_kernel|logit_fold_kernel)\b(?:<([^>]*)>)?")


def _parse(name: str, args: dict):
    m = _NAME.search(name.replace("(int)", ""))
    if m is None:
        return None
    kern = m.group(1)
    if kern == "logit_fold_small_kernel":
        return {"fam": "fold128"}
    if kern == "logit_fold_kernel":
        return {"fam": "fold1024"}
    targs = [a.strip() for a in m.group(2).split(",")]
    dt = "bf16" if "bfloat16" in targs[0] else "f32"
    if kern == "logit_kd_kernel":
        vec, nv, threads, lk, kk = (int(a) for a in targs[1:6])
        fam = f"row{threads}/" + (f"nv{nv}" if nv else "stream")
        assert args["block"][0] == threads, (name, args["block"])
    else:
        vec, nv, lk, kk = (int(a) for a in targs[1:5])
        warps = args["block"][0] // 32
        fam = "ring/8warp" if warps == 8 else "ring/anywarp"
    return {"fam": fam, "dt": dt, "vec": vec, "nv": nv, "mode": (lk, kk)}


def profiled(fn):
    """Runs fn() once under torch.profiler (CUDA activity only); returns (fn's result, the logit kernels launched)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    ks = [_parse(e["name"], e.get("args", {})) for e in events if e.get("cat") == "kernel"]
    return out, [k for k in ks if k is not None]


OBSERVED: set = set()   # ("fam", family) / ("vec", family kind, dtype, VEC) / ("mode", family kind, LK, KK)


def _record(k):
    kind = k["fam"].split("/")[0]
    OBSERVED.add(("fam", k["fam"]))
    if "vec" in k:
        OBSERVED.add(("vec", "stream" if "stream" in k["fam"] else kind, k["dt"], k["vec"]))
        OBSERVED.add(("mode", kind, *k["mode"]))


def assert_launched(case: Case, kernels):
    rows = [k for k in kernels if "vec" in k]
    folds = [k for k in kernels if "vec" not in k]
    assert len(rows) == 1, kernels
    k = rows[0]
    got = (k["fam"], k["dt"], k["vec"], k["mode"])
    assert got == (case.fam, case.dt, case.vec, case.mode), (case.id, got)
    assert [f["fam"] for f in folds] == ([case.fold] if case.fold else []), (case.id, kernels)
    for x in kernels:
        _record(x)


# --------------------------------------------------------------------------- inputs, op, oracle
def _seed(tag: str) -> int:
    return zlib.crc32(tag.encode())


def make_inputs(case: Case):
    """CPU tensors (z, zk, zt, y), logits already rounded to the case's dtype."""
    g = torch.Generator().manual_seed(_seed(case.id))
    dt = DTYPES[case.dt]
    z, zk, zt = (torch.randn(case.B, case.C, generator=g).to(dt) for _ in range(3))
    if case.labels == "soft":
        y = torch.softmax(torch.randn(case.B, case.C, generator=g), -1).to(dt)
    elif case.labels in ("int", "mix"):
        y = torch.randint(0, case.C, (case.B,), generator=g)
    else:
        y = None
    return z, zk, zt, y


def _to_device(t, k):
    """t on the GPU as a contiguous view at element offset k of a larger buffer (k = 0: a plain copy)."""
    if not k:
        return t.cuda()
    buf = torch.zeros(k + t.numel() + 16, dtype=t.dtype, device="cuda")
    v = buf[k:k + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.storage_offset() == k
    return v


def run_op(case: Case, z, zk, zt, y):
    """Forward + backward of Fn.logit_kd_loss on the GPU: (total, parts[3], grad of z, grad of zk), all on the CPU."""
    from deltakd_b200 import functional as Fn
    off = dict(case.off)
    z, zk, zt = (_to_device(t, off.get(n, 0)) for n, t in (("z", z), ("zk", zk), ("zt", zt)))
    y = None if y is None else _to_device(y, off.get("y", 0))
    use_z, use_kd = case.labels is not None, case.kd != "none"
    if use_z and case.frozen != "z":
        z.requires_grad_(True)
    if use_kd and case.frozen != "zk":
        zk.requires_grad_(True)
    lam = None if case.lam is None else torch.tensor(case.lam, device="cuda")
    total, parts = Fn.logit_kd_loss(z if use_z else None, zk if use_kd else None, zt if use_kd else None, y,
                                    kd_kind=case.kd, smoothing=case.smoothing, alpha=case.alpha, tau=case.tau,
                                    return_parts=True, mix_lam=lam)
    total.backward()
    g = lambda t: None if t.grad is None else t.grad.float().cpu()
    return total.item(), parts.cpu().double(), g(z), g(zk)


def oracle(case: Case, z, zk, zt, y, dtype=torch.float64):
    """(total, [total, base, kd], grad z, grad zk) of the closed-form reference, computed in `dtype` on the CPU."""
    use_z, use_kd = case.labels is not None, case.kd != "none"
    z, zk, zt = (t.to(dtype) for t in (z, zk, zt))
    z.requires_grad_(use_z and case.frozen != "z")
    zk.requires_grad_(use_kd and case.frozen != "zk")
    if case.labels == "soft":
        y, base_kind = y.to(dtype), "soft_target"
    elif case.labels == "mix":
        y, base_kind = mixup_target(y, case.C, case.lam, case.smoothing).to(dtype), "soft_target"
    else:
        base_kind = "label_smoothing"
    zero = torch.zeros((), dtype=dtype)
    kd = {"none": lambda: zero, "soft": lambda: O.soft_kd(zk, zt, case.tau), "hard": lambda: O.hard_kd(zk, zt)}[case.kd]()
    if use_z:
        base = O.base_loss(z, y, base_kind, case.smoothing)
        args = O.default_args(smoothing=case.smoothing)
        total = O.distillation_loss(case.kd, (z, zk) if use_kd else z, y, zt, None, None, {}, args, case.alpha,
                                    case.tau, base_kind=base_kind)
    else:
        base, total = zero, kd * case.alpha
    total.backward()
    parts = torch.stack([total.detach(), base.detach(), kd.detach()]).double()
    g = lambda t: None if t.grad is None else t.grad.double()
    return total.item(), parts, g(z), g(zk)


def _close(got, ref, rtol):
    return abs(got - ref) <= rtol * abs(ref)


def assert_matches(case: Case, got, ref):
    lt, gt = (LOSS_RTOL, GRAD_RTOL) if case.dt == "f32" else (BF16_LOSS_RTOL, BF16_GRAD_RTOL)
    assert _close(got[0], ref[0], lt), (case.id, got[0], ref[0])
    for i, name in enumerate(("total", "base", "kd")):
        assert _close(float(got[1][i]), float(ref[1][i]), lt), (case.id, name, float(got[1][i]), float(ref[1][i]))
    for name, a, b in (("g_outputs", got[2], ref[2]), ("g_outputs_kd", got[3], ref[3])):
        assert (a is None) == (b is None), (case.id, name)
        if b is not None:
            assert torch.isfinite(a).all(), (case.id, name)
            assert rel_err(a, b) < gt, (case.id, name, rel_err(a, b))


def check_case(case: Case, inputs=None):
    inputs = make_inputs(case) if inputs is None else inputs
    got, kernels = profiled(lambda: run_op(case, *inputs))
    assert_launched(case, kernels)
    ref = oracle(case, *(t.double() if t is not None and t.is_floating_point() else t for t in inputs))
    assert_matches(case, got, ref)
    return got, ref


# --------------------------------------------------------------------------- the case table
def _paths():
    S = lambda dt, B, C, fam, vec, labels="soft", kd="soft": Case(dt, B, C, labels, kd, fam, vec)
    return [
        # bf16: 16-byte vectors are 8 wide; chunk = 1024 columns at 128 threads
        S("bf16", 8, 1024, "row128/nv1", 8), S("bf16", 8, 1032, "row128/nv2", 8),
        S("bf16", 37, 4096, "row128/nv4", 8), S("bf16", 4, 4104, "row128/stream", 8),
        S("bf16", 4, 4100, "row128/stream", 4), S("bf16", 3, 4099, "row128/stream", 1),
        S("bf16", 8, 508, "row128/nv1", 4), S("bf16", 8, 1020, "row128/nv2", 4), S("bf16", 8, 2044, "row128/nv4", 4),
        S("bf16", 8, 101, "row128/nv1", 1), S("bf16", 8, 250, "row128/nv2", 1), S("bf16", 8, 499, "row128/nv4", 1),
        S("bf16", 8, 1002, "row128/stream", 1),   # C = 2 mod 4: no 2-wide bf16 kernel
        S("bf16", 1023, 1000, "row128/nv1", 8), S("bf16", 1024, 1000, "ring/8warp", 8),
        S("bf16", 1025, 1000, "ring/8warp", 8),
        S("bf16", 1024, 504, "row64/nv1", 8),     # 1008-byte rows: too short for the ring
        S("bf16", 1025, 2000, "row64/nv4", 8, "int"), S("bf16", 1030, 2056, "row128/nv4", 8),
        S("bf16", 1024, 60, "row64/nv1", 4), S("bf16", 1024, 1004, "row64/nv4", 4),
        S("bf16", 1024, 126, "row64/nv2", 1), S("bf16", 1024, 250, "row64/nv4", 1),
        S("bf16", 1024, 1000, "row64/nv2", 8, None),   # KD-only: the ring has no label_kind -1 mode
        # fp32: 16-byte vectors are 4 wide; chunk = 512 columns at 128 threads
        S("f32", 8, 512, "row128/nv1", 4), S("f32", 8, 516, "row128/nv2", 4), S("f32", 256, 1000, "row128/nv2", 4),
        S("f32", 8, 2048, "row128/nv4", 4), S("f32", 8, 2052, "row128/stream", 4),
        S("f32", 8, 250, "row128/nv1", 2), S("f32", 8, 510, "row128/nv2", 2), S("f32", 8, 1002, "row128/nv4", 2),
        S("f32", 8, 1026, "row128/stream", 2),
        S("f32", 8, 127, "row128/nv1", 1), S("f32", 8, 255, "row128/nv2", 1), S("f32", 8, 511, "row128/nv4", 1),
        S("f32", 8, 1001, "row128/stream", 1),
        S("f32", 1023, 1000, "row128/nv2", 4), S("f32", 1024, 1000, "ring/anywarp", 4),
        S("f32", 2048, 512, "ring/8warp", 4), S("f32", 1024, 252, "row64/nv1", 4),   # 1025 x 1000 and 1024 x 104: in _modes
        S("f32", 1024, 1028, "row128/nv4", 4), S("f32", 1024, 4100, "row128/stream", 4),
        S("f32", 1024, 126, "row64/nv1", 2), S("f32", 1024, 250, "row64/nv2", 2), S("f32", 1024, 510, "row64/nv4", 2),
        S("f32", 1024, 63, "row64/nv1", 1), S("f32", 1024, 255, "row64/nv4", 1),
        S("f32", 1024, 500, "row64/nv2", 4, None), S("f32", 1024, 1000, "row64/nv4", 4, None, "hard"),
    ]


# fp32 rows of 4 KB: the ring's warp count follows the number of operand rows the mode stages (3 stages per warp)
_F32_C1000_RING = {("soft", "none"): "ring/8warp", ("int", "none"): "ring/8warp", ("soft", "soft"): "ring/anywarp",
                   ("int", "soft"): "ring/anywarp", ("soft", "hard"): "ring/anywarp", ("int", "hard"): "ring/anywarp"}


def _modes():
    shapes = [  # (dtype, B, C, family of the six modes, VEC, family of KD-only)
        ("bf16", 8, 1000, "row128/nv1", 8, "row128/nv1"), ("f32", 37, 1000, "row128/nv2", 4, "row128/nv2"),
        ("f32", 1024, 104, "row64/nv1", 4, "row64/nv1"), ("bf16", 1030, 504, "row64/nv1", 8, "row64/nv1"),
        ("bf16", 2048, 1000, "ring/8warp", 8, "row64/nv2"), ("f32", 1025, 1000, None, 4, "row64/nv4"),
    ]
    out = []
    for dt, B, C, fam, vec, fam_kd in shapes:
        for labels, kd in MODES:
            f = fam_kd if labels is None else (fam or _F32_C1000_RING[(labels, kd)])
            out.append(Case(dt, B, C, labels, kd, f, vec))
    return out


def _alignment():
    """Each operand on its own at an element offset that rules out the wider vectors."""
    out = []
    for op in ("z", "zk", "zt", "y"):
        out += [Case("f32", 8, 1000, "soft", "soft", "row128/nv4", 2, ((op, 2),)),
                Case("f32", 8, 1000, "soft", "soft", "row128/stream", 1, ((op, 1),)),
                Case("bf16", 8, 1000, "soft", "soft", "row128/nv2", 4, ((op, 4),)),
                Case("bf16", 8, 1000, "soft", "soft", "row128/stream", 1, ((op, 2),)),
                Case("f32", 2048, 512, "soft", "soft", "row64/nv4", 2, ((op, 2),)),      # a ring shape, unaligned
                Case("bf16", 2048, 1000, "soft", "soft", "row64/nv4", 4, ((op, 4),))]
    return out


def _mixed():
    out = []
    for dt in ("f32", "bf16"):
        for B in (8, 37, 2051):
            for kd in ("soft", "hard", "none"):
                for lam in (0.37, 1.0):
                    if B < 1024:
                        fam = "row128/nv2" if dt == "f32" else "row128/nv1"
                    else:
                        fam = _F32_C1000_RING[("int", kd)] if dt == "f32" else "ring/8warp"
                    out.append(Case(dt, B, 1000, "mix", kd, fam, 4 if dt == "f32" else 8, lam=lam))
    return out


def _one_grad():
    out = []
    for dt, B, C, fam, vec in (("f32", 8, 1000, "row128/nv2", 4), ("bf16", 8, 1000, "row128/nv1", 8),
                               ("f32", 2048, 512, "ring/8warp", 4), ("bf16", 2048, 1000, "ring/8warp", 8)):
        for labels, kd in (("soft", "soft"), ("int", "hard")):
            for frozen in ("z", "zk"):
                out.append(Case(dt, B, C, labels, kd, fam, vec, frozen=frozen))
    return out


def _hyper():
    out = []
    for dt, B, C, fam, vec, fam_kd in (("f32", 8, 1000, "row128/nv2", 4, "row128/nv2"),
                                       ("bf16", 2048, 1000, "ring/8warp", 8, "row64/nv2"),
                                       ("f32", 1024, 104, "row64/nv1", 4, "row64/nv1")):
        for labels, kd, kw in (("soft", "soft", dict(alpha=0.0)), ("int", "hard", dict(alpha=0.0)),
                               ("soft", "soft", dict(alpha=1.0)), ("int", "hard", dict(alpha=1.0)),
                               ("int", "soft", dict(smoothing=0.0)), ("int", "none", dict(smoothing=0.0)),
                               ("soft", "soft", dict(tau=0.5)), ("int", "soft", dict(tau=8.0)),
                               (None, "soft", dict(alpha=1.0)), (None, "soft", dict(alpha=0.0, tau=0.5)),
                               (None, "hard", dict(alpha=1.0))):
            out.append(Case(dt, B, C, labels, kd, fam_kd if labels is None else fam, vec, **kw))
    return out


TABLE = {"paths": _paths(), "modes": _modes(), "alignment": _alignment(), "mixed": _mixed(), "one_grad": _one_grad(),
         "hyper": _hyper()}
ALL_CASES = [c for cs in TABLE.values() for c in cs]

# what the dispatcher can reach: every family, the vector widths of each kind of kernel, and the compiled modes
REACHABLE = (
    {("fam", f) for f in ("row128/nv1", "row128/nv2", "row128/nv4", "row128/stream", "row64/nv1", "row64/nv2",
                          "row64/nv4", "ring/8warp", "ring/anywarp", "fold128", "fold1024")}
    | {("vec", kind, dt, v) for kind in ("row128", "row64", "stream") for dt, vs in (("f32", (4, 2, 1)), ("bf16", (8, 4, 1)))
       for v in vs}
    | {("vec", "ring", "f32", 4), ("vec", "ring", "bf16", 8)}
    | {("mode", kind, LK[lab], KK[kd]) for kind in ("row128", "row64", "ring") for lab, kd in MODES[:6]}
    | {("mode", kind, *RUNTIME_MODE) for kind in ("row128", "row64")}
)


@pytest.mark.parametrize("case", ALL_CASES, ids=lambda c: c.id)
def test_dispatch_case_matches_oracle(case):
    check_case(case)


# --------------------------------------------------------------------------- hard-KD ties placed per path
TIE_SHAPES = [  # (dtype, B, C, labels, family, VEC, threads per row)
    ("f32", 8, 1000, "soft", "row128/nv2", 4, 128), ("f32", 8, 1000, None, "row128/nv2", 4, 128),
    ("bf16", 8, 2000, "soft", "row128/nv2", 8, 128), ("bf16", 8, 2000, None, "row128/nv2", 8, 128),
    ("f32", 1024, 510, "soft", "row64/nv4", 2, 64), ("f32", 2048, 512, None, "row64/nv2", 4, 64),
    ("bf16", 1024, 2000, "soft", "row64/nv4", 8, 64), ("bf16", 2048, 1000, None, "row64/nv2", 8, 64),
    ("f32", 8, 2052, "soft", "row128/stream", 4, 128), ("bf16", 8, 4104, None, "row128/stream", 8, 128),
    ("f32", 2048, 512, "soft", "ring/8warp", 4, 32), ("bf16", 2048, 1000, "soft", "ring/8warp", 8, 32),
]


def _tie_rows(C, vec, threads):
    """Column sets of equal teacher maxima, one row each; the CE target is the first column of each set."""
    col = lambda it, tid, v=0: (it * threads + tid) * vec + v
    rows = [
        [col(0, 3, 0), col(1, 3, 0)],           # one lane, chunk 0 and chunk 1
        [col(0, 7, 0), col(1, 2, 0)],           # the lower index in the higher lane
        [col(0, 2, 0), C - 1],                  # a tie with the last column
        [C - 1],                                # the maximum at the last column alone
    ]
    if vec > 1:
        rows.append([col(0, 5, 1 if vec > 2 else 0), col(0, 5, vec - 1)])   # two slots of one thread's vector
    if threads > 32:
        rows.append([col(0, 40, 0), col(1, 1, 0)])   # the lower index in the higher warp
    return rows


@pytest.mark.parametrize("dt,B,C,labels,fam,vec,threads", TIE_SHAPES, ids=lambda v: str(v))
def test_hard_kd_first_max_ties(dt, B, C, labels, fam, vec, threads):
    """Equal teacher maxima placed where each kernel's argmax merges candidates (vector slots, chunks, lanes, warps, the
    row's end): the hard-KD target is the first maximal index, as torch.argmax.  Two more rows have -inf teacher
    classes (masked logits), which hard KD must handle finitely."""
    case = Case(dt, B, C, labels, "hard", fam, vec, alpha=0.5)
    z, zk, zt, y = make_inputs(case)
    ztf = zt.float().clamp(-4.5, 4.5)
    ties = _tie_rows(C, vec, threads)
    for r, cols in enumerate(ties):
        ztf[r, cols] = 6.0
    r = len(ties)
    ztf[r, ::3] = -math.inf                      # masked classes across the row, the maximum is finite
    ztf[r + 1, : C // 2] = -math.inf             # the whole first half (every lane's first chunk) masked
    zt = ztf.to(DTYPES[dt])
    got, ref = check_case(case, (z, zk, zt, y))
    assert math.isfinite(got[0]) and torch.isfinite(got[3]).all()
    first = torch.tensor([cols[0] for cols in ties])
    assert torch.equal(got[3][: len(ties)].argmin(1), first)           # the one-hot of the KD gradient
    assert torch.equal(ref[3][: len(ties)].argmin(1), first)


# --------------------------------------------------------------------------- logit scale, student near the teacher
@pytest.mark.parametrize("labels", ["soft", None])
@pytest.mark.parametrize("B", [256, 2048])
@pytest.mark.parametrize("tau", [1.0, 3.0])
@pytest.mark.parametrize("sigma,eps", [(3.0, 1.0), (3.0, 0.3), (10.0, 1.0), (10.0, 0.3)])
def test_soft_kd_at_trained_logit_scale(sigma, eps, tau, B, labels):
    """Teacher logits N(0, sigma^2), student = teacher + eps * N(0, 1), fp32: the row's KL is a small difference of
    terms of size max / tau.  The fp32 oracle itself misses 1e-5 here, so the gate is relative to it: the kernel's
    error against fp64 must stay within max(1e-5, 4 * e32) for the kd part and the totals (1e-4 for the gradients),
    where e32 is the error of the same oracle run in fp32."""
    fam = {(256, "soft"): "row128/nv2", (256, None): "row128/nv2", (2048, "soft"): "ring/anywarp",
           (2048, None): "row64/nv4"}[(B, labels)]
    case = Case("f32", B, 1000, labels, "soft", fam, 4, alpha=0.5, tau=tau)
    g = torch.Generator().manual_seed(_seed(case.id) + int(sigma * 10 + eps * 100))
    zt = torch.randn(B, 1000, generator=g) * sigma
    zk = zt + eps * torch.randn(B, 1000, generator=g)
    z = torch.randn(B, 1000, generator=g) * sigma
    y = torch.softmax(torch.randn(B, 1000, generator=g), -1) if labels else None
    got, kernels = profiled(lambda: run_op(case, z, zk, zt, y))
    assert_launched(case, kernels)
    d = lambda t: None if t is None else t.double()
    r64 = oracle(case, d(z), d(zk), d(zt), d(y))
    r32 = oracle(case, z, zk, zt, y, dtype=torch.float32)
    rel = lambda a, b: abs(float(a) - float(b)) / abs(float(b))
    for i in (0, 2):   # total and kd part
        e32 = rel(r32[1][i], r64[1][i])
        assert rel(got[1][i], r64[1][i]) <= max(LOSS_RTOL, 4 * e32), (i, float(got[1][i]), float(r64[1][i]), e32)
    if labels:
        assert rel(got[1][1], r64[1][1]) <= LOSS_RTOL
    else:
        assert float(got[1][1]) == 0.0
    for j in (2, 3):
        if r64[j] is not None:
            e32 = rel_err(r32[j], r64[j])
            assert rel_err(got[j], r64[j]) <= max(GRAD_RTOL, 4 * e32), (j, rel_err(got[j], r64[j]), e32)


# --------------------------------------------------------------------------- every family was seen
def test_table_covers_every_reachable_kernel():
    """The union over the table of the kernels seen in profiler traces covers every family, vector width and compiled
    mode the dispatcher can reach.  Cases not run in this session (a -k selection) are run here, launch check only."""
    for case in ALL_CASES:
        if REACHABLE <= OBSERVED:
            break
        _, kernels = profiled(lambda: run_op(case, *make_inputs(case)))
        assert_launched(case, kernels)
    missing = sorted(REACHABLE - OBSERVED, key=str)
    assert not missing, missing
