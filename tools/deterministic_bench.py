"""Cost of the deterministic mode of the feature losses, and the default mode against a parent build.

    python tools/deterministic_bench.py [--B 512] [--iters 30] [--reps 5] [--parent-lib PATH]
                                        [--out profiles/deterministic_mode.json]

For each gradient-bearing feature entry point (align_mse at Dt = 384 and 768, align_nmse, wass_l1 at 384 and 768,
wass_sinkhorn, masked generation, LRKD with rank 32) and both I/O types (fp32 -> bf16x3, bf16 -> bf16) it times one
layer's forward + backward through `functional` (loss, g_s and every head gradient) at B samples of 196 patch tokens,
with the mode off and on (torch.backends.cudnn.deterministic), alternated `reps` times in this one process; each time is
CUDA events around `iters` calls after a warm-up.  With --parent-lib (a libdeltakd_sm100.so built from the parent
commit) the default mode is also timed with that library, alternated with this build, and the loss and g_s of one
default-mode call of each build are compared bit for bit (the head gradients are not: the default mode adds them with
float atomics, so they differ in the last bits from call to call of either build).  --breakdown adds, per I/O type,
the per-kernel CUDA time of the masked-generation call with the mode off and on, and off with the parent library
(torch.profiler, 5 calls each): at B = 512 that call spends a large share of its wall time between kernels.  Per-layer fp32 inputs exceed the 126 MB L2 except for LRKD's; bf16 inputs of the alignment losses are
about 115 MB.  The card's name and power limit are read with `nvidia-smi --query-gpu` in the same run (nothing is
changed).  Writes one JSON file; needs a B200.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deltakd_b200 import _lib  # noqa: E402
from deltakd_b200 import functional as Fn  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}
    dev = torch.cuda.current_device()
    row = [x.strip() for x in out[dev].split(",")] if len(out) > dev else []
    return dict(zip(q.split(","), row))


def make_call(op: str, Dt: int, dtype: torch.dtype, B: int):
    """A closure running one layer's forward + backward of `op` on seeded device inputs."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(Dt)
    s = torch.randn(B, 197, 192, device=dev, generator=g).to(dtype)
    t = torch.randn(B, 198, Dt, device=dev, generator=g).to(dtype)
    torch.manual_seed(0)
    if op == "masked_generation":
        align = torch.nn.Linear(192, Dt).cuda()
        gen = torch.nn.Sequential(torch.nn.Conv2d(Dt, Dt, 3, padding=1), torch.nn.ReLU(),
                                  torch.nn.Conv2d(Dt, Dt, 3, padding=1)).cuda()
        tok = torch.nn.Parameter(torch.zeros(1, 1, Dt, device=dev))
        mask = (torch.rand(B, 196, device=dev, generator=g) < 0.5).float()
        params = [*align.parameters(), *gen.parameters(), tok]
        fwd = lambda x: Fn.masked_generation_loss(x, t, align, tok, gen, scale=1e-6, mask=mask)
    else:
        lin = torch.nn.Linear(192, 32 if op == "lrkd" else Dt).cuda()
        params = list(lin.parameters())
        fwd = {
            "align_mse": lambda x: Fn.align_mse_layers_loss([x], [t], [lin], scale=1e-6),
            "align_nmse": lambda x: Fn.align_normalized_mse_loss([x], [t], [lin]),
            "wass_l1": lambda x: Fn.wass_l1_loss([x], [t], [lin]),
            "wass_sinkhorn": lambda x: Fn.wass_sinkhorn_loss([x], [t], [lin]),
            "lrkd": lambda x: Fn.lrkd_layers_loss([x], [t], [lin], 32, (0.1,)),
        }[op]

    def call():
        x = s.detach().requires_grad_(True)
        for p in params:
            p.grad = None
        loss = fwd(x)
        loss.backward()
        return loss.detach(), x.grad
    return call


def time_us(call, iters: int, deterministic: bool) -> float:
    # the mode is selected through cudnn.deterministic: torch.use_deterministic_algorithms(True) selects it too, but
    # also makes torch fill every new empty tensor (the gradient outputs) with NaN, a cost of torch's, not of the mode
    torch.backends.cudnn.deterministic = deterministic
    try:
        call()   # warm-up of this mode (scratch size, module load)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            call()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / iters
    finally:
        torch.backends.cudnn.deterministic = False


def load_parent(path: str):
    lib = ctypes.CDLL(path)
    for name, (res, args) in _lib.SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def breakdown(call, parent=None, calls: int = 5) -> dict:
    """{mode: {kernel name: CUDA time per call, us}} with the mode off and on, and off with the parent library if given."""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    ours = _lib.lib
    for mode in ("off", "on", "parent_off") if parent is not None else ("off", "on"):
        torch.backends.cudnn.deterministic = mode == "on"
        _lib.lib = parent if mode == "parent_off" else ours
        try:
            call()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(calls):
                    call()
                torch.cuda.synchronize()
        finally:
            torch.backends.cudnn.deterministic = False
            _lib.lib = ours
        rows = [(e.key, e.self_device_time_total / calls) for e in prof.key_averages() if e.self_device_time_total > 0]
        out[mode] = {k[:120]: round(v, 1) for k, v in sorted(rows, key=lambda r: -r[1])}
        out[mode + "_total"] = round(sum(v for _, v in rows), 1)
    return out


CASES = [("align_mse", 384), ("align_mse", 768), ("align_nmse", 384), ("wass_l1", 384), ("wass_l1", 768),
         ("wass_sinkhorn", 384), ("masked_generation", 384), ("lrkd", 384)]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--breakdown", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deterministic_mode.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_bench: needs a CUDA device (no CPU timing is meaningful)")
    ours = _lib.lib
    parent = load_parent(a.parent_lib) if a.parent_lib else None
    res = dict(card=card(), B=a.B, iters=a.iters, reps=a.reps, parent_lib=bool(parent), rows=[])
    warm = make_call("align_mse", 384, torch.float32, a.B)   # clocks up before the first timed case
    time_us(warm, 3 * a.iters, False)
    del warm
    for op, Dt in CASES:
        for dtype in (torch.float32, torch.bfloat16):
            call = make_call(op, Dt, dtype, a.B)
            t = {"off": [], "on": [], "parent_off": []}
            same = None
            if parent is not None:
                loss, gs = (x.clone() for x in call())
                _lib.lib = parent
                try:
                    ploss, pgs = call()
                finally:
                    _lib.lib = ours
                same = dict(loss=bool(torch.equal(loss, ploss)), g_s=bool(torch.equal(gs, pgs)))
            for _ in range(a.reps):
                t["off"].append(time_us(call, a.iters, False))
                t["on"].append(time_us(call, a.iters, True))
                if parent is not None:
                    _lib.lib = parent
                    try:
                        t["parent_off"].append(time_us(call, a.iters, False))
                    finally:
                        _lib.lib = ours
            med = {k: statistics.median(v) for k, v in t.items() if v}
            row = dict(op=op, Dt=Dt, io=str(dtype).replace("torch.", ""), us=({k: [round(x, 1) for x in v] for k, v in t.items() if v}),
                       median_us={k: round(v, 1) for k, v in med.items()}, on_over_off=round(med["on"] / med["off"], 4))
            if "parent_off" in med:
                row["off_over_parent"] = round(med["off"] / med["parent_off"], 4)
                row["parent_bit_identical"] = same
            res["rows"].append(row)
            print(json.dumps(row), flush=True)
            del call
            torch.cuda.empty_cache()
    if a.breakdown:
        res["masked_generation_kernels_us"] = {str(d).replace("torch.", ""): breakdown(make_call("masked_generation", 384, d, a.B), parent)
                                              for d in (torch.float32, torch.bfloat16)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(dict(card=res["card"])))


if __name__ == "__main__":
    main()
