"""Per-layer time of the two feature entry points that take a DeiT-Base teacher, at both teacher widths.

    python tools/teacher_width_bench.py [--B 512] [--iters 20] [--out profiles/teacher_width_768.json]

For op in (dkd_align_mse_fwdbwd, dkd_wass_l1_fwdbwd) x Dt in (384, 768) x I/O in (fp32 -> bf16x3, bf16 -> bf16) it
times one layer's forward + backward (loss, g_s, g_W, g_b) through the C ABI at B samples of 196 patch tokens.  Each
configuration is one CUDA graph that calls the entry point once per input set, over rotating input sets that together
exceed the 126 MB L2; the graph is replayed `iters` times between CUDA events and the time per call is reported.

Roofline per layer (M = B * 196 rows): algorithmic bytes M * (Ds + Dt + Ds) * elt (read s and t, write g_s), FLOPs
3 * 2 * M * Ds * Dt (forward, dgrad, wgrad; bf16x3's three passes count once), against the measured peaks of this
project (HBM 6 548.5 GB/s copy, bf16 1 404 TFLOP/s sustained); the larger of the two lower bounds names the bound.
The card's name and power limit are read once with `nvidia-smi --query-gpu` in the same run (nothing is changed).
Writes one JSON file; needs a B200.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deltakd_b200 import _lib  # noqa: E402

HBM_GBS, BF16_TFLOPS = 6548.5, 1404.0
L2_BYTES = 126 * 2 ** 20
DS, TS, TT = 192, 197, 198


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


def run(entry: str, Dt: int, dtype: torch.dtype, B: int, iters: int) -> dict:
    dev = torch.device("cuda")
    prec = _lib.PREC_BF16X3 if dtype == torch.float32 else _lib.PREC_BF16
    dcode = _lib.F32 if dtype == torch.float32 else _lib.BF16
    elt = torch.finfo(dtype).bits // 8
    n_tok = TS - 1
    M = B * n_tok
    set_bytes = B * (TS * DS * 2 + TT * Dt) * elt           # s, g_s, t
    n_sets = max(2, -(-2 * L2_BYTES // set_bytes))
    g = torch.Generator(device=dev).manual_seed(Dt)
    sets = []
    for _ in range(n_sets):
        s = torch.randn(B, TS, DS, device=dev, generator=g).to(dtype)
        t = torch.randn(B, TT, Dt, device=dev, generator=g).to(dtype)
        sets.append((s, t, torch.empty_like(s)))
    W = torch.randn(Dt, DS, device=dev, generator=g) * DS ** -0.5
    bias = torch.zeros(Dt, device=dev)
    gW, gb = torch.empty_like(W), torch.empty_like(bias)
    loss = torch.zeros((), device=dev)
    nbytes = getattr(_lib.lib, entry + "_workspace_bytes")(B, n_tok, DS, Dt, prec)
    ws_raw = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
    ws = ws_raw[(-ws_raw.data_ptr()) % 1024:][:nbytes]
    stream = torch.cuda.Stream()

    def calls():
        for s, t, gs in sets:
            _lib.call(entry + "_fwdbwd", s.data_ptr(), t.data_ptr(), W.data_ptr(), bias.data_ptr(), B, TS, 1, TT, 2, n_tok,
                      DS, Dt, dcode, prec, 1e-4, gs.data_ptr(), gW.data_ptr(), gb.data_ptr(), loss.data_ptr(),
                      ws.data_ptr(), ws.numel(), stream.cuda_stream)

    with torch.cuda.stream(stream):
        calls()                                           # warm-up: module load, cluster occupancy query
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        calls()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (iters * n_sets)
    alg_bytes = M * (DS + Dt + DS) * elt
    flops = 3 * 2 * M * DS * Dt
    t_hbm = alg_bytes / (HBM_GBS * 1e9) * 1e6
    t_tc = flops / (BF16_TFLOPS * 1e12) * 1e6
    bound = "hbm" if t_hbm >= t_tc else "tensor"
    del sets, ws_raw, graph
    torch.cuda.empty_cache()
    return dict(entry=entry, Dt=Dt, io=str(dtype).replace("torch.", ""), precision="bf16x3" if prec == _lib.PREC_BF16X3 else "bf16",
                B=B, M=M, us_per_layer=round(us, 2), algorithmic_bytes=alg_bytes, flops=flops,
                roofline_us=round(max(t_hbm, t_tc), 2), bound=bound, frac=round(max(t_hbm, t_tc) / us, 3),
                gbs=round(alg_bytes / us / 1e3, 1), tflops=round(flops / us / 1e6, 1), input_sets=n_sets, replays=iters)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "teacher_width_768.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("teacher_width_bench: needs a CUDA device (no CPU timing is meaningful)")
    res = dict(card=card(), peaks=dict(hbm_gbs=HBM_GBS, bf16_tflops_sustained=BF16_TFLOPS), rows=[])
    for entry in ("dkd_align_mse", "dkd_wass_l1"):
        for dtype in (torch.float32, torch.bfloat16):
            for Dt in (384, 768):
                r = run(entry, Dt, dtype, a.B, a.iters)
                res["rows"].append(r)
                print(json.dumps(r), flush=True)
    for entry in ("dkd_align_mse", "dkd_wass_l1"):
        for io in ("float32", "bfloat16"):
            t = {r["Dt"]: r["us_per_layer"] for r in res["rows"] if r["entry"] == entry and r["io"] == io}
            res.setdefault("ratio_768_over_384", {})[f"{entry}/{io}"] = round(t[768] / t[384], 3)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(dict(card=res["card"], ratio_768_over_384=res["ratio_768_over_384"])))


if __name__ == "__main__":
    main()
