"""Time of the masked-generation core at both patch grids: 196 tokens (14 x 14, 224-px inputs) and 576 (24 x 24, 384 px).

    python tools/grid_bench.py [--B 512] [--iters 10] [--repeats 3] [--out profiles/grid_24.json]

For n_tok in (196, 576) x I/O in (fp32 -> bf16x3, bf16 -> bf16) it times one dkd_masked_generation_fwdbwd call (forward
+ every gradient: g_s, align W / b, mask_token, both convolutions' W / b) through the C ABI at B samples, half the
tokens masked.  Each configuration is one CUDA graph that calls the entry point once per input set, over rotating input
sets that together exceed the 126 MB L2; the graph is replayed `iters` times between CUDA events.  The two grids of one
I/O type are timed alternately `repeats` times and the median time per call is reported.

Roofline per call (M = B * n_tok rows): FLOPs = the six convolution GEMMs 6 * 2 * M * 3456 * 384 (forward, dgrad and
wgrad of both convolutions) + the three align GEMMs 3 * 2 * M * 192 * 384, bf16x3's three passes counted once, against
the measured peaks of this project (bf16 1 404 TFLOP/s sustained; HBM 6 548.5 GB/s copy for the algorithmic bytes:
read s, t and the mask, write g_s); the larger of the two lower bounds names the bound.  The workspace size is the
library's own figure (dkd_masked_generation_workspace_bytes).  The card's name and power limit are read once with
`nvidia-smi --query-gpu` in the same run (nothing is changed).  Writes one JSON file; needs a B200.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deltakd_b200 import _lib  # noqa: E402

HBM_GBS, BF16_TFLOPS = 6548.5, 1404.0
L2_BYTES = 126 * 2 ** 20
DS, DT = 192, 384


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


def roofline(B: int, n_tok: int, dtype: torch.dtype) -> dict:
    M = B * n_tok
    elt = torch.finfo(dtype).bits // 8
    flops = 6 * 2 * M * 9 * DT * DT + 3 * 2 * M * DS * DT
    alg_bytes = M * (2 * DS + DT) * elt + M * 4
    t_tc = flops / (BF16_TFLOPS * 1e12) * 1e6
    t_hbm = alg_bytes / (HBM_GBS * 1e9) * 1e6
    return dict(M=M, flops=flops, algorithmic_bytes=alg_bytes, roofline_us=round(max(t_tc, t_hbm), 2),
                bound="tensor" if t_tc >= t_hbm else "hbm")


class Config:
    """Inputs, parameters, gradients, workspace and the captured graph of one (n_tok, I/O) configuration."""

    def __init__(self, n_tok: int, dtype: torch.dtype, B: int):
        dev = torch.device("cuda")
        self.n_tok, self.dtype, self.B = n_tok, dtype, B
        self.prec = _lib.PREC_BF16X3 if dtype == torch.float32 else _lib.PREC_BF16
        dcode = _lib.F32 if dtype == torch.float32 else _lib.BF16
        elt = torch.finfo(dtype).bits // 8
        Ts, Tt = 1 + n_tok, 2 + n_tok
        set_bytes = B * (2 * Ts * DS + Tt * DT) * elt + B * n_tok * 4      # s, g_s, t, mask
        self.n_sets = max(2, -(-2 * L2_BYTES // set_bytes))
        g = torch.Generator(device=dev).manual_seed(n_tok)
        self.sets = []
        for _ in range(self.n_sets):
            s = torch.randn(B, Ts, DS, device=dev, generator=g).to(dtype)
            t = torch.randn(B, Tt, DT, device=dev, generator=g).to(dtype)
            mask = (torch.rand(B, n_tok, device=dev, generator=g) < 0.5).float()
            self.sets.append((s, t, mask, torch.empty_like(s)))
        p = dict(Wa=torch.randn(DT, DS, device=dev, generator=g) * DS ** -0.5, ba=torch.zeros(DT, device=dev),
                 mt=torch.randn(DT, device=dev, generator=g) * 0.1,
                 c1w=torch.randn(DT, DT, 3, 3, device=dev, generator=g) * (9 * DT) ** -0.5, c1b=torch.zeros(DT, device=dev),
                 c2w=torch.randn(DT, DT, 3, 3, device=dev, generator=g) * (9 * DT) ** -0.5, c2b=torch.zeros(DT, device=dev))
        self.params = p
        self.grads = {k: torch.empty_like(v) for k, v in p.items()}
        self.loss = torch.zeros((), device=dev)
        self.ws_bytes = _lib.lib.dkd_masked_generation_workspace_bytes(B, n_tok, DS, DT, self.prec)
        self.ws_raw = torch.empty(self.ws_bytes + 1024, dtype=torch.uint8, device=dev)
        ws = self.ws_raw[(-self.ws_raw.data_ptr()) % 1024:][:self.ws_bytes]
        self.stream = torch.cuda.Stream()
        gr = self.grads

        def calls():
            for s, t, mask, gs in self.sets:
                _lib.call("dkd_masked_generation_fwdbwd", s.data_ptr(), t.data_ptr(), mask.data_ptr(), p["Wa"].data_ptr(),
                          p["ba"].data_ptr(), p["mt"].data_ptr(), p["c1w"].data_ptr(), p["c1b"].data_ptr(), p["c2w"].data_ptr(),
                          p["c2b"].data_ptr(), B, Ts, 1, Tt, 2, DS, DT, dcode, self.prec, 1e-6, gs.data_ptr(),
                          gr["Wa"].data_ptr(), gr["ba"].data_ptr(), gr["mt"].data_ptr(), gr["c1w"].data_ptr(),
                          gr["c1b"].data_ptr(), gr["c2w"].data_ptr(), gr["c2b"].data_ptr(), self.loss.data_ptr(),
                          ws.data_ptr(), ws.numel(), self.stream.cuda_stream)

        with torch.cuda.stream(self.stream):
            calls()                                       # warm-up: module load, cluster occupancy query
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self.stream):
            calls()
        for _ in range(3):
            self.graph.replay()
        torch.cuda.synchronize()

    def time_us(self, iters: int) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            self.graph.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / (iters * self.n_sets)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "grid_24.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("grid_bench: needs a CUDA device (no CPU timing is meaningful)")
    res = dict(card=card(), peaks=dict(hbm_gbs=HBM_GBS, bf16_tflops_sustained=BF16_TFLOPS), B=a.B, rows=[])
    for dtype in (torch.float32, torch.bfloat16):
        cfgs = [Config(n, dtype, a.B) for n in (196, 576)]
        times = {c.n_tok: [] for c in cfgs}
        for _ in range(a.repeats):          # alternate the two grids
            for c in cfgs:
                times[c.n_tok].append(c.time_us(a.iters))
        for c in cfgs:
            us = statistics.median(times[c.n_tok])
            r = dict(n_tok=c.n_tok, io=str(dtype).replace("torch.", ""), precision="bf16x3" if c.prec == _lib.PREC_BF16X3 else "bf16",
                     B=a.B, us_per_call=round(us, 1), us_repeats=[round(x, 1) for x in times[c.n_tok]],
                     workspace_bytes=c.ws_bytes, input_sets=c.n_sets, replays=a.iters, **roofline(a.B, c.n_tok, dtype))
            r["frac"] = round(r["roofline_us"] / us, 3)
            r["tflops"] = round(r["flops"] / us / 1e6, 1)
            res["rows"].append(r)
            print(json.dumps(r), flush=True)
        del cfgs
        torch.cuda.empty_cache()
    for io in ("float32", "bfloat16"):
        t = {r["n_tok"]: r for r in res["rows"] if r["io"] == io}
        res.setdefault("ratio_576_over_196", {})[io] = dict(time=round(t[576]["us_per_call"] / t[196]["us_per_call"], 3),
                                                             frac=round(t[576]["frac"] / t[196]["frac"], 3))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(dict(card=res["card"], ratio_576_over_196=res["ratio_576_over_196"])))


if __name__ == "__main__":
    main()
