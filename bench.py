#!/usr/bin/env python
"""bench.py — DeltaKD distillation-loss hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--no-extras | --extras]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (loss forward + backward through
`deltakd_b200.DistillationLoss`) over one batch of synthetic teacher/student outputs.
Prints ONE JSON line (rank 0).  Keys follow the driver contract; see DESIGN.md §Measurement.

  value        samples/s, whole job, inputs resident in HBM, the step's launches replayed from a
               CUDA graph (no Python between launches); input sets rotate through > L2-size data
  e2e          same metric through the public API with HOST (pinned) inputs: per step H2D of the
               step's tensors, criterion(...) + backward, D2H read of the loss
  roofline     the fused loss op's kernels alone (the C-ABI call, replayed from a CUDA graph and timed
               with CUDA events): algorithmic bytes (or flops) per call / mean call duration
  cpu_baseline the CPU oracle (restatement of the reference's PyTorch loss, `kind: "port"`) timed on
               this box's host cores on a bounded sample of the same workload
  workloads    the other BASELINE.json configs (feature losses at their full batch sizes), each with
               value / e2e / roofline / cpu_baseline, measured the same way (single-GPU runs; skipped by --no-extras,
               forced under torchrun by --extras)
  --impl reference : the reference arm = the same CPU oracle with all host threads (the reference is
               pure PyTorch; /root/reference does not exist on the GPU box)
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

L2_BYTES = 126 * 1024 * 1024
METRIC = "distill-loss fwd+bwd samples/s"


def ncu_traffic():
    """workload -> {"bytes": dram__bytes_read.sum + dram__bytes_write.sum summed over every kernel one call of the fused op
    launches, "kernels": [...], "source": file}: written by tools/ncu_traffic.py from an `ncu` pass of
    `bench.py --ncu-op <workload>` on the final build (profiles/ncu_traffic.json).  Gradient / plane WRITES of the small
    workloads stay in the 126 MB L2 until evicted, so traffic can be below the algorithmic bytes."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except ValueError:
            return {}
    return {}


NCU_TRAFFIC = ncu_traffic()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sus=1400.0, src="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            atexit.register(self.close)   # a run that raises before stop() must not leave nvidia-smi polling
        except OSError:
            self.proc = None
        return self

    def close(self):
        """Ends nvidia-smi and reaps it, so that no process outlives the benchmark."""
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                self.proc.wait()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, windows):
        """windows: list of (t0, t1) wall-clock intervals of the timed regions."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.close()
        rows = [s for t, s in self.samples if any(t0 - 0.05 <= t <= t1 + 0.15 for t0, t1 in windows)]
        rows = rows or [s for _, s in self.samples[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _pin(t):
    return t.pin_memory() if torch.cuda.is_available() else t


# ----------------------------------------------------------------------------- workloads
class Workload:
    """One BASELINE.json config: builds inputs, the step, its algorithmic cost and the CPU oracle step."""
    name = ""
    dtype = "f32"
    B = 0
    bound = "hbm"
    cpu_B = None          # batch of the bounded CPU sample (None -> same as B)
    default_steps = 20

    def __init__(self, device, rank):
        self.device, self.rank = device, rank

    def nsets(self):
        """Rotating input sets so that the working set between reuses exceeds L2."""
        return max(1, int(1.5 * L2_BYTES / max(1, self.bytes_per_set())) + 1) if self.bytes_per_set() < 2 * L2_BYTES else 1

    def algorithmic_flops(self):
        return 0.0

    def input_leaves(self, ds):
        """(name, tensor) for each differentiable input of `step(ds)`."""
        return []

    def outputs(self, ds, loss):
        """name -> tensor: what a caller of `step(ds)` receives, i.e. the loss and the gradients of the differentiable
        inputs and of the student's parameters."""
        out = {"loss": loss.detach()}
        for n, x in self.input_leaves(ds):
            if x.grad is not None:
                out[f"grad_{n}"] = x.grad
        student = getattr(self, "student", None)
        if student is not None:
            for n, p in student.named_parameters():
                if p.grad is not None:
                    out[f"grad_student.{n}"] = p.grad
        return out

    # ---- parity gate: before anything is timed, the step's loss on a sub-batch is checked against the CPU oracle
    parity_rtol = 1e-5      # the north-star loss gate in fp32; bf16 workloads state 2e-2

    def slice_host(self, hs, n):
        raise NotImplementedError

    def parity(self):
        """{"batch", "loss", "oracle", "rel_err", "rtol", "ok"}: loss of one step through the public API on the first
        `cpu_B` samples of input set 0 against the fp32 oracle on the same samples (rank 0 only)."""
        Bc = min(self.cpu_B or self.B, self.B)
        hs = self.slice_host(self.host_sets(1, B=self.B)[0], Bc)
        full_B, self.B = self.B, Bc
        try:
            got = float(self.step(self.to_device(hs)).item())
        finally:
            self.B = full_B
        want = float(self.cpu_step(self.cpu_prepare(hs)).item())
        rel = abs(got - want) / max(abs(want), 1e-30)
        return {"batch": Bc, "loss": got, "oracle": want, "rel_err": rel, "rtol": self.parity_rtol, "ok": rel <= self.parity_rtol}


class LogitKD(Workload):
    """configs[1]: base SoftTargetCE + soft-KD (tau 3, alpha 0.1) on DeiT-Tiny logits, B=256, C=1000, bf16."""
    name = "soft_kd_logits_b256_c1000_bf16"
    dtype = "bf16"
    B, C, kind, alpha, tau = 256, 1000, "soft", 0.1, 3.0
    tdtype = torch.bfloat16
    dominant = "logit_kd_kernel"
    default_steps = 200

    def bytes_per_set(self):
        return 4 * self.B * self.C * self.tdtype.itemsize

    def algorithmic_bytes(self):  # 4 reads + 2 gradient writes (SURVEY §8d cfg2: 6*B*C*elt)
        return 6 * self.B * self.C * self.tdtype.itemsize

    def host_sets(self, n, B=None):
        """One pinned [4, B, C] buffer per set (outputs, outputs_kd, teacher logits, soft labels): a single H2D copy."""
        from deltakd_b200 import synth
        B = B or self.B
        sets = []
        for i in range(n):
            z, zk, zt, y = synth.make_logits(B, self.C, 1234 + self.rank + 17 * i)
            sets.append(_pin(torch.stack([z, zk, zt, y]).to(self.tdtype)))
        return sets

    def slice_host(self, hs, n):
        return hs[:, :n].contiguous()

    def setup(self):
        from deltakd_b200 import DistillationLoss, call_base_loss, synth
        self.args = synth.default_args()
        self.teacher = synth.FeatureReplayModel(384)
        self.crit = DistillationLoss(call_base_loss(self.args), self.teacher, self.kind, self.alpha, self.tau)
        self.inputs = torch.zeros(self.B, 3, 2, 2, device=self.device)  # images feed only the (replayed) teacher

    def to_device(self, hs, slot=None):
        """slot = None: fresh device tensors; slot = k: copy into the persistent device buffer k (the prefetching e2e loop)."""
        if slot is None:
            d = hs.to(self.device, non_blocking=True)
        else:
            slots = self.__dict__.setdefault("_slots", {})
            if slot not in slots or slots[slot].shape != hs.shape:
                slots[slot] = torch.empty_like(hs, device=self.device)
            d = slots[slot]
            d.copy_(hs, non_blocking=True)
        return d[0].requires_grad_(True), d[1].requires_grad_(True), d[2], d[3]

    def input_leaves(self, ds):
        return [("outputs", ds[0]), ("outputs_kd", ds[1])]

    def h2d_bytes(self):
        return self.bytes_per_set()

    def step(self, ds):
        z, zk, zt, y = ds
        self.teacher.set_outputs(zt, None)
        z.grad = zk.grad = None
        loss = self.crit(self.inputs if z.shape[0] == self.inputs.shape[0] else self.inputs[:z.shape[0]], (z, zk), None, None, y, self.args)
        loss.backward()
        return loss

    def op_only(self, ds):
        """Just the fused loss op through the C ABI (forward launch writes the gradients too)."""
        from deltakd_b200 import functional as Fn
        z, zk, zt, y = ds
        return Fn.logit_kd_loss(z, zk, zt, y, kd_kind=self.kind, alpha=self.alpha, tau=self.tau)

    def cpu_prepare(self, hs):
        return tuple(t.float() for t in hs.unbind(0))  # the reference runs fp32 end to end (SURVEY D5)

    def cpu_step(self, cs):
        from oracle import losses as O
        from deltakd_b200 import synth
        z, zk, zt, y = cs
        z = z.detach().requires_grad_(True); zk = zk.detach().requires_grad_(True)
        l = O.distillation_loss(self.kind, (z, zk), y, zt, None, None, {}, synth.default_args(), self.alpha, self.tau)
        l.backward()
        return l


class LogitKDLargeBatch(LogitKD):
    """The same fused logit kernel at B = 16 384 (197 MB of algorithmic traffic): configs[1] itself moves 3 MB and is
    launch-bound by construction (SURVEY 8d), so the kernel's bandwidth fraction is shown on this batch sweep point."""
    name = "soft_kd_logits_b16384_c1000_bf16"
    B = 16384
    cpu_B = 2048
    default_steps = 20


class LogitKDf32(LogitKD):
    """configs[1]'s op in the reference's own dtype (fp32 end to end, SURVEY D5): the same-dtype comparison with the CPU arm."""
    name = "soft_kd_logits_b256_c1000_f32"
    dtype = "f32"
    tdtype = torch.float32


class LogitKDf32B8(LogitKDf32):
    """configs[0]: B = 8 x 1000 classes, fp32 (the reference's CPU-runnable case)."""
    name = "soft_kd_logits_b8_c1000_f32"
    B = 8


class FeatureKD(Workload):
    """Feature-level losses: student block outputs [B,197,192], teacher [B,198,384], heads on the student."""
    kind = ""
    layers = ()
    tdtype = torch.float32
    args_kw = {}
    M_TOK = 196

    def __init__(self, device, rank, B=None):
        super().__init__(device, rank)
        if B is not None and B != self.B:   # cfg5: the global batch of 1024 split over the ranks (B_loc = 1024 / N)
            self.name = self.name.replace(f"_b{self.B}_", f"_b{B}_")
            self.cpu_B = min(self.cpu_B or B, B)
            self.B = B

    def make_args(self):
        from deltakd_b200 import synth
        return synth.default_args(distillation_type=self.kind, **self.args_kw)

    @property
    def parity_rtol(self):
        return 1e-5 if self.tdtype == torch.float32 else 2e-2

    def slice_host(self, hs, n):
        cut = lambda x: None if x is None else x[:n].contiguous()
        return dict(s=[cut(x) for x in hs["s"]], t=[cut(x) for x in hs["t"]], z=cut(hs["z"]), y=cut(hs["y"]), noise=cut(hs["noise"]))

    def bytes_per_set(self):
        return len(self.layers) * self.B * (197 * 192 + 198 * 384) * self.tdtype.itemsize

    def algorithmic_bytes(self):  # per layer: read s, read t, write g_s (SURVEY §8d: M*768*elt)
        return len(self.layers) * self.B * self.M_TOK * 768 * self.tdtype.itemsize

    def host_sets(self, n, B=None):
        from deltakd_b200 import synth
        B = B or self.B
        sets = []
        for i in range(n):
            s, t = synth.make_features(B, 1234 + self.rank + 17 * i, layers=self.layers, **getattr(self, "feat_kw", {}))
            z, _, _, y = synth.make_logits(B, 1000, 99 + self.rank + i)
            sets.append(dict(s=[None if x is None else _pin(x.to(self.tdtype)) for x in s],
                             t=[None if x is None else _pin(x.to(self.tdtype)) for x in t],
                             z=_pin(z), y=_pin(y), noise=_pin(synth.make_noise(B, seed=5 + i))))
        return sets

    def setup(self):
        from deltakd_b200 import DistillationLoss, call_base_loss, synth, heads as H
        self.args = self.make_args()
        self.teacher = synth.FeatureReplayModel(384)
        self.student = synth.FeatureReplayModel(192)
        torch.manual_seed(0)
        H.attach_distillation_heads(self.student, self.teacher, self.args, "deit_tiny_patch16_224")
        self.student = self.student.to(self.device)
        self.crit = DistillationLoss(call_base_loss(self.args), self.teacher, self.kind, 0.1, 3.0)
        self.inputs = torch.zeros(self.B, 3, 2, 2, device=self.device)

    def to_device(self, hs, slot=None):
        if slot is None:
            mv = lambda key, x: None if x is None else x.to(self.device, non_blocking=True)
        else:
            bufs = self.__dict__.setdefault("_slots", {}).setdefault(slot, {})

            def mv(key, x):
                if x is None:
                    return None
                b = bufs.get(key)
                if b is None or b.shape != x.shape:
                    b = bufs[key] = torch.empty_like(x, device=self.device)
                b.copy_(x, non_blocking=True)
                return b.detach()
        d = dict(s=[mv(("s", i), x) for i, x in enumerate(hs["s"])], t=[mv(("t", i), x) for i, x in enumerate(hs["t"])],
                 z=mv("z", hs["z"]), y=mv("y", hs["y"]), noise=mv("noise", hs["noise"]))
        for x in d["s"]:
            if x is not None:
                x.requires_grad_(True)
        d["z"].requires_grad_(True)
        return d

    def input_leaves(self, ds):
        return [("outputs", ds["z"])] + [(f"block{i}", x) for i, x in enumerate(ds["s"]) if x is not None]

    def h2d_bytes(self):
        return self.bytes_per_set() + 2 * self.B * 1000 * 4 + self.B * 196 * 4

    def step(self, ds):
        from unittest import mock
        self.teacher.set_outputs(None, ds["t"])
        for x in ds["s"]:
            if x is not None:
                x.grad = None
        ds["z"].grad = None
        for p in self.student.parameters():
            p.grad = None
        noise = ds["noise"]
        with mock.patch("torch.rand", side_effect=lambda *a, **k: noise):  # fixed mask noise (graph-capturable)
            loss = self.crit(self.inputs[:ds["z"].shape[0]], ds["z"], self.student, ds["s"], ds["y"], self.args)
        loss.backward()
        return loss

    def op_only(self, ds):
        from unittest import mock
        from deltakd_b200 import loss as L
        noise = ds["noise"]
        with mock.patch("torch.rand", side_effect=lambda *a, **k: noise):
            return self.feature_loss(L, ds)

    def cpu_prepare(self, hs):
        return dict(s=[None if x is None else x.float() for x in hs["s"]], t=[None if x is None else x.float() for x in hs["t"]],
                    z=hs["z"].float(), y=hs["y"].float(), noise=hs["noise"])

    def cpu_step(self, cs):
        from oracle import losses as O
        from deltakd_b200 import heads as H
        if not hasattr(self, "_cpu_heads"):
            from deltakd_b200 import synth
            st = synth.FeatureReplayModel(192)
            torch.manual_seed(0)
            H.attach_distillation_heads(st, synth.FeatureReplayModel(384), self.make_args(), "deit_tiny_patch16_224")
            self._cpu_student = st
        heads = H.head_tensors(self._cpu_student)
        for p in heads.values():
            p.grad = None
        s = [None if x is None else x.detach().requires_grad_(True) for x in cs["s"]]
        z = cs["z"].detach().requires_grad_(True)
        l = O.distillation_loss(self.kind, z, cs["y"], None, s, cs["t"], heads, self.make_args(), 0.1, 3.0, noise=cs["noise"])
        l.backward()
        return l


class CurKDEarly(FeatureKD):
    """configs[2]: selective layer-wise hidden-state matching, CurKD early phase (layers 0-2), B=512, fp32."""
    name = "curkd_early_3layers_b512_f32"
    kind, layers, B, cpu_B = "curkd", (0, 1, 2), 512, 64
    args_kw = dict(current_epoch=0)
    dominant = "dkd_align_mse_fwdbwd (planes + 3 tcgen05 GEMMs per layer)"

    def algorithmic_flops(self):
        return len(self.layers) * 3 * 2.0 * self.B * 196 * 192 * 384

    def feature_loss(self, L, ds):
        return L.curkd_loss(self.student, ds["s"], ds["t"], self.args)


class CurKDMid(CurKDEarly):
    name = "curkd_mid_4layers_b512_f32"
    layers = (3, 4, 5, 6)
    args_kw = dict(current_epoch=120)


class MGD(FeatureKD):
    """configs[3]: MGD masked feature reconstruction with the 2-conv generator, B=512, fp32 in / bf16x3 tensor passes."""
    name = "mgd_b512_f32"
    kind, layers, B, cpu_B = "mgd", (11,), 512, 16
    bound = "tensor"
    default_steps = 10
    dominant = "dkd_masked_generation_fwdbwd (implicit-GEMM conv fwd/dgrad/wgrad on tcgen05)"

    def algorithmic_flops(self):  # 6 conv GEMMs + 3 align GEMMs (SURVEY §8d cfg4: 1 642 GFLOP at B=512)
        M = self.B * 196
        return 6 * 2.0 * M * 3456 * 384 + 3 * 2.0 * M * 192 * 384

    def feature_loss(self, L, ds):
        return L.mgd_loss(self.student, ds["s"], ds["t"], self.args)


class WassL1(FeatureKD):
    """configs[4] (l1 variant): WassKD sorted-L1 over tokens, layers 0-2, B=512 per GPU (global 1024 at 2 GPUs)."""
    name = "wasskd_l1_b512_f32"
    kind, layers, B, cpu_B = "wasskd", (0, 1, 2), 512, 32
    args_kw = dict(wasskd_type="l1")
    dominant = "dkd_wass_l1_fwdbwd (align GEMM + on-chip bitonic sort + dgrad/wgrad GEMMs)"

    def algorithmic_flops(self):
        return len(self.layers) * 3 * 2.0 * self.B * 196 * 192 * 384

    def feature_loss(self, L, ds):
        from deltakd_b200 import functional as Fn
        return Fn.wass_l1_loss(ds["s"][:3], ds["t"][:3], list(self.student.align_wasskd), weight=5.0)


class WassSinkhorn(FeatureKD):
    """configs[4] (sinkhorn variant): debiased Sinkhorn divergence per (sample, layer), layers 0-2, B=512 per GPU.
    On-chip bound (MUFU ex2 + eps-step latency): the HBM fraction is reported for completeness, the meaningful
    figure is `exp_per_s` against 16 ex2/clk/SM x 148 SMs."""
    name = "wasskd_sinkhorn_b512_f32"
    kind, layers, B, cpu_B = "wasskd", (0, 1, 2), 512, 1
    default_steps = 5
    args_kw = dict(wasskd_type="sinkhorn")
    feat_kw = dict(scale=0.5, t_shift=0.1)
    dominant = "dkd_wass_sinkhorn_fwdbwd (sinkhorn_kernel<xy>, <xx/yy>: cost matrix in shared memory)"
    N_EPS = 13  # diameter ~59 at this scale (SURVEY 8d)

    def algorithmic_flops(self):
        return len(self.layers) * self.B * (3 * 2.0 * 196 * 196 * 384 + 2 * 2.0 * 196 * 196 * 384 + 3 * 2.0 * 196 * 192 * 384)

    def extra_roofline(self, k_ms):
        exps = len(self.layers) * self.B * (self.N_EPS + 2) * 4 * 196 * 196 * 1.0
        peak = 16 * 148 * 1.965e9
        return {"exp_per_s": exps / (k_ms * 1e-3), "mufu_peak_exp_per_s": peak, "mufu_frac": exps / (k_ms * 1e-3) / peak,
                "note": "bound is MUFU ex2 / eps-step latency (on-chip); hbm frac is n/a by construction"}

    def feature_loss(self, L, ds):
        from deltakd_b200 import functional as Fn
        return Fn.wass_sinkhorn_loss(ds["s"][:3], ds["t"][:3], list(self.student.align_wasskd), weight=5.0)


class LRKD(FeatureKD):
    """configs[4] (LRKD): rank-64 projection matching on layers (0, 1, 11), B=512 per GPU (global 1024 at 2 GPUs)."""
    name = "lrkd_r64_b512_f32"
    kind, layers, B, cpu_B = "lrkd", (0, 1, 11), 512, 32
    args_kw = dict(lrkd_rank=64, lrkd_alpha=0.2, lrkd_beta=0.2, lrkd_gamma=0.2)
    dominant = "dkd_lrkd_fwdbwd (teacher planes, tcgen05 Gram, cluster-resident fp64 Jacobi eigensolver, fused projection GEMMs)"

    def algorithmic_bytes(self):  # per layer: T read twice (Gram, projection) + s + g_s  (SURVEY 8d cfg5)
        return len(self.layers) * self.B * 196 * (2 * 384 + 192 + 192) * 4

    def algorithmic_flops(self):
        M = self.B * 196
        return len(self.layers) * (2.0 * M * 384 * 384 + 2.0 * M * 384 * 64 + 3 * 2.0 * M * 192 * 64)

    def extra_roofline(self, k_ms):
        """The eigensolve is a chain of 384 dependent pair rounds per sweep, not a roofline quantity: its time is reported
        beside the fraction (dkd_lrkd_eigensolve on the Gram matrices of this workload's teacher features, CUDA events)."""
        from deltakd_b200 import functional as Fn
        hs = self.host_sets(1)[0]
        g = []
        for ti in (0, 1, 11):
            t = hs["t"][ti][:, 2:].to(self.device).double().reshape(-1, 384)
            g.append(t.t() @ t)
        g = torch.stack(g)
        best, sweeps = None, None
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _, sweeps = Fn.lrkd_eigensolve(g, k=self.args.lrkd_rank)
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3
            best = us if best is None else min(best, us)
        rest_ms = max(k_ms - best * 1e-3, 1e-6)
        return {"eigensolve_us": best, "eigensolve_sweeps": sweeps.tolist(), "eigensolve_share": best / (k_ms * 1e3),
                "frac_hbm_without_eigensolve": self.algorithmic_bytes() / (rest_ms * 1e-3) / 1e9 / peaks()["hbm"],
                "eigensolve": "3 x 384x384 fp64 one-sided Jacobi, one 16-CTA cluster per matrix (48 SMs), latency-bound; "
                              "the rest of the call is the part the hbm fraction describes"}

    def feature_loss(self, L, ds):
        from deltakd_b200 import functional as Fn
        a = self.args
        return Fn.lrkd_layers_loss([ds["s"][0], ds["s"][1], ds["s"][11]], [ds["t"][0], ds["t"][1], ds["t"][11]],
                                   list(self.student.align), a.lrkd_rank, (a.lrkd_alpha, a.lrkd_beta, a.lrkd_gamma), weight=0.1)

    def parity(self):
        """The loss depends on the (arbitrary) sign of every singular vector (SURVEY 7): the oracle's SVD columns are
        sign-aligned to the basis the kernel returns before the KD term is compared (fp64 oracle: LAPACK fp32 is itself
        only ~1e-4 accurate in the vectors of a 6 272 x 384 Gaussian matrix)."""
        from oracle import losses as O
        from deltakd_b200 import functional as Fn, heads as H
        Bc = min(self.cpu_B or self.B, self.B)
        hs = self.slice_host(self.host_sets(1, B=self.B)[0], Bc)
        ds = self.to_device(hs)
        a = self.args
        coef = (a.lrkd_alpha, a.lrkd_beta, a.lrkd_gamma)
        basis = {}
        got = float(Fn.lrkd_layers_loss([ds["s"][0], ds["s"][1], ds["s"][11]], [ds["t"][0], ds["t"][1], ds["t"][11]],
                                        list(self.student.align), a.lrkd_rank, coef, basis_out=basis).item())
        heads = {k: v.detach().double().cpu() for k, v in H.head_tensors(self.student).items()}
        s64 = [None if x is None else x.double() for x in hs["s"]]
        t64 = [None if x is None else x.double() for x in hs["t"]]
        signs = []
        for j, ti in enumerate((0, 1, 11)):
            _, V, _ = O.lrkd_targets(t64[ti][:, 2:], a.lrkd_rank)
            signs.append(torch.sign((basis["V"][j].double().cpu().t() * V).sum(0)))
        want = float(O.lrkd(s64, t64, heads, a.lrkd_rank, coef, signs=signs).item())
        rel = abs(got - want) / max(abs(want), 1e-30)
        return {"batch": Bc, "loss": got, "oracle": want, "rel_err": rel, "rtol": self.parity_rtol, "ok": rel <= self.parity_rtol,
                "note": "KD term, oracle SVD columns sign-aligned to the kernel's basis"}


class SaliencyMGD(MGD):
    """configs[3] (saliency variant): saliency-MGD method 1 (self-attention diagonal), ratio 0.5, B=512."""
    name = "saliency_mgd_m1_b512_f32"
    kind = "saliency_mgd"
    args_kw = dict(saliency_method=1, saliency_mask_ratio=0.5)

    def algorithmic_flops(self):
        M = self.B * 196
        return super().algorithmic_flops() + 2.0 * M * 384 * 768 + 2.0 * self.B * 8 * 196 * 196 * 48

    def feature_loss(self, L, ds):
        return L.saliency_mgd_loss(self.student, ds["s"], ds["t"], self.args)


class CurKDEarlyBf16(CurKDEarly):
    """CurKD early with bf16 activations (one tcgen05 pass): tensor-pipe-bound form of configs[2]."""
    name = "curkd_early_3layers_b512_bf16"
    dtype = "bf16"
    tdtype = torch.bfloat16
    bound = "tensor"   # SURVEY 8d cfg3: AI = 288 FLOP/B with bf16 I/O, above the ridge (214): the tensor pipe bounds it (94.9 us vs 70.6 us of HBM time)


class MGDBf16(MGD):
    """MGD with bf16 activations (one tcgen05 pass per GEMM)."""
    name = "mgd_b512_bf16"
    dtype = "bf16"
    tdtype = torch.bfloat16


class DeiTKDStep(Workload):
    """End-to-end DeiT-Tiny distillation step (SURVEY 8d "End-to-end"; BASELINE metric "DeiT-Ti KD step img/s"):
    student deit_tiny_distilled fwd (bf16 autocast) -> DistillationLoss (frozen deit_small_distilled teacher forward
    inside, once) -> backward -> fused AdamW, DDP gradient all-reduce over NCCL when world > 1.  The models are the
    plain-PyTorch harness of deltakd_b200/deit.py (timm is absent; model code is outside the hot path), random init,
    synthetic ImageNet-shaped inputs.  The whole step is captured once into a CUDA graph (DKD_BENCH_STEP_GRAPH=0: eager)
    and `step` replays it on the step's inputs."""
    name = "deit_tiny_kd_step_soft_b256_bf16"
    dtype = "bf16"
    B, kind = 256, "soft"
    student_name = "deit_tiny_distilled_patch16_224"
    bound = "tensor"
    graphable = False
    default_steps = 10
    cpu_B = 8
    dominant = "whole step: torch model code (cuBLAS / SDPA) + deltakd loss kernels"

    def bytes_per_set(self):
        return self.B * 3 * 224 * 224 * 4 + self.B * 1000 * 4

    def nsets(self):
        return 2

    def algorithmic_flops(self):   # DeiT paper MACs: student 1.3 G fwd (x3 for fwd+bwd), teacher 4.6 G fwd
        return self.B * 2.0 * (3 * 1.3e9 + 4.6e9)

    def host_sets(self, n, B=None):
        B = B or self.B
        sets = []
        for i in range(n):
            g = torch.Generator().manual_seed(1234 + self.rank + 17 * i)
            x = torch.randn(B, 3, 224, 224, generator=g)
            y = torch.softmax(torch.randn(B, 1000, generator=g), dim=-1)
            sets.append((_pin(x), _pin(y)))
        return sets

    def make_args(self):
        from deltakd_b200 import synth
        return synth.default_args(distillation_type=self.kind, current_epoch=0)

    def _build(self, device):
        from deltakd_b200 import DistillationLoss, call_base_loss, deit, heads as H
        args = self.make_args()
        torch.manual_seed(0)
        row_ops = "dkd" if device.type == "cuda" else "aten"   # the CPU model is the reference-style harness of cpu_baseline
        teacher = deit.create_model("deit_small_distilled_patch16_224", row_ops=row_ops).to(device).eval()
        for p_ in teacher.parameters():
            p_.requires_grad_(False)
        if device.type == "cuda":
            teacher = teacher.to(torch.bfloat16)   # frozen: keep bf16 weights instead of autocast-casting them every step
        student = deit.create_model(self.student_name, row_ops=row_ops).to(device)
        H.attach_distillation_heads(student, teacher, args, self.student_name)
        student = student.to(device).train()
        return args, teacher, student, DistillationLoss, call_base_loss

    def setup(self):
        import torch.distributed as dist
        self.args, self.teacher, self.student, DL, cbl = self._build(self.device)
        self.model = self.student
        self.crit = DL(cbl(self.args), _Autocast(self.teacher), self.kind, 0.1, 3.0)
        # Heads that get no gradient in this phase (CurKD mid/late heads at epoch 0, ...) would stall DDP's reducer
        # (SURVEY D6: the reference has this defect): find them with one tiny dry-run step and freeze them.
        xs = torch.randn(2, 3, 224, 224, device=self.device)
        ys = torch.softmax(torch.randn(2, 1000, device=self.device), dim=-1)
        self.opt = None
        self._graph = None
        self._dry = (xs, ys)
        ddp = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        # Under torchrun the whole-step graph (NCCL all-reduce inside) is used when this workload is the one selected with
        # --workload (verified at 2 and 8 GPUs); as one of several "extras" in a multi-rank process it runs eagerly —
        # capturing a second DDP graph on the same process group after the first was destroyed is not a tested sequence.
        use_graph = os.environ.get("DKD_BENCH_STEP_GRAPH", "1") != "0" and (not ddp or getattr(self, "allow_ddp_graph", True))
        import contextlib
        side = torch.cuda.Stream() if use_graph else None
        if use_graph:
            side.wait_stream(torch.cuda.current_stream())
        # DDP under whole-step capture must be built (and warmed up) on a side stream; the eager path stays on the current one
        with (torch.cuda.stream(side) if use_graph else contextlib.nullcontext()):
            self._dry_loss = self._eager_step((xs, ys), optimize=False).detach().clone()
            for p_ in self.student.parameters():
                if p_.grad is None:
                    p_.requires_grad_(False)
                p_.grad = None
            if ddp:
                self.model = torch.nn.parallel.DistributedDataParallel(self.student, device_ids=[self.device.index])
            self.opt = torch.optim.AdamW([p_ for p_ in self.student.parameters() if p_.requires_grad], lr=5e-4, weight_decay=0.05,
                                         fused=True, capturable=use_graph)
            if use_graph:
                # The whole step (student fwd, frozen teacher fwd, fused loss, backward, DDP all-reduce, fused AdamW) is
                # ONE CUDA graph: the loss path never syncs the host, so nothing in the step needs the CPU — eagerly the
                # ~970 launches of a step cost 18.4 ms of CPU against 16 ms of GPU work.
                self._sx = torch.randn(self.B, 3, 224, 224, device=self.device)
                self._sy = torch.softmax(torch.randn(self.B, 1000, device=self.device), dim=-1)
                for _ in range(11 if ddp else 3):   # DDP needs 11 eager iterations before capture (torch CUDA-graphs notes)
                    self._eager_step((self._sx, self._sy))
        if use_graph:
            torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        if use_graph:
            self.opt.zero_grad(set_to_none=True)
            from deltakd_b200 import _lib
            g = torch.cuda.CUDAGraph()
            c0 = _lib.lib.dkd_launch_count()
            with torch.cuda.graph(g, stream=side):
                self._sloss = self._eager_step((self._sx, self._sy), zero=False)
            self.launches_per_step = int(_lib.lib.dkd_launch_count() - c0)   # libdeltakd kernels inside one replay
            self._graph = g
            torch.cuda.synchronize()

    def to_device(self, hs, slot=None):
        if slot is None:
            return tuple(t.to(self.device, non_blocking=True) for t in hs)
        bufs = self.__dict__.setdefault("_slots", {})
        if slot not in bufs:
            bufs[slot] = tuple(torch.empty_like(t, device=self.device) for t in hs)
        for b, t in zip(bufs[slot], hs):
            b.copy_(t, non_blocking=True)
        return bufs[slot]

    def h2d_bytes(self):
        return self.bytes_per_set()

    def extra_info(self):
        import torch.distributed as dist
        ws = dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1
        nbytes = sum(p_.numel() * p_.element_size() for p_ in self.student.parameters() if p_.requires_grad)
        return {"collective": (f"DDP gradient all-reduce over NCCL ({ws} ranks, {nbytes / 1e6:.1f} MB of fp32 gradients per step, default 25 MB "
                               "buckets) inside the captured step" if ws > 1 else "none (single rank)"),
                "grad_bytes_per_step": nbytes, "img_per_s_per_gpu": None}

    def _eager_step(self, ds, optimize=True, zero=True):
        from deltakd_b200 import forward_with_features
        x, y = ds
        if optimize and zero:
            self.opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if self.kind in ("soft", "hard"):
                out, feats = self.model(x), None
            else:
                out, feats = forward_with_features(self.model, x)
        loss = self.crit(x, out, self.model, feats, y, self.args)
        loss.backward()
        if optimize:
            self.opt.step()
        return loss

    def step(self, ds, optimize=True):
        if self._graph is None:
            return self._eager_step(ds, optimize)
        self._sx.copy_(ds[0], non_blocking=True)   # the graph reads its static input buffers
        self._sy.copy_(ds[1], non_blocking=True)
        self._graph.replay()
        return self._sloss

    op_only = step

    parity_rtol = 3e-2   # bf16 autocast student + bf16 teacher on the GPU vs the fp32 models on the CPU

    def parity(self):
        """The 2-image dry-run step of setup() (same weights: both models are built under manual_seed(0)) against the fp32
        CPU models + oracle loss on the same images."""
        from oracle import losses as O
        from deltakd_b200 import heads as H, features
        xs, ys = (t.detach().float().cpu() for t in self._dry)
        args, teacher, student, _, _ = self._build(torch.device("cpu"))
        with torch.no_grad():
            if self.kind in ("soft", "hard"):
                t_logits, t_feats = teacher(xs), None
                out, s_feats = student(xs), None
            else:
                t_logits, t_feats = features.forward_with_features(teacher, xs)
                out, s_feats = features.forward_with_features(student, xs)
            want = float(O.distillation_loss(self.kind, out, ys, t_logits, s_feats, t_feats, H.head_tensors(student), args, 0.1, 3.0).item())
        got = float(self._dry_loss.item())
        rel = abs(got - want) / max(abs(want), 1e-30)
        return {"batch": int(xs.shape[0]), "loss": got, "oracle": want, "rel_err": rel, "rtol": self.parity_rtol, "ok": rel <= self.parity_rtol}

    def cpu_prepare(self, hs):
        return hs

    def cpu_step(self, cs):
        """Reference-style CPU step: same harness models in fp32 on the host, oracle loss (the reference's arithmetic)."""
        from oracle import losses as O
        from deltakd_b200 import heads as H, features
        if not hasattr(self, "_cpu"):
            args, teacher, student, _, _ = self._build(torch.device("cpu"))
            self._cpu = (args, teacher, student, torch.optim.AdamW(student.parameters(), lr=5e-4, weight_decay=0.05))
        args, teacher, student, opt = self._cpu
        x, y = cs
        opt.zero_grad(set_to_none=True)
        with torch.no_grad():
            if self.kind in ("soft", "hard"):
                t_logits, t_feats = teacher(x), None
            else:
                t_logits, t_feats = features.forward_with_features(teacher, x)
        if self.kind in ("soft", "hard"):
            out, s_feats = student(x), None
        else:
            out, s_feats = features.forward_with_features(student, x)
        l = O.distillation_loss(self.kind, out, y, t_logits, s_feats, t_feats, H.head_tensors(student), args, 0.1, 3.0)
        l.backward()
        opt.step()
        return l


class _Autocast(torch.nn.Module):
    """Runs the frozen teacher under bf16 autocast (SURVEY 8f rank 1: the reference runs it in fp32, twice)."""

    def __init__(self, inner):
        super().__init__()
        self.inner = inner
        self.embed_dim = inner.embed_dim

    @property
    def blocks(self):
        return self.inner.blocks

    def forward(self, x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return self.inner(x.to(torch.bfloat16))


class DeiTKDStepCurKD(DeiTKDStep):
    """The same end-to-end step with the CurKD early-phase feature loss (layers 0-2 hidden-state matching)."""
    name = "deit_tiny_kd_step_curkd_b256_bf16"
    kind = "curkd"
    student_name = "deit_tiny_patch16_224"


HEADLINE = LogitKD
EXTRAS = (DeiTKDStep, DeiTKDStepCurKD, LogitKDf32, LogitKDf32B8, LogitKDLargeBatch, CurKDEarly, CurKDMid, CurKDEarlyBf16, MGD, MGDBf16,
          SaliencyMGD, LRKD, WassL1, WassSinkhorn)
WORKLOADS = {w.name: w for w in (HEADLINE,) + EXTRAS}
# Under torchrun (N > 1) the line also carries the workloads whose step contains a collective — the end-to-end DeiT-Tiny KD
# step with DDP's gradient all-reduce (~34 MB, reference tools/train.py:308) inside the captured step — and BASELINE
# configs[4]: LRKD / WassKD at a GLOBAL batch of 1024 split data-parallel (B_loc = 1024 / N, no data-path collective).
CFG5_GLOBAL_BATCH = 1024
MULTI_RANK_EXTRAS = (DeiTKDStep, DeiTKDStepCurKD, LRKD, WassL1, WassSinkhorn)


# ----------------------------------------------------------------------------- measurement
def cpu_baseline(w: Workload, budget_s: float = 12.0, max_steps: int = 20000):
    torch.set_num_threads(os.cpu_count() or 1)
    Bc = w.cpu_B or w.B
    cs = [w.cpu_prepare(h) for h in w.host_sets(2, B=Bc)]
    w.cpu_step(cs[0])
    t0 = time.perf_counter(); n = 0
    while True:
        w.cpu_step(cs[n % 2]); n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or n >= max_steps:
            break
    return {"value": Bc * n / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} steps of {w.name} at batch {Bc} (fp32 torch-CPU oracle of the reference loss, fwd+bwd), {dt:.1f} s"}


def run_reference(args, w_cls):
    """Reference arm: the reference's CPU implementation of the path (oracle port), all host threads."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    w = w_cls(torch.device("cpu"), 0)
    torch.set_num_threads(os.cpu_count() or 1)
    Bc = w.cpu_B or w.B
    cs = [w.cpu_prepare(h) for h in w.host_sets(2, B=Bc)]
    for i in range(max(args.warmup, 1)):
        w.cpu_step(cs[i % 2])
    t0 = time.perf_counter()
    for i in range(args.steps):
        w.cpu_step(cs[i % 2])
    dt = time.perf_counter() - t0
    v = Bc * args.steps / dt
    sample = f"{args.steps} steps of {w.name} at batch {Bc}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.name, "note": "reference loss path restated for CPU (oracle port), torch CPU fp32, "
                   "all host threads; the reference is pure PyTorch and is not present on the GPU box"},
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_ncu_op(w_cls):
    """One call of the fused op between cudaProfilerStart / Stop (inputs: set 0, after 2 warm-up calls)."""
    torch.cuda.set_device(0)
    w = w_cls(torch.device("cuda", 0), 0)
    w.setup()
    ds = w.to_device(w.host_sets(1)[0])
    for _ in range(2):
        w.op_only(ds)
    torch.cuda.synchronize()
    torch.cuda.profiler.start()
    w.op_only(ds)
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    print(json.dumps({"ncu_op": w.name}))


def _graph_of(fn, reps):
    """Capture `reps` calls of fn() into one CUDA graph (after a side-stream warm-up call)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn(0)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):   # capture on the warm-up stream: the op scratch cached per stream is reused
        last = None
        for i in range(reps):
            last = fn(i)
    g.replay()  # untimed: graph upload
    torch.cuda.synchronize()
    return g, last


DUMP_BYTES = 64 << 20


def dump_outputs(outs, path):
    """Writes each output as <path>/<name>.npy, float64 if it is float64 and float32 otherwise.  An output with more elements
    than its share of DUMP_BYTES is written as a sample: the flattened tensor at sorted indices drawn from a generator
    seeded with 0, so the sample is the same in every run with the same shapes."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // (8 * max(1, len(outs)))
    for name, t in outs.items():
        t = t.detach()
        if t.numel() > share:
            idx = torch.randint(0, t.numel(), (share,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        t = t.double() if t.dtype == torch.float64 else t.float()
        np.save(os.path.join(path, f"{name}.npy"), t.cpu().numpy())


ROUNDS = 11   # each round times EXACTLY K steps between barrier + synchronize; ms_per_step is the median round


def _timed_replay(g, barrier, allmax=None, rounds=1):
    """`rounds` timed replays of a K-step graph, each bracketed by barrier + torch.cuda.synchronize on both sides and
    timed with CUDA events on the replay stream; per round the MAX over ranks is taken, then the median over rounds
    (a single 20-step region of a 7 us step is 0.15 ms: one scheduling hiccup on one of 8 ranks moves it by 10 %).
    Returns (ms of the median round, (wall t0, t1))."""
    times = []
    t0 = time.time()
    for _ in range(rounds):
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        barrier()
        times.append(e0.elapsed_time(e1))
    if allmax is not None:
        times = allmax(times)
    times.sort()
    return times[len(times) // 2], (t0, time.time())


def measure(w: Workload, K: int, W: int, world: int, barrier, allmax, pk, with_cpu: bool, dump_dir=None):
    """dump_dir: if set, rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    from deltakd_b200 import _lib
    w.setup()
    # ---- parity gate (rank 0 computes, every rank learns the verdict): nothing is timed unless the loss matches the oracle
    par = None
    if w.rank == 0 and os.environ.get("DKD_BENCH_PARITY", "1") != "0":
        try:
            par = w.parity()
        except Exception as e:   # a crash of the check is a failed check
            par = {"ok": False, "error": f"{type(e).__name__}: {e}"[:300]}
    bad = allmax([0.0 if (par is None or par["ok"]) else 1.0])[0]
    if bad:
        raise AssertionError(f"{w.name}: loss does not match the CPU oracle: {par}")
    nsets = w.nsets()
    host = w.host_sets(nsets)
    dsets = [w.to_device(h) for h in host]
    torch.cuda.synchronize()
    windows = []

    # ---- device-resident throughput: eager warm-up, then K steps replayed from a CUDA graph
    for i in range(W):
        w.step(dsets[i % nsets])
    torch.cuda.synchronize()
    c0 = _lib.lib.dkd_launch_count()
    if getattr(w, "graphable", True):
        graph, last = _graph_of(lambda i: w.step(dsets[(W + i) % nsets]), K)
        launches = (_lib.lib.dkd_launch_count() - c0) * K // (K + 1)   # the capture pass ran fn K+1 times
        rounds = ROUNDS if K * 1.0 < 2000 else 1
        ms, win = _timed_replay(graph, barrier, allmax, rounds)
        windows.append(win)
        loss_val = float(last.item())
        if dump_dir and w.rank == 0:   # before the graph, which owns the last step's gradients, is released
            dump_outputs(w.outputs(dsets[(W + K - 1) % nsets], last), dump_dir)
        del graph

        # ---- the fused loss op alone (C-ABI call without the autograd rescale), same rotation, own graph
        kg, _ = _graph_of(lambda i: w.op_only(dsets[(W + i) % nsets]), K)
        k_ms, win = _timed_replay(kg, barrier, None, min(rounds, 5))
        windows.append(win)
        k_ms /= K
        del kg
    else:   # K whole steps between two events (the step holds an optimizer and, multi-GPU, DDP's all-reduce); 3 rounds, median
        rounds_ms = []
        t0 = time.time()
        for _ in range(3):
            barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(K):
                last = w.step(dsets[(W + i) % nsets])
            e1.record()
            torch.cuda.synchronize()
            barrier()
            rounds_ms.append(e0.elapsed_time(e1))
        windows.append((t0, time.time()))
        rounds_ms = sorted(allmax(rounds_ms))
        ms = rounds_ms[1]
        launches = _lib.lib.dkd_launch_count() - c0
        if getattr(w, "_graph", None) is not None:   # replays do not pass through the library's host-side counter
            launches = w.launches_per_step * K
        loss_val = float(last.item())
        if dump_dir and w.rank == 0:
            dump_outputs(w.outputs(dsets[(W + K - 1) % nsets], last), dump_dir)
        k_ms = ms / K

    # ---- end to end through the public API with host buffers
    # (a) serial: copy in, step, read the loss back (a host synchronisation) — every step waits for the previous one
    for i in range(W):
        w.step(w.to_device(host[i % nsets])).item()
    barrier()
    torch.cuda.synchronize()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e2.record()
    for i in range(K):
        w.step(w.to_device(host[(W + i) % nsets])).item()
    e3.record()
    torch.cuda.synchronize()
    windows.append((t0, time.time()))
    ms_e2e_serial = allmax([e2.elapsed_time(e3)])[0]
    # (b) the way an input pipeline feeds a training loop: the same K host->device copies and K loss read-backs, all inside
    # the timed region, but the copy of step i+1 runs on a second stream while step i computes, and the losses land in pinned
    # memory that is read after the one synchronisation at the end (possible because the loss path never syncs the host)
    main, copy_stream = torch.cuda.current_stream(), torch.cuda.Stream()
    loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()
    done = [None, None]        # per device input slot: the step that last read it has finished

    def fetch(i):
        slot = i & 1
        with torch.cuda.stream(copy_stream):
            if done[slot] is not None:
                copy_stream.wait_event(done[slot])
            ds_ = w.to_device(host[i % nsets], slot=slot)
            ev_ = torch.cuda.Event()
            ev_.record(copy_stream)
        return ds_, ev_, slot

    for i in range(2):         # allocate the two device slots outside the timed region
        fetch(i)
    barrier()
    torch.cuda.synchronize()
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e4.record()
    nxt = fetch(W)
    for i in range(K):
        ds_, ev_, slot = nxt
        main.wait_event(ev_)
        if i + 1 < K:
            nxt = fetch(W + i + 1)
        loss_host[i].copy_(w.step(ds_).detach(), non_blocking=True)
        done[slot] = torch.cuda.Event()
        done[slot].record(main)
    e5.record()
    torch.cuda.synchronize()
    windows.append((t0, time.time()))
    if not bool(torch.isfinite(loss_host).all()):
        raise RuntimeError(f"{w.name}: non-finite loss in the pipelined end-to-end loop")
    ms_e2e_prefetch = allmax([e4.elapsed_time(e5)])[0]
    del nxt
    # (c) launch-bound steps: one CUDA graph per step = the H2D copies of that step's pinned host inputs + the public-API
    # forward / backward + the D2H copy of the loss; the host launches it and WAITS for the loss before the next step
    ms_e2e_graph = None
    if getattr(w, "graphable", True):
        ng = min(nsets, 4)
        loss_pin = torch.zeros(ng, dtype=torch.float32).pin_memory()

        def one(j):
            def fn(_):
                loss_pin[j].copy_(w.step(w.to_device(host[(W + j) % nsets], slot="graph")).detach(), non_blocking=True)
            return fn
        graphs = [_graph_of(one(j), 1)[0] for j in range(ng)]
        for j in range(min(W, ng)):
            graphs[j].replay()
        barrier()
        torch.cuda.synchronize()
        e6, e7 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e6.record()
        acc = 0.0
        for i in range(K):
            graphs[i % ng].replay()
            main.synchronize()
            acc += float(loss_pin[i % ng])
        e7.record()
        torch.cuda.synchronize()
        windows.append((t0, time.time()))
        if acc != acc:
            raise RuntimeError(f"{w.name}: non-finite loss in the graph end-to-end loop")
        ms_e2e_graph = allmax([e6.elapsed_time(e7)])[0]
        del graphs
    e2e_modes = {"serial": ms_e2e_serial, "prefetch": ms_e2e_prefetch}
    if ms_e2e_graph is not None:
        e2e_modes["graph"] = ms_e2e_graph
    e2e_best = min(e2e_modes, key=e2e_modes.get)
    ms_e2e = e2e_modes[e2e_best]

    if w.bound == "hbm":
        ach, peak, unit, alg = w.algorithmic_bytes() / (k_ms * 1e-3) / 1e9, pk["hbm"], "GB/s", w.algorithmic_bytes()
    else:
        ach, peak, unit, alg = w.algorithmic_flops() / (k_ms * 1e-3) / 1e12, pk["bf16_sus"], "TFLOP/s", w.algorithmic_flops()
    res = {
        "workload": w.name, "value": world * w.B * K / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms / K, "steps": K,
        "dtype": w.dtype, "batch_per_gpu": w.B, "loss": loss_val, "parity": par,
        "rounds": "median of %d rounds of K steps, max over ranks per round" % (ROUNDS if getattr(w, "graphable", True) else 3),
        "l2": (f"{nsets} rotating input sets ({nsets * w.bytes_per_set() / 2**20:.0f} MiB > 126 MiB L2)" if nsets > 1
               else f"one input set of {w.bytes_per_set() / 2**20:.0f} MiB (> 126 MiB L2)"),
        "e2e": {"value": world * w.B * K / (ms_e2e * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": w.h2d_bytes(),
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / K,
                "mode": e2e_best,
                "modes": {"serial": "copy in, DistillationLoss forward + backward, loss.item() (host sync) every step",
                          "prefetch": "the same calls; the H2D copy of step i+1 runs on a second stream while step i computes, losses land in "
                                      "pinned memory and are read after the one synchronize at the end",
                          "graph": "one CUDA graph per step (H2D copies of the pinned inputs + the captured public-API forward / backward + D2H "
                                   "copy of the loss); the host waits for every step's loss"},
                "ms_per_step_by_mode": {k: v / K for k, v in e2e_modes.items()},
                "note": "value = the best of the modes above; in every mode each step's H2D input copy and D2H loss copy are inside the timed region",
                "serial_ms_per_step": ms_e2e_serial / K},
        "gpu_launches": int(launches),
        "roofline": {"bound": w.bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                     "traffic": NCU_TRAFFIC.get(w.name, {}).get("bytes"), "traffic_source": NCU_TRAFFIC.get(w.name, {}).get("source"),
                     "kernel": w.dominant, "kernel_us": k_ms * 1e3, "peak_source": pk["src"],
                     ("algorithmic_bytes" if w.bound == "hbm" else "algorithmic_flops"): alg},
    }
    if not getattr(w, "graphable", True):
        res["timing"] = ("K replays of the whole-step CUDA graph (fwd + loss + bwd + DDP all-reduce + AdamW), CUDA events, max over ranks"
                         if getattr(w, "_graph", None) is not None else "eager steps (optimizer + DDP inside), CUDA events, max over ranks")
    if w.bound == "hbm" and w.algorithmic_flops():
        res["roofline"]["algorithmic_flops"] = w.algorithmic_flops()
    try:   # both fractions where both algorithmic quantities are defined (SURVEY 8d: "report both")
        res["roofline"]["frac_hbm"] = w.algorithmic_bytes() / (k_ms * 1e-3) / 1e9 / pk["hbm"]
        if w.algorithmic_flops():
            res["roofline"]["frac_tensor"] = w.algorithmic_flops() / (k_ms * 1e-3) / 1e12 / pk["bf16_sus"]
    except Exception:
        pass
    if hasattr(w, "extra_roofline"):
        res["roofline"].update(w.extra_roofline(k_ms))
    if hasattr(w, "extra_info"):
        res.update(w.extra_info())
        res["img_per_s_per_gpu"] = w.B * K / (ms * 1e-3)
        table = os.environ.get("DKD_BENCH_KERNEL_TABLE")
        if table:   # evidence helper: per-kernel device times of 3 more steps (CUPTI through torch.profiler; all ranks step,
            #         rank 0 records) — names the NCCL all-reduce kernel and its share of the step; never a bench number
            from torch.profiler import ProfilerActivity, profile
            barrier()
            if w.rank == 0:
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for i in range(3):
                        w.step(dsets[i % nsets])
                    torch.cuda.synchronize()
                with open(f"{table}_{w.name}_n{world}.txt", "w") as fh:
                    fh.write(f"# {w.name}, {world} rank(s), 3 steps on rank 0 (torch.profiler / CUPTI); step = {ms / K:.3f} ms (max over ranks)\n")
                    fh.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=45, max_name_column_width=90))
            else:
                for i in range(3):
                    w.step(dsets[i % nsets])
                torch.cuda.synchronize()
            barrier()
    if with_cpu:
        res["cpu_baseline"] = cpu_baseline(w, budget_s=12.0 if isinstance(w, LogitKD) else 6.0)
    del dsets, host
    torch.cuda.empty_cache()
    return res, windows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default=HEADLINE.name, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only")
    ap.add_argument("--extras", action="store_true", help="also run the other workloads under torchrun (default: single-GPU runs only)")
    ap.add_argument("--ncu-op", action="store_true",
                    help="profiling helper: warm up, then run ONE call of the workload's fused op inside cudaProfilerStart/Stop "
                         "(use with `ncu --profile-from-start off`; tools/ncu_traffic.py turns the CSV into profiles/ncu_traffic.json)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of the selected workload computed (loss and "
                         "gradients) as DIR/<name>.npy, at most 64 MB in all (larger outputs as a fixed sample); the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.ncu_op):
        ap.error("--dump-outputs writes the outputs of the timed GPU path; it does not apply to --impl reference or --ncu-op")
    w_cls = WORKLOADS[args.workload]
    if args.steps is None:
        args.steps = w_cls.default_steps
    if args.impl == "reference":
        return run_reference(args, w_cls)
    if args.ncu_op:
        return run_ncu_op(w_cls)

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist_on = world > 1
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if dist_on:
        import torch.distributed as dist
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")   # required for NCCL collectives inside a captured step
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist_on:
            dist.barrier()

    def allmax(vals):
        if not dist_on:
            return vals
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    W = max(args.warmup, 3)
    pk = peaks()
    sampler = ClockSampler(local).start() if rank == 0 else None
    with_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline

    head, windows = measure(w_cls(dev, rank), args.steps, W, world, barrier, allmax, pk, with_cpu, args.dump_outputs)
    extras = []
    # The other configs are reported beside the headline on single-GPU runs; a multi-rank run measures the selected
    # workload only unless --extras is given (keeps the 1 -> 8 scaling runs short; per-workload multi-GPU lines are
    # taken with --workload, see profiles/).
    if not args.no_extras and w_cls is HEADLINE:
        todo = EXTRAS if (world == 1 or args.extras) else MULTI_RANK_EXTRAS
        for cls in todo:
            try:
                if world > 1 and issubclass(cls, FeatureKD) and cls in (LRKD, WassL1, WassSinkhorn):
                    wl = cls(dev, rank, B=CFG5_GLOBAL_BATCH // world)
                else:
                    wl = cls(dev, rank)
                r, win = measure(wl, min(args.steps, cls.default_steps), W, world, barrier, allmax, pk, with_cpu)
                if world > 1 and isinstance(wl, FeatureKD):
                    r["global_batch"] = wl.B * world
            except Exception as e:  # one failing extra must not cost the headline line; it is reported, not hidden
                r, win = {"workload": cls.name, "error": f"{type(e).__name__}: {e}"[:400]}, []
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
            extras.append(r)
            windows += win

    if rank == 0:
        clocks = sampler.stop(windows)
        out = {
            "metric": METRIC, "value": head["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": W, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic",
            "config": {"workload": head["workload"], "batch_per_gpu": head["batch_per_gpu"],
                       "timing": head.get("timing", "CUDA-graph replay of K steps, CUDA events, max over ranks"), "l2": head["l2"],
                       "teacher": ("frozen DeiT-Small teacher forward inside the step" if "deit" in head["workload"]
                                   else "teacher outputs replayed (inputs of the loss path)"), "loss": head["loss"],
                       "parity": head.get("parity"), "rounds": head.get("rounds")},
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "clocks": clocks,
        }
        if "cpu_baseline" in head:
            out["cpu_baseline"] = head["cpu_baseline"]
        if extras:
            out["workloads"] = extras
        print(json.dumps(out))
    if dist_on:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
