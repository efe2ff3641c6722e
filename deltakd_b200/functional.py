"""torch.autograd.Function wrappers over the C ABI (include/deltakd.h).

PyTorch is plumbing here: it owns device memory and streams; every number is
produced by libdeltakd_sm100's kernels.  All losses are fused forward+backward:
the forward launch also writes the gradients for d(loss)=1 and `backward` only
rescales them on the device when the incoming grad is not 1
(`dkd_scale_if_not_one`, no host sync).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}


_raw_stream = torch._C._cuda_getCurrentRawStream   # torch.cuda.current_stream() costs ~15 us of Python per call


def _stream() -> int:
    """cudaStream_t of torch's current stream on the current device (plain int: the argtypes convert it)."""
    return _raw_stream(torch._C._cuda_getDevice())


def _ptr(t):
    return None if t is None else t.data_ptr()


def _require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("deltakd_b200 runs on CUDA (sm_100) tensors only; there is no CPU path")


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"unsupported dtype {t.dtype}: the kernels take float32 or bfloat16 storage "
                        "(float16 is upcast at the Python boundary; use autocast(dtype=torch.bfloat16) for a "
                        "half-width path)") from None


def _f16_up(t):
    """float16 activations (the reference trainer's `--amp` autocast default, tools/engine.py:24) are upcast to
    float32 with an ordinary differentiable cast: autograd hands the gradient back in float16.  The kernels' half
    width storage type is bfloat16; float16 -> float32 is exact, so nothing is lost."""
    if t is not None and t.dtype == torch.float16:
        return t.float()
    return t


def _f16_up_list(ts):
    return [_f16_up(t) for t in ts]


# Scratch arenas are cached per (device, STREAM, tag): two streams (or two threads on their own streams) running the
# same op never share a ticket counter or an arena.  Within one stream the launches are ordered, so reuse is safe.
# zero-initialised variant: kernels leave their counters reset
_WS: dict = {}


def _workspace(device: torch.device, tag: str, nbytes: int, stream: int | None = None) -> torch.Tensor:
    key = (device.index, _stream() if stream is None else stream, tag)
    ws = _WS.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(max(nbytes, 1024), dtype=torch.uint8, device=device)
        if not torch.cuda.is_current_stream_capturing():   # memory of a graph's private pool must not outlive the graph
            _WS[key] = ws
    return ws


def _rescale_(grad_out: torch.Tensor, *grads):
    """g *= grad_out on the device for every gradient, skipped when grad_out == 1 (decided on the
    device, no host sync).  Tensors of one dtype are rescaled two per launch."""
    go = grad_out
    if go.dtype != torch.float32 or not go.is_contiguous():
        go = go.to(torch.float32).contiguous()
    live = [g for g in grads if g is not None and g.numel() > 0]
    fn, go_ptr, st = _lib.lib.dkd_scale_if_not_one, go.data_ptr(), _stream()
    if len(live) == 2 and live[0].dtype == live[1].dtype:     # the logit losses: both gradients in one launch
        a, b = live
        rc = fn(a.data_ptr(), a.numel(), b.data_ptr(), b.numel(), _DT[a.dtype], go_ptr, st)
        if rc:
            _lib.check(rc, "dkd_scale_if_not_one")
        return grads
    while live:
        a = live.pop(0)
        j = next((k for k, g in enumerate(live) if g.dtype == a.dtype), None)
        b = live.pop(j) if j is not None else None
        rc = fn(a.data_ptr(), a.numel(), None if b is None else b.data_ptr(), 0 if b is None else b.numel(),
                _DT[a.dtype], go_ptr, st)
        if rc:
            _lib.check(rc, "dkd_scale_if_not_one")
    return grads


def _take_grads(ctx):
    """Gradients precomputed by the fused forward launch.  They are handed to autograd ONCE and rescaled in place, so a
    second backward through the same node (retain_graph=True, a loss reused in two graphs) is refused loudly instead of
    returning twice-scaled or missing gradients.  Re-run the forward for a second backward."""
    grads = ctx.grads
    if grads is None:
        raise RuntimeError("deltakd_b200: this loss was already backpropagated; the fused forward+backward kernels hold "
                           "their gradients for a single backward pass (call the criterion again instead of "
                           "retain_graph=True)")
    ctx.grads = None
    return grads


_once = torch.autograd.function.once_differentiable


# --------------------------------------------------------------------------- logit losses
_LOGIT_WS: dict = {}
_LOGIT_FN = _lib.lib.dkd_logit_kd_fwdbwd   # bound once: this call is on the per-step latency path of configs[1]


def _plain(t: torch.Tensor) -> torch.Tensor:
    """`t` without autograd history (detach() only when there is one: it costs ~4 us of host time)."""
    return t.detach() if t.requires_grad else t


def _contig(t: torch.Tensor) -> torch.Tensor:
    return t if t.is_contiguous() else t.contiguous()


def _logit_ws_bytes(B: int) -> int:
    n = _LOGIT_WS.get(B)
    if n is None:
        n = _LOGIT_WS[B] = int(_lib.lib.dkd_logit_kd_workspace_bytes(B))
    return n


class _LogitKD(torch.autograd.Function):
    @staticmethod
    def forward(ctx, outputs, outputs_kd, teacher_logits, labels, label_kind, kd_kind, smoothing, alpha, tau, parts_out, mix_lam=None):
        ref = outputs if outputs is not None else outputs_kd
        B, Cn = ref.shape
        dt = _dtype_code(ref)
        need_g0 = label_kind >= 0 and ctx.needs_input_grad[0]
        need_g1 = kd_kind != 0 and ctx.needs_input_grad[1]
        g0 = torch.empty_like(outputs) if need_g0 else None
        g1 = torch.empty_like(outputs_kd) if need_g1 else None
        loss3 = torch.empty(3, dtype=torch.float32, device=ref.device)
        st = _stream()
        ws = _workspace(ref.device, "logit_kd", _logit_ws_bytes(B), st)
        rc = _LOGIT_FN(_ptr(outputs), _ptr(outputs_kd), _ptr(teacher_logits), _ptr(labels),
                       label_kind, kd_kind, B, Cn, dt, float(smoothing), float(alpha), float(tau), _ptr(mix_lam),
                       _ptr(g0), _ptr(g1), loss3.data_ptr(), ws.data_ptr(), ws.numel(), st)
        if rc:
            _lib.check(rc, "dkd_logit_kd_fwdbwd")
        ctx.grads = (g0, g1)
        parts_out.append(loss3)  # {total, base, kd}, detached side channel for logging
        return loss3[0]

    @staticmethod
    @_once
    def backward(ctx, grad_total):
        g0, g1 = _take_grads(ctx)
        return _rescale_(grad_total, g0, g1) + (None,) * 9


_KD_KINDS = {"none": 0, "soft": 1, "hard": 2}


def logit_kd_loss(outputs, outputs_kd, teacher_logits, labels, *, kd_kind: str, smoothing: float = 0.1,
                  alpha: float = 0.0, tau: float = 1.0, return_parts: bool = False, mix_lam=None):
    """Fused base CE (+ soft / hard KD) on logits.

    labels: float [B,C] soft targets -> SoftTargetCrossEntropy; int64 [B] -> LabelSmoothingCrossEntropy(smoothing);
    None -> KD term only (returns alpha*kd).  kd_kind in {"none","soft","hard"}.
    mix_lam (fp32 device scalar, int labels only): the target of row r is timm Mixup's soft label
    lam*smooth_onehot(labels[r]) + (1-lam)*smooth_onehot(labels[B-1-r]), generated inside the kernel.
    Returns the 0-dim fp32 total `base*(1-alpha) + kd*alpha` (or base alone for "none").
    """
    kk = _KD_KINDS[kd_kind]
    ref = outputs if outputs is not None else outputs_kd
    if ref.dtype == torch.float16 or (teacher_logits is not None and teacher_logits.dtype == torch.float16) or \
            (labels is not None and labels.dtype == torch.float16):   # the reference's --amp path: exact upcast, see _f16_up
        outputs, outputs_kd, teacher_logits = _f16_up(outputs), _f16_up(outputs_kd), _f16_up(teacher_logits)
        if labels is not None and labels.dtype == torch.float16:
            labels = labels.float()
        ref = outputs if outputs is not None else outputs_kd
    _require_cuda(outputs, outputs_kd, teacher_logits, labels)
    if ref.dim() != 2:
        raise ValueError(f"logits must be [B, C], got {tuple(ref.shape)}")
    if labels is None:
        lk = -1
        outputs = None
    elif labels.dtype == torch.int64:
        lk = 1
        if labels.shape != (ref.shape[0],):
            raise ValueError(f"int labels must be [B], got {tuple(labels.shape)}")
    else:
        lk = 0
        if labels.shape != ref.shape:
            raise ValueError(f"soft labels must be [B, C] like the logits, got {tuple(labels.shape)}")
        if labels.dtype != ref.dtype:
            labels = labels.to(ref.dtype)
    if kk:
        if outputs_kd is None or teacher_logits is None:
            raise ValueError("KD needs outputs_kd and teacher_logits")
        if outputs_kd.shape != ref.shape or teacher_logits.shape != ref.shape:
            raise ValueError("outputs_kd / teacher_logits must have the shape of outputs")
        if teacher_logits.dtype != ref.dtype:
            teacher_logits = teacher_logits.to(ref.dtype)
        if outputs_kd.dtype != ref.dtype:
            raise TypeError("outputs and outputs_kd must share a dtype")
        teacher_logits = _contig(_plain(teacher_logits))
        outputs_kd = _contig(outputs_kd)
    else:
        outputs_kd = teacher_logits = None
    if outputs is not None:
        outputs = _contig(outputs)
    if labels is not None:
        labels = _contig(_plain(labels))
    if mix_lam is not None:
        if lk != 1:
            raise ValueError("mix_lam needs int64 class labels")
        mix_lam = mix_lam.detach().to(device=ref.device, dtype=torch.float32).reshape(1)
    parts = []
    total = _LogitKD.apply(outputs, outputs_kd, teacher_logits, labels, lk, kk, smoothing, alpha, tau, parts, mix_lam)
    return (total, parts[0]) if return_parts else total


# --------------------------------------------------------------------------- precision policy
_PRECISION = {"mode": None}


def set_matmul_precision(mode):
    """'bf16x3' (hi/lo split, 3 tcgen05 passes, ~2^-16: meets the fp32 parity gates), 'bf16' (one pass),
    or None = by input dtype (float32 -> bf16x3, bfloat16 -> bf16)."""
    if mode not in (None, "bf16", "bf16x3"):
        raise ValueError(mode)
    _PRECISION["mode"] = mode


def _precision_for(t: torch.Tensor) -> int:
    mode = _PRECISION["mode"]
    if mode is None:
        mode = "bf16x3" if t.dtype == torch.float32 else "bf16"
    return _lib.PREC_BF16X3 if mode == "bf16x3" else _lib.PREC_BF16


def _deterministic() -> bool:
    """True when the feature losses run in their deterministic mode (DKD_PREC_DETERMINISTIC): bit-reproducible weight,
    bias and mask-token gradients.  It follows torch state, read at every call: torch.use_deterministic_algorithms(True),
    or torch.backends.cudnn.deterministic = True, which the reference trainer sets to pin the cuDNN convolutions that
    the masked-generation kernels replace."""
    return torch.are_deterministic_algorithms_enabled() or bool(torch.backends.cudnn.deterministic)


def _grad_precision_for(t: torch.Tensor) -> int:
    """`precision` of a gradient-bearing feature entry point: _precision_for, plus the deterministic bit when requested."""
    prec = _precision_for(t)
    return prec | _lib.PREC_DETERMINISTIC if _deterministic() else prec


def _scratch(device: torch.device, tag: str, nbytes: int) -> torch.Tensor:
    """Uninitialised, 1024-byte aligned scratch cached per (device, stream, tag)."""
    key = (device.index, _stream(), "scratch:" + tag)
    ws = _WS.get(key)
    if ws is None or ws.numel() < nbytes + 1024:
        ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
        if not torch.cuda.is_current_stream_capturing():
            _WS[key] = ws
    off = (-ws.data_ptr()) % 1024
    return ws[off:off + nbytes]


# --------------------------------------------------------------------------- hidden-state matching
_LAYER_STREAMS = True   # tests switch it off to get the single-stream reference
_SIDE_STREAMS: dict = {}


def _side_streams(device: torch.device, n: int):
    """n persistent side streams of `device` (the per-layer calls of the multi-layer feature losses fork onto them)."""
    lst = _SIDE_STREAMS.setdefault(device.index if device.index is not None else torch.cuda.current_device(), [])
    while len(lst) < n:
        lst.append(torch.cuda.Stream(device=device))
    return lst[:n]


class _AlignMseLayers(torch.autograd.Function):
    """sum_i scale * || Linear_i(s_i[:, 1:]) - t_i[:, 2:] ||^2 over the selected layers (fused fwd+bwd)."""

    @staticmethod
    def forward(ctx, entry, scale, n_layers, s_off, t_off, *tensors):
        s_list = tensors[:n_layers]
        t_list = tensors[n_layers:2 * n_layers]
        w_list = tensors[2 * n_layers:3 * n_layers]
        b_list = tensors[3 * n_layers:4 * n_layers]
        dev = s_list[0].device
        # The layers are independent: each runs on its own stream (own scratch: the scratch cache is keyed by stream), so the
        # last, partly filled wave of one layer's persistent kernels (784 row tiles on 148 SMs = 5.3 waves; 512 Sinkhorn CTAs
        # = 3.5 waves) overlaps the next layer's first kernels instead of idling two thirds of the SMs.  Outputs are
        # allocated on the calling stream, which forks before the first launch and joins after the last.
        multi = n_layers > 1 and _LAYER_STREAMS
        loss_parts = torch.zeros(n_layers if multi else 1, dtype=torch.float32, device=dev)
        main = torch.cuda.current_stream(dev)
        sides = _side_streams(dev, n_layers - 1) if multi else []
        grads, outs = [], []
        for i in range(n_layers):
            s, W, b = s_list[i], w_list[i], b_list[i]
            need_s = ctx.needs_input_grad[5 + i]
            need_w = ctx.needs_input_grad[5 + 2 * n_layers + i]
            need_b = b is not None and ctx.needs_input_grad[5 + 3 * n_layers + i]
            g_s = torch.empty_like(s) if need_s else None
            g_W = torch.empty_like(W) if (need_w or need_b) else None
            g_b = torch.empty_like(b) if need_b else None
            outs.append((g_s, g_W, g_b))
            grads.append((g_s, g_W if need_w else None, g_b))
        for st in sides:
            st.wait_stream(main)
        for i in reversed(range(n_layers)):   # side streams first, the calling stream (layer 0) last
            s, t, W, b = s_list[i], t_list[i], w_list[i], b_list[i]
            B, Ts, Ds = s.shape
            _, Tt, Dt = t.shape
            n_tok = Ts - s_off
            dt = _dtype_code(s)
            prec = _grad_precision_for(s)
            g_s, g_W, g_b = outs[i]
            nbytes = getattr(_lib.lib, entry + "_workspace_bytes")(B, n_tok, Ds, Dt, prec)
            with torch.cuda.stream(main if (i == 0 or not multi) else sides[i - 1]):
                ws = _scratch(dev, entry, nbytes)
                _lib.call(entry + "_fwdbwd", _ptr(s), _ptr(t), _ptr(W), _ptr(b), B, Ts, s_off, Tt, t_off, n_tok,
                          Ds, Dt, dt, prec, float(scale), _ptr(g_s), _ptr(g_W), _ptr(g_b),
                          loss_parts.data_ptr() + (4 * i if multi else 0), _ptr(ws), ws.numel(), _stream())
        for st in sides:
            main.wait_stream(st)
        loss = loss_parts.sum() if multi else loss_parts[0]
        ctx.grads = grads
        ctx.n_layers = n_layers
        return loss

    @staticmethod
    @_once
    def backward(ctx, grad_out):
        n = ctx.n_layers
        grads = _take_grads(ctx)
        flat = [g for trip in grads for g in trip]
        _rescale_(grad_out, *flat)
        gs = [g[0] for g in grads]
        gw = [g[1] for g in grads]
        gb = [g[2] for g in grads]
        return (None, None, None, None, None, *gs, *([None] * n), *gw, *gb)


# (student, teacher) embedding widths each feature entry point's tcgen05 tile configurations are built for
_DEIT_TS = (192, 384)   # deit_tiny -> deit_small, the pair of every exp/*.sh script
_DEIT_TB = (192, 768)   # deit_tiny -> deit_base
_PAIR_NAMES = {_DEIT_TS: "deit_tiny -> deit_small", _DEIT_TB: "deit_tiny -> deit_base"}
SUPPORTED_PAIRS = {
    "dkd_align_mse": (_DEIT_TS, _DEIT_TB),
    "dkd_wass_l1": (_DEIT_TS, _DEIT_TB),
    "dkd_align_nmse": (_DEIT_TS,),
    "dkd_wass_sinkhorn": (_DEIT_TS,),
    "masked generation": (_DEIT_TS,),
    "LRKD": (_DEIT_TS,),
}
# patch-token counts (square grids, patch 16) of the entry points whose kernels are built for given grids: the generator
# convolutions and the Sinkhorn cost matrix.  Every other entry point takes any token count.
_GRID_NAMES = {196: "14 x 14 grid: 224-px inputs", 576: "24 x 24 grid: 384-px inputs"}
SUPPORTED_GRID_TOKENS = {
    "masked generation": (196, 576),
    "dkd_wass_sinkhorn": (196,),
}


def _check_feature_pair(s, t, s_off, t_off, op: str):
    """Validates one (student, teacher) feature pair for the entry point `op` (a key of SUPPORTED_PAIRS) and states the
    pairs it supports in the error: every feature loss is built for DeiT-Tiny -> DeiT-Small widths (192 -> 384), which
    is what all 19 exp/*.sh scripts of the reference use, and the hidden-state matching and WassKD-l1 losses also for a
    DeiT-Base teacher (192 -> 768).  Masked generation and Sinkhorn also check the patch-token count against
    SUPPORTED_GRID_TOKENS.  Other timm pairs (e.g. a 384-wide student) and grids are rejected here, at the first call,
    instead of failing deep inside a launch."""
    _require_cuda(s, t)
    if s.dim() != 3 or t.dim() != 3 or s.shape[0] != t.shape[0]:
        raise ValueError(f"features must be [B, tokens, dim]; got {tuple(s.shape)} and {tuple(t.shape)}")
    if s.shape[1] - s_off != t.shape[1] - t_off:
        raise ValueError(f"patch-token counts differ: student {s.shape[1] - s_off} vs teacher {t.shape[1] - t_off}")
    pairs = SUPPORTED_PAIRS[op]
    if (s.shape[2], t.shape[2]) not in pairs:
        built = " and ".join(f"{ds} -> {dt} ({_PAIR_NAMES[(ds, dt)]})" for ds, dt in pairs)
        raise ValueError(f"deltakd_b200 {op}: built for student/teacher widths {built}; got {s.shape[2]} -> {t.shape[2]}. "
                         "See INTEGRATION.md 'Supported model matrix'.")
    grids = SUPPORTED_GRID_TOKENS.get(op)
    if grids is not None and s.shape[1] - s_off not in grids:
        built = " or ".join(f"{n} patch tokens ({_GRID_NAMES[n]}, patch 16)" for n in grids)
        raise ValueError(f"deltakd_b200 {op}: built for {built}; got {s.shape[1] - s_off}. "
                         "See INTEGRATION.md 'Supported model matrix'.")


def align_mse_layers_loss(s_feats, t_feats, linears, scale: float, s_off: int = 1, t_off: int = 2,
                          _entry: str = "dkd_align_mse"):
    """scale * sum_i sum((linears[i](s_feats[i][:, s_off:]) - t_feats[i][:, t_off:])**2), 0-dim fp32."""
    n = len(linears)
    s_list, t_list, w_list, b_list = [], [], [], []
    for s, t, lin in zip(_f16_up_list(s_feats), _f16_up_list(t_feats), linears):
        _check_feature_pair(s, t, s_off, t_off, op=_entry)
        t = t.detach()
        if t.dtype != s.dtype:
            t = t.to(s.dtype)
        s_list.append(s.contiguous())
        t_list.append(t.contiguous())
        w_list.append(lin.weight.float().contiguous() if lin.weight.dtype != torch.float32 else lin.weight.contiguous())
        b_list.append(None if lin.bias is None else lin.bias.float().contiguous())
    return _AlignMseLayers.apply(_entry, scale, n, s_off, t_off, *s_list, *t_list, *w_list, *b_list)


def align_normalized_mse_loss(s_feats, t_feats, linears, s_off: int = 1, t_off: int = 2):
    """sum_i mean((normalize(linears[i](s_i[:, s_off:])) - normalize(t_i[:, t_off:]))**2), L2-normalised per token over the
    channel axis (diffkd branch, loss.py:139-140,149).  0-dim fp32; weight it with ordinary tensor arithmetic (the
    DiffKD weight w_t.mean() is a device scalar) — backward rescales the stored gradients on the device."""
    B, Ts, _ = s_feats[0].shape
    numel = B * (Ts - s_off) * t_feats[0].shape[-1]
    return align_mse_layers_loss(s_feats, t_feats, linears, 1.0 / numel, s_off, t_off, _entry="dkd_align_nmse")


def wass_l1_loss(s_feats, t_feats, linears, weight: float = 5.0, s_off: int = 1, t_off: int = 2):
    """weight * mean_i mean|sort_tokens(linears[i](s_i[:, s_off:])) - sort_tokens(t_i[:, t_off:])| (loss.py:187-199,226).
    `weight` (the reference's x5) is folded into the kernels so backward needs no rescale pass."""
    n = len(linears)
    B, Ts, _ = s_feats[0].shape
    Dt = t_feats[0].shape[-1]
    numel = B * (Ts - s_off) * Dt
    return align_mse_layers_loss(s_feats, t_feats, linears, weight / (n * numel), s_off, t_off, _entry="dkd_wass_l1")


def wass_sinkhorn_loss(s_feats, t_feats, linears, weight: float = 5.0, s_off: int = 1, t_off: int = 2):
    """weight * mean_i [ sum_b Sinkhorn(linears[i](s_i[b, s_off:]), t_i[b, t_off:]) / (B*N) ]  (loss.py:200-226), with
    Sinkhorn = geomloss.SamplesLoss("sinkhorn", blur=0.05) as restated in oracle/sinkhorn.py."""
    n = len(linears)
    B, Ts, _ = s_feats[0].shape
    return align_mse_layers_loss(s_feats, t_feats, linears, weight / (n * B * (Ts - s_off)), s_off, t_off,
                                 _entry="dkd_wass_sinkhorn")


# --------------------------------------------------------------------------- masked generation (MGD family)
class _MaskedGeneration(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scale, s_off, t_off, probe, t, mask, s, Wa, ba, mask_token, c1w, c1b, c2w, c2b):
        B, Ts, Ds = s.shape
        _, Tt, Dt = t.shape
        dev = s.device
        prec = _grad_precision_for(s)
        need = ctx.needs_input_grad[6:]
        g_s = torch.empty_like(s) if need[0] else None
        outs = [g_s]
        for flag, ref in zip(need[1:], (Wa, ba, mask_token, c1w, c1b, c2w, c2b)):
            outs.append(torch.empty_like(ref) if (flag and ref is not None) else None)
        # weight gradients come together with their bias gradient's GEMM inputs; nothing else to couple
        loss = torch.zeros((), dtype=torch.float32, device=dev)
        nbytes = _lib.lib.dkd_masked_generation_workspace_bytes(B, Ts - s_off, Ds, Dt, prec)
        ws = _scratch(dev, "mgd", nbytes)
        _lib.call("dkd_masked_generation_fwdbwd", _ptr(s), _ptr(t), _ptr(mask), _ptr(Wa), _ptr(ba), _ptr(mask_token),
                  _ptr(c1w), _ptr(c1b), _ptr(c2w), _ptr(c2b), B, Ts, s_off, Tt, t_off, Ds, Dt, _dtype_code(s), prec,
                  float(scale), *[_ptr(o) for o in outs], _ptr(loss), _ptr(ws), ws.numel(), _stream())
        if probe is not None:   # verification hook: the hidden activations (ReLU gate) the backward pass used
            P = 2 if (prec & ~_lib.PREC_DETERMINISTIC) == _lib.PREC_BF16X3 else 1
            M = B * (Ts - s_off)
            off = _lib.lib.dkd_masked_generation_hidden_offset(B, Ts - s_off, Ds, Dt, prec)
            probe["hidden"] = ws[off:off + P * M * Dt * 2].view(torch.bfloat16).view(P, B, Ts - s_off, Dt).clone()
        ctx.grads = outs
        return loss

    @staticmethod
    @_once
    def backward(ctx, grad_out):
        outs = _take_grads(ctx)
        _rescale_(grad_out, *outs)
        return (None, None, None, None, None, None, *outs)


def masked_generation_loss(s_feat, t_feat, align, mask_token, generation, *, scale: float, mask=None,
                           mask_ratio=None, noise=None, s_off: int = 1, t_off: int = 2, probe: dict | None = None):
    """scale * sum(mask * (generation(where(mask, mask_token, align(s[:, s_off:]))) - t[:, t_off:])**2).

    The patch tokens form a square grid: N = 196 (14 x 14, 224-px inputs) or 576 (24 x 24, 384-px inputs), the same N
    for student and teacher (SUPPORTED_GRID_TOKENS).
    `mask` [B,N] (1 = masked) is used if given; otherwise it is drawn like the reference's
    random_masking: noise = torch.rand(B, N, device) (misc.py:14) -> rank -> mask (dkd_mask_rank).
    `probe` (verification only): receives "mask" and "hidden" = the generator's post-ReLU activations as bf16 planes
    [P, B, N, Dt], i.e. the ReLU gate the fused backward used (tests compare gradients given that gate)."""
    s_feat, t_feat = _f16_up(s_feat), _f16_up(t_feat)
    _check_feature_pair(s_feat, t_feat, s_off, t_off, op="masked generation")
    B = s_feat.shape[0]
    L = s_feat.shape[1] - s_off
    if mask is None:
        if noise is None:
            noise = torch.rand(B, L, device=s_feat.device)
        len_keep = int(L * (1 - mask_ratio))
        mask, _, _ = mask_rank(noise, len_keep, want_shuffle=False)
    mask = mask.detach().to(torch.float32).contiguous()
    conv1, conv2 = generation[0], generation[2]
    t = t_feat.detach()
    if t.dtype != s_feat.dtype:
        t = t.to(s_feat.dtype)
    f32 = lambda x: None if x is None else (x if x.dtype == torch.float32 else x.float()).contiguous()
    if probe is not None:
        probe["mask"] = mask
    return _MaskedGeneration.apply(scale, s_off, t_off, probe, t.contiguous(), mask, s_feat.contiguous(), f32(align.weight),
                                   f32(align.bias), f32(mask_token.reshape(-1)), f32(conv1.weight), f32(conv1.bias),
                                   f32(conv2.weight), f32(conv2.bias))


# --------------------------------------------------------------------------- masking
def mask_rank(score: torch.Tensor, len_keep: int, want_shuffle: bool = True):
    """(mask fp32 [B,L], ids_restore int64 [B,L], ids_shuffle int64 [B,L] | None) from fp32 scores."""
    _require_cuda(score)
    if score.dim() != 2:
        raise ValueError("score must be [B, L]")
    score = score.detach().to(torch.float32).contiguous()
    B, L = score.shape
    mask = torch.empty(B, L, dtype=torch.float32, device=score.device)
    ids_restore = torch.empty(B, L, dtype=torch.int64, device=score.device)
    ids_shuffle = torch.empty(B, L, dtype=torch.int64, device=score.device) if want_shuffle else None
    _lib.call("dkd_mask_rank", _ptr(score), B, L, int(len_keep), _ptr(mask), _ptr(ids_restore),
              _ptr(ids_shuffle), _stream())
    return mask, ids_restore, ids_shuffle


# --------------------------------------------------------------------------- saliency scores (no gradient)
def _token_rows(x: torch.Tensor):
    """(tensor, T) such that token i of sample b starts at data_ptr + (b*T + i)*D elements; copies only if the
    view is not row-contiguous (a `feat[:, 2:]` slice of a contiguous [B, T, D] tensor is used in place)."""
    B, n, D = x.shape
    if x.stride(2) == 1 and x.stride(1) == D and (B == 1 or (x.stride(0) % D == 0 and x.stride(0) >= n * D)):
        return x, (n if B == 1 else x.stride(0) // D)
    x = x.contiguous()
    return x, n


def saliency_score_selfdiag(x, qk_weight, qk_bias, num_heads: int = 8):
    """SimpleAttention.forward (models.py:46-56): [B, N, D] tokens -> [B, N] head-mean diagonal of softmax(QK^T/sqrt(hd))."""
    _require_cuda(x, qk_weight)
    x = x.detach()
    x, T = _token_rows(x)
    B, n, D = x.shape
    prec = _precision_for(x)
    score = torch.empty(B, n, dtype=torch.float32, device=x.device)
    nbytes = _lib.lib.dkd_saliency_selfdiag_workspace_bytes(B, n, D, prec)
    ws = _scratch(x.device, "saliency", nbytes)
    f32 = lambda w: None if w is None else w.detach().float().contiguous()
    w, b = f32(qk_weight), f32(qk_bias)
    _lib.call("dkd_saliency_selfdiag_score", _ptr(x), B, T, 0, n, D, _dtype_code(x), _ptr(w), _ptr(b), num_heads, prec,
              _ptr(score), _ptr(ws), ws.numel(), _stream())
    return score


def _cls_score(xq, xq_stride, xk, xk_stride, n_keys, B, D, dt, wq, bq, wk, bk, num_heads, query_is_key, device):
    score = torch.empty(B, n_keys, dtype=torch.float32, device=device)
    _lib.call("dkd_saliency_cls_score", xq, xq_stride, xk, xk_stride, n_keys, B, D, dt, _ptr(wq), _ptr(bq), _ptr(wk),
              _ptr(bk), num_heads, query_is_key, _ptr(score), _stream())
    return score


def saliency_score_cls_row(teacher_feat, qk_weight, qk_bias, num_heads: int = 8):
    """saliency_masking method 2 (misc.py:88-116): teacher_feat [B, 2+N, D] with CLS, DIST at 0, 1; CLS-query attention
    over [CLS] + patches, head-mean, patch columns only -> [B, N]."""
    _require_cuda(teacher_feat, qk_weight)
    t = teacher_feat.detach().contiguous()
    B, Tt, D = t.shape
    w = qk_weight.detach().float().contiguous()
    b = None if qk_bias is None else qk_bias.detach().float().contiguous()
    esz = t.element_size()
    xk = C.c_void_p(t.data_ptr() + 2 * D * esz)
    wk = w[D:]
    bk = None if b is None else b[D:]
    return _cls_score(_ptr(t), Tt * D, xk, Tt * D, Tt - 2, B, D, _dtype_code(t), w, b, wk, bk, num_heads, 1, t.device)


def saliency_score_cross(x_query, x_key, q_weight, q_bias, k_weight, k_bias, num_heads: int = 8):
    """SimpleCrossAttention.forward (models.py:24-35) for one query token per sample: -> [B, 1, Nk]."""
    _require_cuda(x_query, x_key, q_weight, k_weight)
    if x_query.dim() != 3 or x_query.shape[1] != 1:
        raise ValueError("saliency_score_cross supports a single query token per sample ([B, 1, D])")
    xq = x_query.detach()
    xk, Tk = _token_rows(x_key.detach())
    if xq.dtype != xk.dtype:
        xq = xq.to(xk.dtype)
    if xq.stride(2) != 1:
        xq = xq.contiguous()
    B, n, D = xk.shape
    f32 = lambda w: None if w is None else w.detach().float().contiguous()
    s = _cls_score(_ptr(xq), xq.stride(0) if B > 1 else D, _ptr(xk), Tk * D, n, B, D, _dtype_code(xk), f32(q_weight), f32(q_bias),
                   f32(k_weight), f32(k_bias), num_heads, 0, xk.device)
    return s.unsqueeze(1)


# --------------------------------------------------------------------------- LRKD (low-rank projection matching)
def _ptr_array(tensors):
    return (C.c_void_p * len(tensors))(*[0 if t is None else t.data_ptr() for t in tensors])


class _LrkdLayers(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rank, coef, s_off, t_off, n_layers, basis_out, *tensors):
        s_list = tensors[:n_layers]
        t_list = tensors[n_layers:2 * n_layers]
        w_list = tensors[2 * n_layers:3 * n_layers]
        b_list = tensors[3 * n_layers:4 * n_layers]
        s0, t0 = s_list[0], t_list[0]
        dev = s0.device
        B, Ts, Ds = s0.shape
        _, Tt, Dt = t0.shape
        n_tok = Ts - s_off
        prec = _grad_precision_for(s0)
        dt = _dtype_code(s0)
        g_s = [torch.empty_like(s) if ctx.needs_input_grad[6 + i] else None for i, s in enumerate(s_list)]
        need_w = [ctx.needs_input_grad[6 + 2 * n_layers + i] for i in range(n_layers)]
        need_b = [b_list[i] is not None and ctx.needs_input_grad[6 + 3 * n_layers + i] for i in range(n_layers)]
        g_W = [torch.empty_like(w) if (need_w[i] or need_b[i]) else None for i, w in enumerate(w_list)]
        g_b = [torch.empty_like(b_list[i]) if need_b[i] else None for i in range(n_layers)]
        loss = torch.zeros((), dtype=torch.float32, device=dev)
        vk = [torch.empty(rank, Dt, dtype=torch.float32, device=dev) for _ in range(n_layers)] if basis_out is not None else [None] * n_layers
        sv = [torch.empty(rank, dtype=torch.float32, device=dev) for _ in range(n_layers)] if basis_out is not None else [None] * n_layers
        sweeps = torch.zeros(n_layers, dtype=torch.int32, device=dev) if basis_out is not None else None
        nbytes = _lib.lib.dkd_lrkd_workspace_bytes(n_layers, B, n_tok, Ds, Dt, rank, dt, prec)
        if nbytes == 0:
            raise ValueError(f"LRKD: unsupported geometry (layers={n_layers}, Dt={Dt})")
        ws = _scratch(dev, "lrkd", nbytes)
        coef_arr = (C.c_float * n_layers)(*[float(c) for c in coef])
        _lib.call("dkd_lrkd_fwdbwd", n_layers, _ptr_array(s_list), _ptr_array(t_list), _ptr_array(w_list), _ptr_array(b_list),
                  coef_arr, B, Ts, s_off, Tt, t_off, n_tok, Ds, Dt, rank, dt, prec, _ptr_array(g_s), _ptr_array(g_W),
                  _ptr_array(g_b), _ptr(loss), _ptr_array(vk), _ptr_array(sv), _ptr(sweeps), _ptr(ws), ws.numel(), _stream())
        if basis_out is not None:
            basis_out.update(V=vk, S=sv, sweeps=sweeps)
        ctx.grads = (g_s, [g if need_w[i] else None for i, g in enumerate(g_W)], g_b)
        ctx.n_layers = n_layers
        return loss

    @staticmethod
    @_once
    def backward(ctx, grad_out):
        n = ctx.n_layers
        gs, gw, gb = _take_grads(ctx)
        _rescale_(grad_out, *gs, *gw, *gb)
        return (None,) * 6 + (*gs, *([None] * n), *gw, *gb)


def lrkd_layers_loss(s_feats, t_feats, linears, rank: int, coef, weight: float = 1.0, s_off: int = 1, t_off: int = 2,
                     basis_out: dict | None = None):
    """weight * sum_l coef[l] * mean((T_l V_k - Linear_l(s_l[:, s_off:]))**2), T_l = t_l[:, t_off:] flattened to [B*N, Dt] and
    V_k its top-`rank` right singular vectors (loss.py:80-103, 314-330: U_k S_k == T V_k).  0-dim fp32.
    `basis_out` (dict) receives V (list of [rank, Dt]), S (singular values) and the Jacobi sweep counts."""
    n = len(linears)
    s_list, t_list, w_list, b_list = [], [], [], []
    for s, t, lin in zip(_f16_up_list(s_feats), _f16_up_list(t_feats), linears):
        _check_feature_pair(s, t, s_off, t_off, op="LRKD")
        if lin.weight.shape[0] != rank:
            raise ValueError(f"LRKD head projects to {lin.weight.shape[0]} dims but rank is {rank}")
        t = t.detach()
        if t.dtype != s.dtype:
            t = t.to(s.dtype)
        s_list.append(s.contiguous())
        t_list.append(t.contiguous())
        w_list.append(lin.weight.float().contiguous() if lin.weight.dtype != torch.float32 else lin.weight.contiguous())
        b_list.append(None if lin.bias is None else lin.bias.float().contiguous())
    coef = [float(c) * float(weight) for c in coef]
    return _LrkdLayers.apply(rank, coef, s_off, t_off, n, basis_out, *s_list, *t_list, *w_list, *b_list)


def lrkd_eigensolve(gram: torch.Tensor, k: int = 384, algo: int = 0):
    """Eigen-decomposition of symmetric PSD matrices [L, 384, 384] (fp64, cuda) by the LRKD eigensolver alone
    (dkd_lrkd_eigensolve).  Returns (W, sweeps): W[l, j, :] = lambda_j v_j in an unspecified order of j (row norms =
    eigenvalues), sweeps int32 [L].  k: leading eigenpairs wanted (the rest may be left unconverged).  The input is
    not modified."""
    if gram.dtype != torch.float64 or gram.dim() != 3 or gram.shape[1] != 384 or gram.shape[2] != 384 or not gram.is_cuda:
        raise ValueError(f"lrkd_eigensolve expects a cuda fp64 tensor [L, 384, 384], got {gram.dtype} {tuple(gram.shape)}")
    w = gram.contiguous().clone()
    sweeps = torch.zeros(w.shape[0], dtype=torch.int32, device=w.device)
    ws = _scratch(w.device, "lrkd_eig", _lib.lib.dkd_lrkd_eigensolve_workspace_bytes())
    _lib.call("dkd_lrkd_eigensolve", _ptr(w), w.shape[0], int(k), _ptr(sweeps), int(algo), _ptr(ws), ws.numel(), _stream())
    return w, sweeps


class _FixedHead:
    def __init__(self, weight):
        self.weight, self.bias = weight, None


def lrkd_projected_loss(teacher_features, student_features, rank: int, coef):
    """The reference's free function lrkd_loss (loss.py:314-330) on ALREADY projected student features [B, N, rank]
    and sliced teacher features [B, N, Dt].  Runs the same fused kernels with an identity head: the projected
    features are zero-padded to the kernel's student width (192) and matched through W = [I_rank | 0]."""
    import torch.nn.functional as F
    s_pad, heads = [], []
    for s in student_features:
        if s.shape[-1] != rank or rank > 192:
            raise ValueError(f"projected student features must be [B, N, rank<=192], got {tuple(s.shape)} for rank {rank}")
        s_pad.append(F.pad(s, (0, 192 - rank)))
        w = torch.zeros(rank, 192, dtype=torch.float32, device=s.device)
        w[:, :rank] = torch.eye(rank, device=s.device)
        heads.append(_FixedHead(w))
    return lrkd_layers_loss(s_pad, list(teacher_features), heads, rank, coef, s_off=0, t_off=0)


# --------------------------------------------------------------------------- token-stream row ops (SURVEY 8f rank 1)
class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_dtype):
        D = x.shape[-1]
        x2 = x.contiguous().view(-1, D)
        M = x2.shape[0]
        y = torch.empty(x.shape, dtype=out_dtype, device=x.device)
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        stats = torch.empty(2, M, dtype=torch.float32, device=x.device) if need else None
        if bias is not None and bias.dtype != weight.dtype:
            bias = bias.to(weight.dtype)
        _lib.call("dkd_layernorm_fwd", x2.data_ptr(), weight.data_ptr(), _ptr(bias), M, D, _DT[x2.dtype], _dtype_code(weight),
                  _DT[out_dtype], float(eps), y.data_ptr(), None if stats is None else stats[0].data_ptr(),
                  None if stats is None else stats[1].data_ptr(), _stream())
        if need:
            ctx.save_for_backward(x2, weight, stats)
            ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x2, weight, stats = ctx.saved_tensors
        M, D = x2.shape
        dy2 = dy.contiguous().view(M, D)
        dx = torch.empty_like(x2) if ctx.needs_input_grad[0] else None
        want_p = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        dgb = torch.empty(2, D, dtype=torch.float32, device=x2.device) if want_p else None
        nbytes = _lib.lib.dkd_layernorm_bwd_workspace_bytes(M, D)
        ws = _scratch(x2.device, "layernorm_bwd", nbytes)
        _lib.call("dkd_layernorm_bwd", dy2.data_ptr(), x2.data_ptr(), weight.data_ptr(), stats[0].data_ptr(), stats[1].data_ptr(),
                  M, D, _dtype_code(dy2), _DT[x2.dtype], _DT[weight.dtype], _ptr(dx), None if dgb is None else dgb[0].data_ptr(),
                  None if dgb is None else dgb[1].data_ptr(), ws.data_ptr(), ws.numel(), _stream())
        dw = dgb[0].to(weight.dtype) if ctx.needs_input_grad[1] else None
        db = dgb[1].to(weight.dtype) if (ctx.needs_input_grad[2] and ctx.has_bias) else None
        return (None if dx is None else dx.view(dy.shape)), dw, db, None, None


def layer_norm(x: torch.Tensor, weight: torch.Tensor, bias, eps: float = 1e-6, out_dtype=None) -> torch.Tensor:
    """LayerNorm over the last dimension in one pass each way (dkd_layernorm_fwd / _bwd).  `out_dtype` lets the caller
    take the normalised activations directly in the GEMM input type (under autocast: bf16) instead of casting after."""
    _require_cuda(x, weight, bias)
    return _LayerNorm.apply(x, weight, bias, eps, out_dtype or x.dtype)


def column_sum(a: torch.Tensor) -> torch.Tensor:
    """fp32 [N] = a.view(-1, N).sum(0) (dkd_colsum): the bias gradient of a Linear over a [B*T, N] token stream."""
    _require_cuda(a)
    N = a.shape[-1]
    a2 = a.contiguous().view(-1, N)
    M = a2.shape[0]
    out = torch.empty(N, dtype=torch.float32, device=a.device)
    nbytes = _lib.lib.dkd_colsum_workspace_bytes(M, N)
    ws = _scratch(a.device, "colsum", nbytes)
    _lib.call("dkd_colsum", a2.data_ptr(), M, N, _dtype_code(a2), out.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
    return out


class _LinearTokens(torch.autograd.Function):
    """y = x W^T + b on a token stream, GEMMs by cuBLAS (library GEMMs), bias gradient by dkd_colsum."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.bfloat16)
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return torch.nn.functional.linear(x, weight, bias)

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dy2 = dy.reshape(-1, dy.shape[-1])
        dx = (dy2 @ weight).view(x.shape) if ctx.needs_input_grad[0] else None
        dw = dy2.t() @ x.reshape(-1, x.shape[-1]) if ctx.needs_input_grad[1] else None
        db = None
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = column_sum(dy2).to(dy.dtype)
        return dx, dw, db


def linear_tokens(x, weight, bias):
    """nn.Linear on [.., T, K] with the bias gradient reduced by dkd_colsum (ATen's `sum(0)` of a [B*197, N] bf16 gradient
    takes 81 us per call on a B200; the column reduction is one HBM pass)."""
    N = weight.shape[0]
    if N % 8 != 0 or N > 2048 or x.numel() // x.shape[-1] < 1024:
        return torch.nn.functional.linear(x, weight, bias)   # small / odd shapes (classifier heads): library path
    return _LinearTokens.apply(x, weight, bias)


def _head_copy(src: torch.Tensor, dst: torch.Tensor) -> None:
    """dst[b,h,n,:] = src[b,h,n,:] for two [B,H,N,hd] views with arbitrary (b,h,n) strides and contiguous head rows."""
    B, H, N, hd = src.shape
    sb, sh, sn, s1 = src.stride()
    db, dh, dn, d1 = dst.stride()
    if (s1 != 1 and hd > 1) or (d1 != 1 and hd > 1) or src.dtype != dst.dtype or dst.shape != src.shape:
        raise ValueError("head copy needs same-shaped views with contiguous head rows")
    _lib.call("dkd_head_copy", src.data_ptr(), dst.data_ptr(), B, H, N, hd, src.element_size(), sb, sh, sn, db, dh, dn, _stream())


def _head_copy_ok(t: torch.Tensor) -> bool:
    e = t.element_size()
    return (t.is_cuda and t.dim() == 4 and t.stride(3) == 1 and (t.shape[3] * e) % 16 == 0 and t.data_ptr() % 16 == 0
            and all((s * e) % 16 == 0 for s in t.stride()[:3]))


class _MergeHeads(torch.autograd.Function):
    """[B,H,N,hd] attention output (any head-row strides) -> [B,N,H*hd] contiguous, one dkd_head_copy each way."""

    @staticmethod
    def forward(ctx, x):
        B, H, N, hd = x.shape
        y = torch.empty(B, N, H * hd, dtype=x.dtype, device=x.device)
        _head_copy(x, y.view(B, N, H, hd).transpose(1, 2))
        ctx.shape = (B, H, N, hd)
        return y

    @staticmethod
    def backward(ctx, dy):
        B, H, N, hd = ctx.shape
        dy = dy.contiguous()
        dx = torch.empty(B, H, N, hd, dtype=dy.dtype, device=dy.device)
        _head_copy(dy.view(B, N, H, hd).transpose(1, 2), dx)
        return dx


class _SplitQKV(torch.autograd.Function):
    """Packed projections [B,N,3*H*hd] -> q, k, v as [B,H,N,hd] views; the backward writes dq, dk, dv straight into one
    packed gradient (three dkd_head_copy launches) instead of ATen's select-backward zero fills / cat."""

    @staticmethod
    def forward(ctx, qkv, H):
        B, N, C3 = qkv.shape
        hd = C3 // (3 * H)
        ctx.dims = (B, N, H, hd)
        v5 = qkv.view(B, N, 3, H, hd)
        return tuple(v5[:, :, i].transpose(1, 2) for i in range(3))

    @staticmethod
    def backward(ctx, dq, dk, dv):
        B, N, H, hd = ctx.dims
        ref = next(g for g in (dq, dk, dv) if g is not None)
        out = torch.empty(B, N, 3, H, hd, dtype=ref.dtype, device=ref.device)
        for i, g in enumerate((dq, dk, dv)):
            dst = out[:, :, i].transpose(1, 2)
            if g is None:
                dst.zero_()
            else:
                _head_copy(g if _head_copy_ok(g) else g.contiguous(), dst)
        return out.view(B, N, 3 * H * hd), None


def split_qkv(qkv: torch.Tensor, num_heads: int):
    """q, k, v [B,H,N,hd] views of a packed [B,N,3*C] projection (see _SplitQKV)."""
    _require_cuda(qkv)
    hd = qkv.shape[-1] // (3 * num_heads)
    if not qkv.is_contiguous() or (hd * qkv.element_size()) % 16 != 0:
        B, N, _ = qkv.shape
        return qkv.reshape(B, N, 3, num_heads, hd).permute(2, 0, 3, 1, 4).unbind(0)
    return _SplitQKV.apply(qkv, num_heads)


def merge_heads(x: torch.Tensor) -> torch.Tensor:
    """[B,H,N,hd] -> [B,N,H*hd] (a view when the strides already allow it)."""
    _require_cuda(x)
    B, H, N, hd = x.shape
    t = x.transpose(1, 2)
    if t.is_contiguous():
        return t.reshape(B, N, H * hd)
    if not _head_copy_ok(x):
        return t.reshape(B, N, H * hd)
    return _MergeHeads.apply(x)
