"""ctypes binding of libdeltakd_sm100.so (C ABI declared in include/deltakd.h).

There is no fallback: if the shared library has not been built, importing this
module raises, and every compute call on a non-sm_100 device raises
RuntimeError(dkd_last_error()).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdeltakd_sm100.so")

F32, BF16 = 0, 1
PREC_BF16, PREC_BF16X3 = 0, 1
PREC_DETERMINISTIC = 0x100   # OR'ed into the precision of the gradient-bearing feature entry points
OK = 0

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python deltakd_b200/csrc/build.py` "
        "(deltakd_b200 has no CPU or eager fallback)")

lib = C.CDLL(LIB_PATH)

_p, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); tests/test_abi.py checks this table against include/deltakd.h
SIGNATURES = {
    "dkd_version": (_i, []),
    "dkd_last_error": (C.c_char_p, []),
    "dkd_check_device": (_i, []),
    "dkd_launch_count": (C.c_ulonglong, []),
    "dkd_logit_kd_workspace_bytes": (_sz, [_i64]),
    "dkd_logit_kd_fwdbwd": (_i, [_p, _p, _p, _p, _i, _i, _i64, _i64, _i, _f, _f, _f, _p, _p, _p, _p, _p, _sz, _p]),
    "dkd_step_workspace_bytes": (_sz, []),
    "dkd_step_epilogue": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _p, C.c_double, C.c_double, _f, _f, _f, C.c_double, _i, _f, _f, _i, _i, _p, _p,
                               _sz, _p]),
    "dkd_topk_hits": (_i, [_p, _p, _i64, _i64, _i, _i, _i, _p, _p]),
    "dkd_mix_batch": (_i, [_p, _i64, _i64, _i, _i, _p, _i, _i, _i, _i, _i, _p]),
    "dkd_mask_rank": (_i, [_p, _i64, _i64, _i64, _p, _p, _p, _p]),
    "dkd_scale_if_not_one": (_i, [_p, _i64, _p, _i64, _i, _p, _p]),
    "dkd_align_mse_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i]),
    "dkd_masked_generation_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i]),
    "dkd_masked_generation_hidden_offset": (_sz, [_i64, _i, _i, _i, _i]),
    "dkd_masked_generation_fwdbwd": (_i, [_p] * 10 + [_i64, _i, _i, _i, _i, _i, _i, _i, _i, _f] + [_p] * 10 + [_sz, _p]),
    "dkd_align_nmse_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i]),
    "dkd_align_nmse_fwdbwd": (_i, [_p, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p, _p, _p, _p, _p, _sz, _p]),
    "dkd_wass_l1_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i]),
    "dkd_wass_l1_fwdbwd": (_i, [_p, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p, _p, _p, _p, _p, _sz, _p]),
    "dkd_wass_sinkhorn_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i]),
    "dkd_wass_sinkhorn_fwdbwd": (_i, [_p, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p, _p, _p, _p, _p, _sz, _p]),
    "dkd_saliency_selfdiag_workspace_bytes": (_sz, [_i64, _i, _i, _i]),
    "dkd_saliency_selfdiag_score": (_i, [_p, _i64, _i, _i, _i, _i, _i, _p, _p, _i, _i, _p, _p, _sz, _p]),
    "dkd_saliency_cls_score": (_i, [_p, _i64, _p, _i64, _i, _i64, _i, _i, _p, _p, _p, _p, _i, _i, _p, _p]),
    "dkd_lrkd_workspace_bytes": (_sz, [_i, _i64, _i, _i, _i, _i, _i, _i]),
    "dkd_lrkd_fwdbwd": (_i, [_i, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p,
                             _p, _sz, _p]),
    "dkd_lrkd_eigensolve_workspace_bytes": (_sz, []),
    "dkd_lrkd_eigensolve": (_i, [_p, _i, _i, _p, _i, _p, _sz, _p]),
    "dkd_layernorm_fwd": (_i, [_p, _p, _p, _i64, _i, _i, _i, _i, _f, _p, _p, _p, _p]),
    "dkd_layernorm_bwd_workspace_bytes": (_sz, [_i64, _i]),
    "dkd_layernorm_bwd": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _i, _i, _p, _p, _p, _p, _sz, _p]),
    "dkd_head_copy": (_i, [_p, _p, _i64, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _i64, _i64, _p]),
    "dkd_colsum_workspace_bytes": (_sz, [_i64, _i]),
    "dkd_colsum": (_i, [_p, _i64, _i, _i, _p, _p, _sz, _p]),
    "dkd_align_mse_fwdbwd": (_i, [_p, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p, _p, _p, _p, _p, _sz, _p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return (lib.dkd_last_error() or b"").decode()


def check(rc: int, what: str) -> None:
    if rc != OK:
        raise RuntimeError(f"{what} failed ({rc}): {last_error()}")


def call(name: str, *args) -> None:
    check(getattr(lib, name)(*args), name)
