"""CPU: how `functional` selects the deterministic mode of the feature losses from torch state, and the flag's value in
the ctypes binding against include/deltakd.h."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def flags():
    was_alg, was_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    was_cudnn = torch.backends.cudnn.deterministic
    torch.use_deterministic_algorithms(False)
    torch.backends.cudnn.deterministic = False
    yield
    torch.use_deterministic_algorithms(was_alg, warn_only=was_warn)
    torch.backends.cudnn.deterministic = was_cudnn


def test_header_and_binding_agree():
    from deltakd_b200 import _lib
    src = open(os.path.join(ROOT, "include", "deltakd.h")).read()
    m = re.search(r"DKD_PREC_DETERMINISTIC\s*=\s*(0x[0-9a-fA-F]+|\d+)", src)
    assert m is not None
    assert int(m.group(1), 0) == _lib.PREC_DETERMINISTIC == 0x100
    assert _lib.PREC_DETERMINISTIC & (_lib.PREC_BF16 | _lib.PREC_BF16X3) == 0


@pytest.mark.parametrize("how", [None, "torch", "torch_warn_only", "cudnn", "both"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_flag_selection(flags, how, dtype):
    from deltakd_b200 import _lib
    from deltakd_b200 import functional as Fn
    if how in ("torch", "both"):
        torch.use_deterministic_algorithms(True)
    if how == "torch_warn_only":
        torch.use_deterministic_algorithms(True, warn_only=True)
    if how in ("cudnn", "both"):
        torch.backends.cudnn.deterministic = True
    x = torch.zeros(1, dtype=dtype)
    base = _lib.PREC_BF16X3 if dtype == torch.float32 else _lib.PREC_BF16
    assert Fn._precision_for(x) == base                 # saliency and every other caller: never the bit
    want = base | _lib.PREC_DETERMINISTIC if how else base
    assert Fn._deterministic() == bool(how)
    assert Fn._grad_precision_for(x) == want


def test_selection_is_read_at_each_call(flags):
    from deltakd_b200 import _lib
    from deltakd_b200 import functional as Fn
    x = torch.zeros(1)
    assert not Fn._grad_precision_for(x) & _lib.PREC_DETERMINISTIC
    torch.backends.cudnn.deterministic = True
    assert Fn._grad_precision_for(x) & _lib.PREC_DETERMINISTIC
    torch.backends.cudnn.deterministic = False
    assert not Fn._grad_precision_for(x) & _lib.PREC_DETERMINISTIC


def test_workspace_queries_without_a_device():
    """The workspace sizes of the mode depend on the shapes only: they are answered on a machine without a GPU, grow
    with the flag, and the masked-generation hidden activations do not move."""
    from deltakd_b200 import _lib
    lib, DET = _lib.lib, _lib.PREC_DETERMINISTIC
    for base in (_lib.PREC_BF16, _lib.PREC_BF16X3):
        for B in (1, 37, 512):
            for fn, Dts in (("dkd_align_mse", (384, 768)), ("dkd_wass_l1", (384, 768)), ("dkd_align_nmse", (384,)),
                            ("dkd_wass_sinkhorn", (384,)), ("dkd_masked_generation", (384,))):
                ws = getattr(lib, fn + "_workspace_bytes")
                for Dt in Dts:
                    assert ws(B, 196, 192, Dt, base | DET) > ws(B, 196, 192, Dt, base), (fn, Dt, B)
            for dt in (_lib.F32, _lib.BF16):
                assert lib.dkd_lrkd_workspace_bytes(3, B, 196, 192, 384, 32, dt, base | DET) > \
                    lib.dkd_lrkd_workspace_bytes(3, B, 196, 192, 384, 32, dt, base)
            assert lib.dkd_masked_generation_hidden_offset(B, 196, 192, 384, base | DET) == \
                lib.dkd_masked_generation_hidden_offset(B, 196, 192, 384, base)
