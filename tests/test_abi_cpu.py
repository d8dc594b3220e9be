"""CPU tier: the C-ABI shared library builds, loads and exports every symbol that include/npgp.h declares (no compute
call is made: there is no GPU here), and the product refuses to run without CUDA instead of falling back."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "npgp.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(npgp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from nonstationary_precip_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "run `python -m nonstationary_precip_b200.build` (or __graft_entry__.build())"
    handle = ctypes.CDLL(_lib.LIB_PATH)
    syms = declared_symbols()
    assert len(syms) >= 25
    missing = [s for s in syms if not hasattr(handle, s)]
    assert not missing, missing
    # every declared symbol has a ctypes signature in the binding, and vice versa
    assert set(syms) == set(_lib.exported_symbols())
    assert handle.npgp_version() == 100


def test_no_cpu_fallback():
    from nonstationary_precip_b200 import ops
    from nonstationary_precip_b200._lib import NpgpError
    x = torch.rand(4, 2, dtype=torch.float64)
    ell = torch.ones(2, 4, dtype=torch.float64)
    with pytest.raises((NpgpError, RuntimeError)):
        ops.gibbs_diag_fwd(x, ell, x, ell)


def test_argument_errors_are_reported_without_a_gpu():
    from nonstationary_precip_b200 import _lib
    lib = _lib.lib()
    assert lib.npgp_gibbs_diag_fwd(2, -1, 4, None, None, None, None, None, None, 4, None, None, None) == -1
    assert lib.npgp_potrf_workspace_bytes(1024) > 8 * 1024 * 1024


def test_int8_gemm_argument_errors_without_a_gpu():
    """npgp_rowquad_i8 / npgp_syrk_i8 validate shapes, alignment and workspace before any launch."""
    from nonstationary_precip_b200 import _lib
    lib = _lib.lib()
    a = 4096  # fake, 16-byte aligned device addresses: the calls below must return before touching them
    assert lib.npgp_rowquad_i8_workspace_bytes(65536, 1024) >= 65536 * 1024 * 7 + 1024 * 1024 * 7  # 7 byte digits
    assert lib.npgp_rowquad_i8(10, 48, a, 48, a, 48, a, 48, None, a, 1 << 40, None) == -2     # M % 64 != 0
    assert lib.npgp_rowquad_i8(10, 64, a, 63, a, 64, a, 64, None, a, 1 << 40, None) == -2     # odd ldk
    assert lib.npgp_rowquad_i8(10, 64, a + 8, 64, a, 64, a, 64, None, a, 1 << 40, None) == -2  # K not 16-byte aligned
    assert lib.npgp_rowquad_i8(10, 64, a, 64, a, 64, a, 64, None, a, 16, None) == -3           # workspace too small
    assert lib.npgp_rowquad_i8(10, 64, None, 64, a, 64, a, 64, None, a, 1 << 40, None) == -1   # NULL operand
    assert lib.npgp_rowquad_i8(0, 64, None, 64, None, 64, None, 64, None, None, 0, None) == 0  # empty: nothing to do
    assert lib.npgp_syrk_i8(10, 192, 1.0, a, 192, None, None, 0.0, 0, a, 192, a, 1 << 40, None) == -2  # M % 128 != 0
    assert lib.npgp_syrk_i8(10, 128, 1.0, a, 128, None, None, 0.0, 0, a, 128, a, 16, None) == -3
