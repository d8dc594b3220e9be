"""CPU tier of the C-ABI posterior sampler (npgp_svgp_sample_workspace_bytes / _sample_prepare / _sample): argument errors
without a device, the size of the caller's sample workspace, and the declarations in include/npgp.h."""
import ctypes
import os

import pytest

from svgp_cases import make_problem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cfg(variant=0, d=2, M=256, B=1000):
    from nonstationary_precip_b200._lib import SvgpConfig
    return SvgpConfig(variant=variant, d=d, M=M, B_local=B, N_total=1 << 20, B_global=B, world_size=1)


def test_sample_entry_points_reject_a_null_plan():
    from nonstationary_precip_b200._lib import lib
    a = 4096  # fake device addresses: the calls must return before touching them
    assert lib().npgp_svgp_sample_prepare(None, a, 16, 0, a, 1 << 40, None) == -1
    assert lib().npgp_svgp_sample(None, 10, a, 0, a, 0, a, 10, a, 1 << 40, None) == -1
    assert lib().npgp_o8_gemm_digits(-1, 64, 128, a, None, a, a, a, a, 64, None) == -1


def test_sample_workspace_rejects_bad_sample_counts_and_configs():
    from nonstationary_precip_b200._lib import lib
    c = cfg()
    for S in (0, -3, 1025):
        assert lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(c), S) == -1
    assert lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(c), 1024) > 0
    assert lib().npgp_svgp_sample_workspace_bytes(None, 16) == -1
    assert lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(cfg(M=200)), 16) == -1  # M % 128
    assert lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(cfg(variant=1, d=4)), 16) == -1


@pytest.mark.parametrize("variant,d,M,B", [(0, 2, 1024, 65536), (1, 3, 128, 640)])
def test_sample_workspace_grows_with_the_padded_sample_count(variant, d, M, B):
    from nonstationary_precip_b200._lib import lib
    c = cfg(variant, d, M, B)
    size = lambda S: lib().npgp_svgp_sample_workspace_bytes(ctypes.byref(c), S)
    assert size(1) == size(16) == size(64)
    assert size(65) == size(128) > size(64)
    # per 64 more draws: W^T and E^T Ls^T (64 x M doubles each), the planes of W^T (64 x M x 7 bytes) and exponents, and the
    # B_local x 64 chunk of K W, each rounded up to 256 bytes
    per64 = 2 * 64 * M * 8 + 64 * M * 7 + 64 * 4 + B * 64 * 8
    assert 0 <= size(128) - size(64) - per64 < 4 * 256
    # G = P^T P and its planes come once
    assert size(64) > M * M * 8 + M * M * 7 + per64


def test_sample_symbols_are_declared():
    from test_abi_cpu import declared_symbols
    syms = declared_symbols()
    for s in ("npgp_svgp_sample_workspace_bytes", "npgp_svgp_sample_prepare", "npgp_svgp_sample", "npgp_o8_gemm_digits"):
        assert s in syms


def test_sample_needs_m_multiple_of_128():
    from nonstationary_precip_b200.svgp import SVGPGibbs
    x, y, Z, kw, N = make_problem("diag", B=32, M=24, d=2)
    model = SVGPGibbs("diag", Z, N, **kw)
    with pytest.raises(ValueError):
        model.sample(x, 4)
