"""CPU tier of the C-ABI prediction (npgp_svgp_predict_prepare / npgp_svgp_predict): argument errors without a device, and the
plan's workspace and theta sizes, which prediction must not grow (it streams rows through the training step's buffers)."""
import ctypes

import pytest
import torch

from svgp_cases import make_problem


def test_predict_entry_points_reject_a_null_plan():
    from nonstationary_precip_b200._lib import lib
    a = 4096  # fake device addresses: the calls must return before touching them
    assert lib().npgp_svgp_predict_prepare(None, a, None, None) == -1
    assert lib().npgp_svgp_predict(None, 10, a, None, a, a, a, None, None, None, None, None) == -1


@pytest.mark.parametrize("variant,d,M,B,ws_bytes,theta", [(1, 3, 1024, 65536, 1246604036, 1055756),
                                                          (0, 2, 1024, 65536, 1257379076, 1053698),
                                                          (1, 3, 128, 640, 4092676, 17292),
                                                          (0, 3, 256, 1000, 16699652, 67330)])
def test_workspace_and_theta_sizes_unchanged(variant, d, M, B, ws_bytes, theta):
    from nonstationary_precip_b200._lib import SvgpConfig, lib
    cfg = SvgpConfig(variant=variant, d=d, M=M, B_local=B, N_total=1 << 20, B_global=B, world_size=1)
    assert lib().npgp_svgp_workspace_bytes(ctypes.byref(cfg)) == ws_bytes
    assert lib().npgp_svgp_theta_size(ctypes.byref(cfg)) == theta


def test_predictive_needs_m_multiple_of_128():
    from nonstationary_precip_b200.svgp import SVGPGibbs
    x, y, Z, kw, N = make_problem("diag", B=32, M=24, d=2)
    model = SVGPGibbs("diag", Z, N, **kw)
    with pytest.raises(ValueError):
        model.predictive(x, y)
