"""CPU tier of the streamed SGPR prediction entries (npgp_o8_trinorm_digits, npgp_sgpr_predict_finish,
npgp_sgpr_rownorm_parts): declarations in include/npgp.h, exports of libnpgp.so, and argument errors without a device."""
import ctypes

import pytest

NEW = ("npgp_o8_trinorm_digits", "npgp_sgpr_predict_workspace_bytes", "npgp_sgpr_predict_finish", "npgp_sgpr_rownorm_parts")


def test_sgpr_predict_symbols_are_declared_bound_and_exported():
    from test_abi_cpu import declared_symbols
    from nonstationary_precip_b200 import _lib
    syms = declared_symbols()
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for s in NEW:
        assert s in syms and s in _lib.exported_symbols() and hasattr(handle, s)


A = 4096  # fake device addresses: every call below must return before touching them


def trinorm(n=256, N=256, Kd=256, Ms=0, a=A, a_expo=None, a_scale=A, b=A, b_expo=A, q=A, q_stride=256):
    from nonstationary_precip_b200._lib import lib
    return lib().npgp_o8_trinorm_digits(n, N, Kd, Ms, a, a_expo, a_scale, b, b_expo, q, q_stride, None)


@pytest.mark.parametrize("kw", [dict(a=None), dict(a_scale=None), dict(b=None), dict(b_expo=None), dict(q=None),
                                dict(N=96), dict(N=100), dict(Kd=0), dict(Kd=-32), dict(Kd=48), dict(Kd=16416, N=16448),
                                dict(Ms=32), dict(Ms=-64), dict(Ms=256), dict(Ms=320), dict(q_stride=255), dict(n=-1)])
def test_trinorm_rejects_bad_arguments(kw):
    assert trinorm(**kw) == -1


def test_finish_and_rownorm_reject_bad_arguments():
    from nonstationary_precip_b200._lib import lib
    fin = lib().npgp_sgpr_predict_finish
    # (n, qn, qn_stride, nb_t, nb_s, qv, qv_stride, nb_v, mean, y, s, noise, os_t, var_f, var_y, lpd, sums, work, bytes, stream)
    ok = [100, A, 100, 0, 2, A, 100, 2, A, A, A, A, None, A, A, A, A, A, 1 << 20, None]
    bad = {1: None, 2: 99, 3: -1, 5: None, 6: 50, 10: None, 11: None, 13: None, 17: None, 18: 8}
    for k, v in bad.items():
        args = list(ok)
        args[k] = v
        assert fin(*args) == -1, k
    args = list(ok)
    args[3] = 1  # a temporal component needs os_t
    assert fin(*args) == -1
    args = list(ok)
    args[9] = None  # sums and lpd need y
    assert fin(*args) == -1
    assert lib().npgp_sgpr_predict_workspace_bytes(-1) == -1
    assert lib().npgp_sgpr_predict_workspace_bytes(65536) >= 2 * 256 * 8
    rn = lib().npgp_sgpr_rownorm_parts
    assert rn(10, 64, None, 64, A, 10, None) == -1
    assert rn(10, 64, A, 63, A, 10, None) == -1
    assert rn(10, 64, A, 64, A, 9, None) == -1
    assert rn(-1, 64, A, 64, A, 10, None) == -1
