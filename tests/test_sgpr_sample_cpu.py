"""CPU tier of the SGPR posterior sampler's entries (npgp_sample_normals, npgp_sgpr_sample_finish, and the digit contraction
npgp_o8_gemm_digits that sgpr.py now wraps): declarations in include/npgp.h, exports of libnpgp.so, and argument errors
without a device."""
import ctypes

import pytest

NEW = ("npgp_sample_normals", "npgp_sgpr_sample_finish", "npgp_o8_gemm_digits")

A = 4096  # fake device addresses: every call below must return before touching them


def test_sgpr_sample_symbols_are_declared_bound_and_exported():
    from test_abi_cpu import declared_symbols
    from nonstationary_precip_b200 import _lib, ops
    syms = declared_symbols()
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for s in NEW:
        assert s in syms and s in _lib.exported_symbols() and hasattr(handle, s)
    assert callable(ops.o8_gemm_digits) and callable(ops.sample_normals) and callable(ops.sgpr_sample_finish)


def finish(**kw):
    from nonstationary_precip_b200._lib import lib
    a = dict(n=100, S=16, mean=A, qn=A, qn_stride=100, nb_t=0, nb_s=2, F=A, ldf=64, s=A, noise=A, os_t=None, add_noise=0,
             seed=1, row0=0, out=A, ldo=100)
    a.update(kw)
    return lib().npgp_sgpr_sample_finish(*a.values(), None)


@pytest.mark.parametrize("kw", [dict(n=-1), dict(S=0), dict(S=1025), dict(nb_t=-1), dict(nb_s=-1), dict(row0=-1),
                                dict(row0=(1 << 48) - 99), dict(mean=None), dict(F=None), dict(s=None), dict(out=None),
                                dict(ldf=15), dict(ldo=99), dict(nb_t=1), dict(add_noise=1, noise=None), dict(qn=None),
                                dict(qn_stride=99)])
def test_finish_rejects_bad_arguments(kw):
    assert finish(**kw) == -1


def test_finish_accepts_the_edges_of_its_ranges_without_launching_on_empty_input():
    assert finish(n=0) == 0  # nothing to do: returns before any pointer is looked at
    assert finish(n=0, mean=None, F=None, out=None) == 0
    assert finish(n=0, row0=1 << 48) == 0


def test_sample_normals_rejects_bad_arguments():
    from nonstationary_precip_b200._lib import lib
    f = lib().npgp_sample_normals
    assert f(-1, 4, 64, 0, A, None) == -1
    assert f(64, -1, 64, 0, A, None) == -1
    assert f(64, 65, 64, 0, A, None) == -1  # Sp < S
    assert f(64, 4, 64, 0, None, None) == -1
    assert f(0, 4, 64, 0, None, None) == 0 and f(64, 0, 0, 0, None, None) == 0  # empty: nothing to write


def test_sample_argument_errors_come_before_any_device_work():
    import torch
    from nonstationary_precip_b200.sgpr import SGPRPosterior
    post = SGPRPosterior.__new__(SGPRPosterior)  # the checks run before the snapshot is touched
    x = torch.zeros(10, 2, dtype=torch.float64)
    for S in (0, 1025):
        with pytest.raises(ValueError):
            post.sample(x, S)
    with pytest.raises(ValueError):
        post.sample(x, 4, row_offset=-1)
    with pytest.raises(ValueError):
        post.sample(x, 4, row_offset=(1 << 48) - 9)
