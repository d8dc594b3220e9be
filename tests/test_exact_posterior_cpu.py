"""CPU tier of the exact Gibbs GP's posterior snapshot (DiagonalExactGP.posterior): the finishing kernel's declaration in
include/npgp.h, its export and binding, its argument errors without a device, the snapshot's argument errors, and the map
options of experiments/spatial_exp.py."""
import ctypes

import pytest
import torch

A = 4096  # fake device addresses: every call below must return before touching them


def test_exact_finish_is_declared_bound_and_exported():
    from test_abi_cpu import declared_symbols
    from nonstationary_precip_b200 import _lib, ops
    s = "npgp_exact_predict_finish"
    assert s in declared_symbols() and s in _lib.exported_symbols() and hasattr(ctypes.CDLL(_lib.LIB_PATH), s)
    assert callable(ops.exact_predict_finish)


def finish(**kw):
    from nonstationary_precip_b200._lib import lib
    a = dict(n=100, qn=A, qn_stride=100, nb=2, mean=A, y=A, s=A, noise=A, add_var=1e-4, var_f=A, var_y=A, lpd=A, sums=A,
             work=A, work_bytes=1 << 20)
    a.update(kw)
    return lib().npgp_exact_predict_finish(*a.values(), None)


@pytest.mark.parametrize("kw", [dict(n=-1), dict(nb=-1), dict(s=None), dict(noise=None), dict(var_f=None), dict(y=None),
                                dict(mean=None), dict(qn=None), dict(qn_stride=99), dict(work=None), dict(work_bytes=8)])
def test_exact_finish_rejects_bad_arguments(kw):
    assert finish(**kw) == -1


def test_exact_finish_returns_on_empty_input():
    assert finish(n=0) == 0
    assert finish(n=0, qn=None, s=None, var_f=None) == 0


def small_model(n=5, D=2):
    from nonstationary_precip_b200.gp_base import GaussianLikelihood
    from nonstationary_precip_b200.models.gibbs_kernels import LogNormalPriorProcess
    from nonstationary_precip_b200.models.nonstationary_models import DiagonalExactGP
    g = torch.Generator().manual_seed(0)
    x, y = torch.rand(n, D, generator=g, dtype=torch.float64), torch.rand(n, generator=g, dtype=torch.float64)
    return DiagonalExactGP(x, y, GaussianLikelihood().double(), LogNormalPriorProcess(input_dim=D).double(),
                           num_dim=D).double()


@pytest.mark.parametrize("shape", [(3, 3), (3,), (2, 1, 2)])
def test_posterior_rejects_knots_of_the_wrong_shape(shape):
    with pytest.raises(ValueError, match="knots must have shape"):
        small_model().posterior(knots=torch.zeros(*shape, dtype=torch.float64))


def test_posterior_rejects_more_columns_than_the_digit_engine_takes():
    with pytest.raises(ValueError, match="16384"):
        small_model(n=5).posterior(knots=torch.zeros(16380, 2, dtype=torch.float64))  # 16385 columns, padded to 16512


def test_sample_argument_errors_come_before_any_device_work():
    from nonstationary_precip_b200.sgpr import SGPRPosterior
    post = SGPRPosterior.__new__(SGPRPosterior)  # DiagonalExactGP.posterior returns this class; checks run first
    x = torch.zeros(10, 2, dtype=torch.float64)
    for S in (0, 1025):
        with pytest.raises(ValueError):
            post.sample(x, S)
    for off in (-1, (1 << 48) - 9):
        with pytest.raises(ValueError):
            post.sample(x, 4, row_offset=off)


def test_spatial_exp_map_options_default_to_off():
    from experiments import spatial_exp as se
    a = se.parse_args([])
    assert a.map_grid == 0 and a.map_samples == 0
    b = se.parse_args(["--map_grid", "64", "--map_samples", "4", "--map_out", "m.npz"])
    assert (b.map_grid, b.map_samples, b.map_out) == (64, 4, "m.npz")
    assert {k: v for k, v in vars(b).items() if not k.startswith("map_")} == \
        {k: v for k, v in vars(a).items() if not k.startswith("map_")}
