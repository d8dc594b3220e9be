"""CPU tier of the regional-sum posterior (npgp_gibbs_*_segsum, npgp_segment_colwsum, npgp_svgp_region_moments): every
documented argument error before any launch, the workspace queries, the declarations in include/npgp.h and the label -> offsets
helper of SVGPGibbs.region_posterior."""
import ctypes

import pytest
import torch

A = 4096  # fake, 256-byte aligned device addresses: the calls below must return before touching them


def cfg(variant=0, d=2, M=256, B=1000):
    from nonstationary_precip_b200._lib import SvgpConfig
    return SvgpConfig(variant=variant, d=d, M=M, B_local=B, N_total=1 << 20, B_global=B, world_size=1)


def diag(D=2, n=10, x=A, ell=A, R=3, seg=A, full=1, part=0, nparts=1, Gd=A, G=A, ldg=3, work=A, nbytes=1 << 40):
    from nonstationary_precip_b200._lib import lib
    return lib().npgp_gibbs_diag_segsum(D, n, x, ell, None, R, seg, full, part, nparts, None, Gd, G, ldg, work, nbytes, None)


def full(d=3, n=10, S=A, R=3, full=1, ldg=3, work=A, nbytes=1 << 40):
    from nonstationary_precip_b200._lib import lib
    return lib().npgp_gibbs_full_segsum(d, n, A, S, 1e-5, None, R, A, full, 0, 1, None, A, A, ldg, work, nbytes, None)


def test_pair_sum_argument_errors_before_any_launch():
    from nonstationary_precip_b200._lib import lib
    assert diag(R=0) == -1 and diag(n=-1) == -1 and diag(n=1 << 31) == -1
    assert diag(D=0) == -1 and diag(D=7) == -1 and full(d=4) == -1 and full(d=1) == -1
    assert diag(x=None) == -1 and diag(ell=None) == -1 and diag(seg=None) == -1 and diag(Gd=None) == -1
    assert diag(work=None) == -1 and full(S=None) == -1
    assert diag(G=None) == -1  # G is needed with full
    assert diag(part=1, nparts=1) == -1 and diag(part=-1) == -1 and diag(nparts=0) == -1
    assert diag(ldg=2) == -1 and full(ldg=2) == -1
    assert diag(work=A + 8) == -2 and full(work=A + 16) == -2
    need = lib().npgp_segsum_workspace_bytes(10, 3, 1)
    assert diag(nbytes=need - 1) == -3 and full(nbytes=need - 1) == -3
    assert diag(full=0, G=None, nbytes=lib().npgp_segsum_workspace_bytes(10, 3, 0) - 1) == -3


def test_segment_colwsum_argument_errors_before_any_launch():
    from nonstationary_precip_b200._lib import lib
    f = lambda n=10, M=8, K=A, ldk=8, R=2, seg=A, out=A, ldo=8, work=A, nb=1 << 30, row0=0: lib().npgp_segment_colwsum(
        n, M, K, ldk, None, row0, R, seg, out, ldo, work, nb, None)
    assert f(n=-1) == -1 and f(M=0) == -1 and f(R=0) == -1 and f(ldk=7) == -1 and f(ldo=7) == -1 and f(row0=-1) == -1
    assert f(K=None) == -1 and f(seg=None) == -1 and f(out=None) == -1 and f(work=None) == -1
    assert f(work=A + 4) == -2
    assert f(nb=lib().npgp_segment_colwsum_workspace_bytes(10, 8) - 1) == -3
    assert f(n=0, K=None) == 0  # nothing to add
    assert lib().npgp_segment_colwsum_workspace_bytes(-1, 8) == -1 and lib().npgp_segment_colwsum_workspace_bytes(8, 0) == -1


def test_region_moments_argument_errors_before_any_launch():
    from nonstationary_precip_b200._lib import lib
    assert lib().npgp_svgp_region_moments(None, 10, A, None, 3, A, A, 0, 0, 1, A, A, None, 3, A, 1 << 40, None) == -1


def test_workspace_queries_are_monotone_and_reject_bad_arguments():
    from nonstationary_precip_b200._lib import lib
    seg = lambda n, R, f: lib().npgp_segsum_workspace_bytes(n, R, f)
    assert seg(-1, 3, 0) == -1 and seg(1 << 31, 3, 0) == -1 and seg(10, 0, 0) == -1
    c = cfg()
    reg = lambda n, R, f, cf=c: lib().npgp_svgp_region_workspace_bytes(ctypes.byref(cf), n, R, f)
    assert reg(-1, 3, 1) == -1 and reg(10, 0, 1) == -1 and reg(1 << 31, 3, 1) == -1
    assert lib().npgp_svgp_region_workspace_bytes(None, 10, 3, 1) == -1
    assert reg(10, 3, 1, cfg(M=200)) == -1 and reg(10, 3, 1, cfg(variant=1, d=4)) == -1
    for f in (0, 1):
        for sizes in ([0, 1, 255, 256, 257, 5000, 1 << 16, 1 << 20], ):
            for R in (1, 7, 64, 1024):
                a = [seg(n, R, f) for n in sizes]
                b = [reg(n, R, f) for n in sizes]
                assert a == sorted(a) and b == sorted(b) and min(a) > 0 and min(b) > 0
            for n in (100, 1 << 20):
                a = [seg(n, R, f) for R in (1, 2, 64, 1024, 1 << 14)]
                b = [reg(n, R, f) for R in (1, 2, 64, 1024, 1 << 14)]
                assert a == sorted(a) and b == sorted(b)
    assert seg(1 << 20, 1024, 1) > seg(1 << 20, 1024, 0)
    # the full matrix at n = 2^20 rows and 1024 regions: at most (4096 + 1023)^2 / 2 item partials
    assert seg(1 << 20, 1024, 1) < 8 * 5120 * 5121 // 2 + 64 * 1024


def test_region_symbols_are_declared():
    from test_abi_cpu import declared_symbols
    syms = declared_symbols()
    for s in ("npgp_segsum_workspace_bytes", "npgp_gibbs_diag_segsum", "npgp_gibbs_full_segsum", "npgp_segment_colwsum",
              "npgp_segment_colwsum_workspace_bytes", "npgp_svgp_region_workspace_bytes", "npgp_svgp_region_moments"):
        assert s in syms


def test_label_to_offsets_helper_on_cpu_tensors():
    from nonstationary_precip_b200.svgp import region_segments
    g = torch.Generator().manual_seed(0)
    for R in (1, 5, 40):
        labels = torch.randint(0, R, (300,), generator=g)
        order, seg = region_segments(labels, R)
        assert seg.dtype == torch.int64 and seg[0] == 0 and seg[-1] == 300
        assert torch.equal(labels[order], torch.sort(labels, stable=True).values)
        assert torch.equal(seg[1:] - seg[:-1], torch.bincount(labels, minlength=R))
        for r in range(R):  # stable: the rows of a region keep their order
            rows = order[seg[r]:seg[r + 1]]
            assert torch.equal(rows, torch.nonzero(labels == r).reshape(-1))
    for bad in (torch.tensor([0, 1, 3]), torch.tensor([-1, 0, 1])):
        _, seg = region_segments(bad, 3)
        assert seg[0] != 0 or seg[-1] != 3


def test_region_posterior_needs_m_multiple_of_128():
    from nonstationary_precip_b200.svgp import SVGPGibbs
    from svgp_cases import make_problem
    x, y, Z, kw, N = make_problem("diag", B=32, M=24, d=2)
    model = SVGPGibbs("diag", Z, N, **kw)
    with pytest.raises(ValueError):
        model.region_posterior(x, torch.zeros(32, dtype=torch.long), 1)
