"""Posterior of weighted regional sums behind the C ABI (csrc/gibbs_segsum.cu: npgp_gibbs_*_segsum, npgp_segment_colwsum;
csrc/svgp_step.cu: npgp_svgp_region_moments, through SVGPGibbs.region_posterior): the pair sums against dense kernel matrices
and against the forward tile kernels at 65536 rows, the plan call against the dense SVGP posterior covariance, one-row regions
against the marginals, the invariances, the gap to the sampler's covariance, the plan-state rules, CUDA-graph capture and a
C program."""
import math
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

from test_svgp_predict_gpu import B, CASES, N_ROWS, ROOT, build, oracle_field, rel

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


def region_matrix(seg, n, w):
    """A (R x n): A[r, i] = w_i for i in region r (CPU)."""
    seg = seg.cpu()
    R = seg.numel() - 1
    A = torch.zeros(R, n)
    for r in range(R):
        A[r, seg[r]:seg[r + 1]] = w[seg[r]:seg[r + 1]]
    return A


def layouts(n, g):
    """one region; ragged with an empty and a one-row region; 300 random regions (int64 offsets, CPU)"""
    out = [torch.tensor([0, n])]
    if n >= 3:
        out.append(torch.tensor([0, 1, 1, n // 3, n // 3 + 1, n]))
    cuts = torch.sort(torch.randint(0, n + 1, (299,), generator=g)).values
    out.append(torch.cat([torch.tensor([0]), cuts, torch.tensor([n])]))
    return out


def weight_sets(n, g):
    return [None, 0.5 + torch.rand(n, generator=g), torch.randn(n, generator=g)]


def diag_points(n, D, g):
    x = torch.rand(n, D, generator=g) * 2 - 1
    ell = torch.exp(math.log(0.3) + 0.3 * torch.randn(D, n, generator=g))
    return x, ell


def full_points(n, d, g):
    from oracle import gibbs_oracle as o
    x = torch.rand(n, d, generator=g) * 2 - 1
    Dm = torch.diag(torch.full((d,), 0.8))
    S = o.sigma_from_H(0.5 * torch.randn(n, d, generator=g), Dm) * 0.1
    iu = torch.triu_indices(d, d)
    return x, S, S[:, iu[0], iu[1]].contiguous()


def dense_kappa(kind, x, f):
    from oracle import gibbs_oracle as o
    K = o.gibbs_diag_K(x, x, f, f) if kind == "diag" else o.gibbs_full_K(x, x, f, f, 1e-5)
    K.fill_diagonal_(1.0)
    return K


def segsum(kind, x, fp, seg, w, full, part=0, nparts=1):
    from nonstationary_precip_b200 import ops
    c = lambda t: None if t is None else t.cuda()
    if kind == "diag":
        return ops.gibbs_diag_segsum(c(x), c(fp), c(seg), w=c(w), full=full, part=part, nparts=nparts)
    return ops.gibbs_full_segsum(c(x), c(fp), c(seg), w=c(w), full=full, part=part, nparts=nparts)


@pytest.mark.parametrize("kind,D", [("diag", D) for D in range(1, 7)] + [("full", 2), ("full", 3)])
def test_pair_sums_against_dense_kernel_matrices(kind, D):
    g = torch.Generator().manual_seed(100 * D + len(kind))
    for n in (1, 127, 128, 129, 1000):
        if kind == "diag":
            x, fp = diag_points(n, D, g)
            K = dense_kappa(kind, x, fp)
        else:
            x, S, fp = full_points(n, D, g)
            K = dense_kappa(kind, x, S)
        for seg in layouts(n, g):
            for w in weight_sets(n, g):
                wv = w if w is not None else torch.ones(n)
                A = region_matrix(seg, n, wv)
                # (+ 1e-300: kernel values below exp(-708) come out as that instead of 0 on the device)
                want, bound = A @ K @ A.T, 1e-13 * (A.abs() @ K.abs() @ A.abs().T) + 1e-300
                Gd, G = segsum(kind, x, fp, seg, w, True)
                Gd, G = Gd.cpu(), G.cpu()
                assert ((G - want).abs() <= bound).all(), (n, seg.numel() - 1, ((G - want).abs() / bound).max().item())
                assert torch.equal(Gd, torch.diagonal(G)) and torch.equal(G, G.T)
                Gd0, G0 = segsum(kind, x, fp, seg, w, False)
                assert G0 is None and torch.equal(Gd0.cpu(), Gd)
                assert torch.equal(segsum(kind, x, fp, seg, w, True)[1].cpu(), G)


@pytest.mark.parametrize("kind,d", [("diag", 2), ("full", 3)])
def test_pair_sums_at_65536_rows_against_forward_tiles(kind, d):
    """A 256 x 256 grid in 16 blocks of 64 x 64 cells, rows sorted by block; the reference reduces FP64 tiles of the existing
    forward kernel (x against x, one 4096-row block against another) in torch, with the same-row entries replaced by 1."""
    from nonstationary_precip_b200 import ops
    g = torch.Generator().manual_seed(5 + d)
    t = (torch.arange(256) + 0.5) / 128 - 1
    gy, gx = torch.meshgrid(t, t, indexing="ij")
    blk = (gy.reshape(-1).add(1).mul(2).floor().clamp_max(3) * 4 + gx.reshape(-1).add(1).mul(2).floor().clamp_max(3)).long()
    order = torch.sort(blk, stable=True).indices
    pts = torch.stack([gx.reshape(-1), gy.reshape(-1)], 1)[order]
    n, R = 65536, 16
    seg = torch.arange(R + 1) * 4096
    w = (0.5 + torch.rand(n, generator=g)).cuda()
    if kind == "diag":
        x = pts.contiguous().cuda()
        fp = torch.exp(math.log(0.05) + 0.3 * torch.sin(3 * x.T))
        fwd = lambda a, b: ops.gibbs_diag_fwd(x[a], fp[:, a], x[b], fp[:, b])
    else:
        x = torch.cat([pts, 0.3 * torch.sin(4 * pts[:, :1])], 1).contiguous().cuda()
        _, S, fp = full_points(n, 3, g)
        fp = fp.cuda() * 0.05
        fwd = lambda a, b: ops.gibbs_full_fwd(x[a], fp[a], x[b], fp[b], 1e-5)
    want = torch.empty(R, R, device="cuda")
    for r in range(R):
        a = slice(4096 * r, 4096 * (r + 1))
        for rp in range(R):
            b = slice(4096 * rp, 4096 * (rp + 1))
            K = fwd(a, b)
            if r == rp:
                K.fill_diagonal_(1.0)
            want[r, rp] = w[a] @ K @ w[b]
    Gd, G = segsum(kind, x, fp, seg, w, True)
    assert rel(G, want) <= 1e-12 and rel(Gd, torch.diagonal(want)) <= 1e-12
    Gd0, _ = segsum(kind, x, fp, seg, w, False)
    assert torch.equal(Gd0, Gd)


def test_segment_colwsum_against_torch():
    from nonstationary_precip_b200 import ops
    g = torch.Generator().manual_seed(3)
    n, M, row0 = 1500, 200, 700
    K = torch.randn(n, M, generator=g)
    w = torch.randn(n, generator=g)
    for seg in ([0, 3000], [0, 700, 701, 701, 1000, 1010, 1900, 2200, 3000], list(range(0, 3001, 1))):
        seg = torch.tensor(seg)
        R = seg.numel() - 1
        want = torch.zeros(R, M)
        for r in range(R):
            lo, hi = max(int(seg[r]), row0) - row0, min(int(seg[r + 1]), row0 + n) - row0
            if hi > lo:
                want[r] = w[lo:hi] @ K[lo:hi]
        out = torch.full((R, M + 3), 2.0, device="cuda")[:, :M]
        got = ops.segment_colwsum(K.cuda(), seg.cuda(), w.cuda(), row0=row0, out=out) - 2.0
        bound = 1e-14 * (torch.zeros(R, M).index_add_(0, torch.bucketize(torch.arange(row0, row0 + n), seg[1:], right=True),
                                                      (w[:, None] * K).abs()) + 1)
        assert ((got.cpu() - want).abs() <= bound).all()
        assert torch.equal(ops.segment_colwsum(K.cuda(), seg.cuda(), w.cuda(), row0=row0) + 0.0,
                           ops.segment_colwsum(K.cuda(), seg.cuda(), w.cuda(), row0=row0))


def dense_posterior(model, x, field, noise=False, P=None):
    """CPU: the n x n posterior covariance s kappa + jitter_xx I + A^T (S - I) A and the mean A^T m in the oracle's whitened
    form, A = P K_zx, and the absolute-value versions of its terms (|K_xz| |P^T| ... |P| |K_zx|).  P: the inverse Cholesky factor
    of Kzz + jitter_zz I, by default the oracle's own (torch on the CPU); the field is the one the C path computed
    (predictive(field=True))."""
    from oracle import gibbs_oracle as o
    c = lambda t: t.detach().cpu()
    s = torch.nn.functional.softplus(c(model.p["raw_outputscale"]))
    Z, m, Ls = c(model.p["Z"]), c(model.p["m"]), torch.tril(c(model.p["Ls"]))
    x, f = c(x), c(field)
    if model.variant == "diag":
        ez = torch.exp(c(model.p["log_ell_z"]))
        Kzz, Kxz, kap = s * o.gibbs_diag_K(Z, Z, ez, ez), s * o.gibbs_diag_K(x, Z, f, ez), o.gibbs_diag_K(x, x, f, f)
    else:
        from nonstationary_precip_b200.ops import sym_unpack
        Sz = o.sigma_from_H(c(model.p["H"]), c(model.p["D"]))
        Sx = sym_unpack(f, model.d)
        Kzz, Kxz = s * o.gibbs_full_K(Z, Z, Sz, Sz, 1e-5), s * o.gibbs_full_K(x, Z, Sx, Sz, 1e-5)
        kap = o.gibbs_full_K(x, x, Sx, Sx, 1e-5)
    kap.fill_diagonal_(1.0)
    if P is None:
        L = torch.linalg.cholesky(Kzz + model.jitter_zz * torch.eye(model.M))
        P = torch.linalg.solve_triangular(L, torch.eye(model.M), upper=False)
    P = c(P)
    A = P @ Kxz.T
    E = Ls @ Ls.T - torch.eye(model.M)
    n = x.shape[0]
    jit = model.jitter_xx + (1e-4 + torch.nn.functional.softplus(c(model.p["raw_noise"])) if noise else 0.0)
    PK = P.abs() @ Kxz.abs().T
    lowrank_abs = PK.T @ E.abs() @ PK
    return dict(mean=A.T @ m, abs_mean=PK.T @ m.abs(), cov=s * kap + jit * torch.eye(n) + A.T @ E @ A,
                abs_cov=s * kap + jit * torch.eye(n) + lowrank_abs, lowrank_abs=lowrank_abs, A=A, s=s, kap=kap, E=E)


def plan_P(model):
    return model._plan_view(model._plan(B, 1, B), 2, model.M * model.M).view(model.M, model.M)


def check_against_dense(model, x, labels, R, w, r, noise=False):
    """Against the dense posterior with the plan's inverse factor P (it never forms u = P^T m or C = P^T E P), to 1e-11 of each
    term's absolute value; and against the oracle's own Cholesky to 1e-8 of it: two factorisations of Kzz round apart by
    eps * cond(Kzz), as the existing predict tests find between the C path and the oracle."""
    field = model.predictive(x, field=True, chunk=B).field
    Aw = torch.zeros(R, x.shape[0])
    Aw[labels.cpu(), torch.arange(x.shape[0])] = w.cpu()
    refs = []
    for tol, P in ((1e-11, plan_P(model)), (1e-8, None)):
        ref = dense_posterior(model, x, field, noise, P)
        mb = tol * Aw.abs() @ ref["abs_mean"]
        cb = tol * Aw.abs() @ ref["abs_cov"] @ Aw.abs().T
        mean, cov = Aw @ ref["mean"], Aw @ ref["cov"] @ Aw.T
        assert ((r.mean.cpu() - mean).abs() <= mb).all(), (tol, ((r.mean.cpu() - mean).abs() / mb).max().item())
        assert ((r.cov.cpu() - cov).abs() <= cb).all(), (tol, ((r.cov.cpu() - cov).abs() / cb).max().item())
        refs.append(ref)
    assert torch.equal(r.var, torch.diagonal(r.cov)) and torch.equal(r.cov, r.cov.T)
    return refs[0], Aw


@pytest.mark.parametrize("variant,d,M", CASES)
def test_plan_call_against_the_dense_posterior(variant, d, M):
    model, x, y, Z, p = build(variant, d, M, seed=M + d + 1)
    g = torch.Generator().manual_seed(M)
    R = 37
    labels = torch.randint(0, R, (N_ROWS,), generator=g).cuda()
    w = (torch.randn(N_ROWS, generator=g) + 0.3).cuda()
    r = model.region_posterior(x, labels, R, w, chunk=B)
    assert model.check_status() == 0
    check_against_dense(model, x, labels, R, w, r)
    rn = model.region_posterior(x, labels, R, w, noise=True, chunk=B)
    check_against_dense(model, x, labels, R, w, rn, noise=True)
    rv = model.region_posterior(x, labels, R, w, cov=False, chunk=B)
    assert rv.cov is None and torch.equal(rv.mean, r.mean) and rel(rv.var, r.var) <= 1e-13


def test_plan_call_where_the_low_rank_term_cancels_most_of_s_g():
    """Inducing points dense relative to the lengthscale: the posterior variance of a region is a small difference."""
    model, x, y, Z, p = build("diag", 2, 256, seed=4)
    with torch.no_grad():
        model.p["log_ell_z"].fill_(math.log(0.9))
        model.prior_c.fill_(math.log(0.9))
        model.p["Ls"].copy_(torch.eye(256, device="cuda") * 0.05)
    labels = (x[:, 0] > 0).long() + 2 * (x[:, 1] > 0).long()
    w = torch.ones(N_ROWS, device="cuda")
    r = model.region_posterior(x, labels, 4, w, chunk=B)
    ref, Aw = check_against_dense(model, x, labels, 4, w, r)
    sG = (Aw @ (ref["s"] * ref["kap"]) @ Aw.T).diagonal()
    assert (r.var.cpu() < 0.05 * sG).all()  # most of s G cancels


def test_one_row_regions_reproduce_the_marginals():
    model, x, y, Z, p = build("full", 3, 128, seed=9)
    pred = model.predictive(x, field=True, chunk=B)
    lab = torch.arange(N_ROWS, device="cuda")
    r = model.region_posterior(x, lab, N_ROWS, cov=False, chunk=B)
    assert (pred.var > 1e-6).all()  # no clamp active
    # predictive forms K(x, Z) as fixed-point digit planes (entries to 2^-54 s), this call in FP64: the two differ by that
    # quantisation times sum_j |u_j| (mean) and sum_jl |C_jl| |k_l| (variance) at most
    M = model.M
    u = model._plan_view(model._plan(B, 1, B), 4, M)
    Cm = model._plan_view(model._plan(B, 1, B), 3, M * M).view(M, M)
    s = torch.nn.functional.softplus(model.p["raw_outputscale"])
    K = model._kernel_fwd(x, pred.field, model.p["Z"], model._field_z(), s)
    q = 2.0 ** -53 * s
    mb = 1e-13 * pred.mean.abs().max() + q * u.abs().sum()
    vb = 1e-12 * pred.var.abs() + 2 * q * (K.abs() @ Cm.abs()).sum(1)
    assert ((r.mean - pred.mean).abs() <= mb).all(), ((r.mean - pred.mean).abs() / mb).max().item()
    assert ((r.var - pred.var).abs() <= vb).all(), ((r.var - pred.var).abs() / vb).max().item()
    rn = model.region_posterior(x, lab, N_ROWS, noise=True, cov=False, chunk=B)
    noise = 1e-4 + torch.nn.functional.softplus(model.p["raw_noise"])
    assert rel(rn.var - r.var, noise.expand(N_ROWS)) <= 1e-13 and torch.equal(rn.mean, r.mean)


@pytest.mark.parametrize("variant,d,M", CASES[1:3])
def test_invariances(variant, d, M):
    model, x, y, Z, p = build(variant, d, M, seed=21)
    g = torch.Generator().manual_seed(2)
    R = 23
    labels = torch.randint(0, R, (N_ROWS,), generator=g).cuda()
    w = (0.5 + torch.rand(N_ROWS, generator=g)).cuda()
    a = model.region_posterior(x, labels, R, w, chunk=B)
    b = model.region_posterior(x, labels, R, w, chunk=B)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    two = model.region_posterior(x, labels, R, 2 * w, chunk=B)
    assert torch.equal(two.mean, 2 * a.mean) and torch.equal(two.cov, 4 * a.cov) and torch.equal(two.var, 4 * a.var)
    # other summation orders: bounded by the absolute-value version of each term (Y^T C Y cancels)
    field = model.predictive(x, field=True, chunk=B).field
    ref = dense_posterior(model, x, field, P=plan_P(model))
    Aw = torch.zeros(R, N_ROWS)
    Aw[labels.cpu(), torch.arange(N_ROWS)] = w.cpu()
    mabs, cabs = (Aw @ ref["abs_mean"]).cuda(), (Aw @ ref["abs_cov"] @ Aw.T).cuda()
    close = lambda q, tol: ((q.mean - a.mean).abs() <= tol * mabs).all() and ((q.cov - a.cov).abs() <= tol * cabs).all()
    perm = torch.randperm(N_ROWS, generator=g).cuda()
    assert close(model.region_posterior(x[perm], labels[perm], R, w[perm], chunk=B), 1e-12)
    assert close(model.region_posterior(x, labels, R, w, chunk=512), 1e-13)
    for nparts in (2, 3, 5):
        parts = [model.region_posterior(x, labels, R, w, part=k, nparts=nparts, chunk=B) for k in range(nparts)]
        tot = type(a)(*(sum(q[i] for q in parts) for i in range(3)))
        assert close(tot, 1e-13) and torch.equal(tot.var, torch.diagonal(tot.cov))


def test_gap_to_the_sampler_is_the_off_diagonal_residual():
    """The sampler's draws have covariance k^T P^T S P k' + delta r (the Nystrom residual's diagonal only).  For a dense cluster
    of positively weighted rows the exact regional variance exceeds the one implied by that covariance by exactly the double sum
    of the dropped off-diagonal residuals; and regional sums of many draws average to mean_R."""
    model, x, y, Z, p = build("diag", 2, 128, seed=8)
    xc = (x[:400] * 0.1 + 0.2).contiguous()  # a cluster well inside one lengthscale
    labels = torch.zeros(400, dtype=torch.long, device="cuda")
    labels[200:] = 1
    w = (0.5 + torch.rand(400, generator=torch.Generator().manual_seed(1))).cuda()
    r = model.region_posterior(xc, labels, 2, w, chunk=B)
    field = model.predictive(xc, field=True, chunk=B).field
    ref = dense_posterior(model, xc, field, P=plan_P(model))
    A, E, s, kap = ref["A"], ref["E"], ref["s"], ref["kap"]
    Q = A.T @ A  # k^T P^T P k'
    resid = (s * kap - Q)
    samp = A.T @ (E + torch.eye(model.M)) @ A + torch.diag(torch.diagonal(resid) + model.jitter_xx)
    Aw = torch.zeros(2, 400)
    Aw[labels.cpu(), torch.arange(400)] = w.cpu()
    off = resid - torch.diag(torch.diagonal(resid))
    gap = r.cov.cpu() - Aw @ samp @ Aw.T
    want = Aw @ off @ Aw.T
    bound = 1e-10 * (Aw @ (s * kap + ref["lowrank_abs"]) @ Aw.T)
    assert ((gap - want).abs() <= bound).all(), ((gap - want).abs() / bound).max().item()
    assert (torch.diagonal(want) > 0).all()  # the sampler understates the variance of the sums
    draws = torch.cat([model.sample(xc, 1024, seed=3 + k, chunk=B) for k in range(4)])
    sums = draws @ Aw.T.cuda()
    se = sums.std(0) / math.sqrt(4096)
    assert ((sums.mean(0) - r.mean).abs() <= 4 * se).all()


def c_region(model, ent, x, w, seg, R, out, work, nbytes, cov=True, part=0, nparts=1):
    from nonstationary_precip_b200._lib import lib, ptr, stream
    mean, var, cv = out
    return lib().npgp_svgp_region_moments(ent["handle"], x.shape[0], ptr(x), ptr(w), R, ptr(seg), ptr(model.theta), 0, part,
                                          nparts, ptr(mean), ptr(var), ptr(cv) if cov else None, R, work, nbytes, stream())


def region_work(model, ent, n, R):
    import ctypes
    from nonstationary_precip_b200._lib import lib
    nb = lib().npgp_svgp_region_workspace_bytes(ctypes.byref(ent["cfg"]), n, R, 1)
    t = torch.empty(nb // 8 + 64, device="cuda")
    return t, t.data_ptr() + (-t.data_ptr()) % 256, nb


def test_plan_state_rules_and_capture():
    from nonstationary_precip_b200._lib import lib, ptr, stream
    from nonstationary_precip_b200.svgp import region_segments
    model, x, y, Z, p = build("full", 3, 128, seed=12)
    model.use_c_engine()
    ent = model._plan(B, 1, B)
    h, th, st = ent["handle"], ptr(model.theta), stream()
    R = 11
    labels = torch.randint(0, R, (N_ROWS,), generator=torch.Generator().manual_seed(4)).cuda()
    order, seg = region_segments(labels, R)
    xs, w = x[order].contiguous(), torch.rand(N_ROWS, device="cuda")
    t, wp, nb = region_work(model, ent, N_ROWS, R)
    out = (torch.empty(R, device="cuda"), torch.empty(R, device="cuda"), torch.empty(R, R, device="cuda"))
    assert c_region(model, ent, xs, w, seg, R, out, wp, nb) == -1  # no prepare yet
    xb, yb = x[:B].contiguous(), y[:B].contiguous()
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0
    assert lib().npgp_svgp_elbo_fwd(h, ptr(xb), ptr(yb), th, ptr(model.grad), None, st) == 0
    assert c_region(model, ent, xs, w, seg, R, out, wp, nb) == -1  # a forward invalidates the prepared factors
    assert c_region(model, ent, xs, w, seg, R, out, wp, nb - 256) == -1
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0
    assert c_region(model, ent, xs, w, seg, R, out, wp, nb - 256) == -3
    assert c_region(model, ent, xs, w, seg, R, out, wp + 8, nb) == -2
    assert c_region(model, ent, xs, w, seg, R, out, wp, nb, part=2, nparts=2) == -1
    # prediction and draws are bitwise the same before and after a region call
    pa, sa = model.predictive(x, field=True, chunk=B), model.sample(x, 16, seed=2, chunk=B)
    first = model.region_posterior(xs, labels[order], R, w, chunk=B)
    pb, sb = model.predictive(x, field=True, chunk=B), model.sample(x, 16, seed=2, chunk=B)
    assert all(torch.equal(u, v) for u, v in zip(pa, pb) if u is not None) and torch.equal(sa, sb)
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0
    assert c_region(model, ent, xs, w, seg, R, out, wp, nb) == 0
    assert torch.equal(out[0], first.mean) and torch.equal(out[2], first.cov)
    assert lib().npgp_svgp_elbo_bwd(h, ptr(xb), th, ptr(model.grad), st) == -1  # the saved forward is gone
    # capture of prepare + region call; replay on other rows first
    xin, win = torch.zeros_like(xs), torch.zeros_like(w)
    got = tuple(torch.empty_like(t) for t in out)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        assert lib().npgp_svgp_predict_prepare(h, th, ptr(model.status), stream()) == 0
        assert c_region(model, ent, xin, win, seg, R, got, wp, nb) == 0
    for a, b in ((xs.flip(0) * 0.9, w.flip(0)), (xs, w)):
        xin.copy_(a)
        win.copy_(b)
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(got[0], first.mean) and torch.equal(got[1], first.var) and torch.equal(got[2], first.cov)
    # a seg that does not run from 0 to n, or decreases: NaN outputs, return code 0
    assert lib().npgp_svgp_predict_prepare(h, th, None, st) == 0
    for bad in (seg + 1, torch.cat([seg[:1], seg[2:3], seg[1:2], seg[3:]])):
        assert c_region(model, ent, xs, w, bad.contiguous(), R, out, wp, nb) == 0
        assert all(t.isnan().all() for t in out)
    r = model.region_posterior(x, labels + 1, R, chunk=B)  # label R is out of range
    assert all(t.isnan().all() for t in r)


def build_demo(tmp_path):
    exe = str(tmp_path / "svgp_region_demo")
    libdir = os.path.join(ROOT, "nonstationary_precip_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cmd = ["gcc", "-O2", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
           os.path.join(ROOT, "tools", "c_demo", "svgp_region_demo.c"), "-o", exe, "-L", libdir, "-lnpgp",
           "-L", os.path.join(cuda, "lib64"), "-lcudart", "-lm", "-Wl,-rpath," + libdir]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


@pytest.mark.parametrize("variant", ["full", "diag"])
def test_c_program_trains_then_sums_regions_like_python(variant, tmp_path):
    from nonstationary_precip_b200.svgp import region_segments
    exe = build_demo(tmp_path)
    M, d, iters, n, R = 128, 3, 3, N_ROWS, 9
    model, xt, yt, Z, p = build(variant, d, M, seed=31, n=n)
    x, y = xt[:B].contiguous(), yt[:B].contiguous()
    model.use_c_engine()
    labels = torch.randint(0, R, (n,), generator=torch.Generator().manual_seed(6)).cuda()
    order, seg = region_segments(labels, R)
    xs, w = xt[order].contiguous(), (0.5 + torch.rand(n, generator=torch.Generator().manual_seed(7))).cuda()
    consts = ([model.row_os.reshape(-1), model.row_lam.reshape(-1)] if variant == "full" else
              [model.prior_c.reshape(-1), model.prior_os.reshape(-1), model.prior_lam.reshape(-1)])
    blob = torch.cat([t.detach().reshape(-1).cpu() for t in [x, y, model.theta, model.mask] + consts]).numpy()
    prob, out = str(tmp_path / "problem.bin"), str(tmp_path / "out.bin")
    with open(prob, "wb") as f:
        f.write(struct.pack("8i", 1 if variant == "full" else 0, d, M, B, model.N, 1, 1, iters))
        f.write(blob.astype(np.float64).tobytes())
        f.write(struct.pack("2i", n, R))
        f.write(torch.cat([xs.reshape(-1), w]).cpu().numpy().astype(np.float64).tobytes())
        f.write(seg.cpu().numpy().astype(np.int64).tobytes())
    r = subprocess.run([exe, prob, out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.stdout, r.stderr)
    got = np.fromfile(out, dtype=np.float64)
    n_pad = model.theta.numel()
    assert got.size == 2 * R + R * R + n_pad
    mean, var, cov, theta = np.split(got, np.cumsum([R, R, R * R]))
    model.theta.copy_(torch.from_numpy(theta))
    want = model.region_posterior(xs, labels[order], R, w, chunk=B)
    assert np.array_equal(mean, want.mean.cpu().numpy()) and np.array_equal(var, want.var.cpu().numpy())
    assert np.array_equal(cov, want.cov.cpu().numpy().reshape(-1))
