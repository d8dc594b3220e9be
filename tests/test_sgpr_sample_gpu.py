"""Posterior sample fields of the streamed SGPR models (sgpr.py: posterior().sample()): the draws against
mean + K (V^T E) + sqrt(r) xi formed in FP64 from regenerated normals, the exactness of their covariance against the dense
joint predictives of the reference's models, the moments of many draws, the invariances the Philox keys promise, the
finishing kernel npgp_sgpr_sample_finish and the generator npgp_sample_normals against their formulas, and the snapshot and
no-host-sync properties of the sampler."""
import math

import pytest
import torch

from oracle import gibbs_oracle as o
from test_sgpr_predict_gpu import diag_problem, rel, st_problem

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


def normals(n, seed, offset):
    """n standard normals normal_from_index(seed, offset + i), regenerated through npgp_dsvi_sample (mu 0, var 1)."""
    from nonstationary_precip_b200 import ops
    return ops.dsvi_sample(torch.zeros(n, device="cuda"), torch.ones(n, device="cuda"), seed=seed, offset=offset)


def problem(kind, M, seed, n=900, use_i8=True):
    model, x, y = diag_problem(n, M, 2, seed) if kind == "diag" else st_problem(n, M, seed)
    model.use_i8 = use_i8
    return model, x, y


def rows_for(kind, n, seed, spread=1.0):
    g = torch.Generator().manual_seed(seed)
    if kind == "diag":
        return ((torch.rand(n, 2, generator=g) * 2 - 1) * spread).cuda()
    return torch.cat([torch.rand(n, 1, generator=g) * 6 - 3, (torch.rand(n, 2, generator=g) * 2 - 1) * spread], 1).cuda()


def features(post, xs):
    """The FP64 feature rows k(x) (n, W) of the snapshot: Gibbs K (diag) or [K_t | K_s] (st)."""
    from nonstationary_precip_b200 import ops
    ell = post.predictive(xs, field=True).field
    if post.kind == "st":
        return torch.cat([ops.rbfper_fwd(xs[:, 0].contiguous(), post.zt, post.hyp),
                          ops.gibbs_diag_fwd(xs[:, 1:3].contiguous(), ell, post.zs, post.ell_z)], 1)
    return ops.gibbs_diag_fwd(xs, ell, post.Z, post.ell_z)


@torch.no_grad()
def p_factor(model):
    """P = L^-1 of the model's current Kzz (blockdiag(P_t, P_s) for the spatio-temporal model), as posterior() forms it."""
    if model.Z.shape[1] == 3:
        _, _, _, _, (_, _, Ps), (_, _, Pt), _ = model._z_side()
        return torch.block_diag(Pt, Ps).contiguous()
    return model._z_side()[2][2].contiguous()


def residual(post, K, P):
    """r(x) = [st] max(os_t - |P_t k_t|^2, 0) + s max(1 - |P_s k_s|^2, 0), and the bound |k_c|^2 |P_c|_F^2 on the size of
    the terms of each norm that the rounding of the row-norm kernels is relative to (as in test_sgpr_predict_gpu.py)."""
    q = (K @ P.T) ** 2
    size = lambda cols: (K[:, cols] ** 2).sum(1) * (P[cols, cols] ** 2).sum()  # noqa: E731
    if post.kind == "st":
        M = post.M
        t, sp = slice(0, M), slice(M, 2 * M)
        r = (post.hyp[3] - q[:, t].sum(1)).clamp_min(0) + post.s * (1 - q[:, sp].sum(1)).clamp_min(0)
        return r, size(t) + post.s * size(sp)
    return post.s * (1 - q.sum(1)).clamp_min(0), post.s * size(slice(None))


def sgpr_gibbs_predict_cov(x, y, Z, log_ell_z, x_new, outputscale, noise, prior_c, prior_os, prior_lam):
    """Dense joint predictive of DiagonalSparseGP.predict in eval mode, from the oracle's parts as oracle.sgpr_gibbs_predict
    forms its marginals: Lr Lr^T + diag(corr) - Lr (I - B^-1) Lr^T, corr = clamp(s - q_ii, 0) (gibbs_kernels.py:228-232)."""
    M = Z.shape[0]
    ell_z = torch.exp(log_ell_z)
    Lz = o.psd_cholesky(o.gibbs_diag_K(Z, Z, ell_z, ell_z))
    xa = torch.cat([x, x_new], 0)
    Ka = o.gibbs_diag_K(xa, Z, o.field_interp_diag(xa, Z, ell_z, prior_c, prior_os, prior_lam), ell_z)
    R = math.sqrt(float(outputscale)) * torch.linalg.solve_triangular(Lz, Ka.T, upper=False).T
    n = x.shape[0]
    Lr, At = R[n:], R[:n] / math.sqrt(float(noise))
    Bm = torch.eye(M) + At.T @ At
    mean = Lr @ torch.linalg.solve(Bm, At.T @ y) / math.sqrt(float(noise))
    corr = (outputscale - (Lr * Lr).sum(-1)).clamp_min(0.0)
    return mean, Lr @ Lr.T + torch.diag(corr) - Lr @ (torch.eye(M) - torch.linalg.inv(Bm)) @ Lr.T


def oracle_cov(kind, model, x, y, xs):
    c = lambda t: t.detach().cpu()  # noqa: E731
    sp = torch.nn.functional.softplus
    s, noise = sp(c(model.raw_outputscale)).reshape(()), (1e-4 + sp(c(model.raw_noise))).reshape(())
    if kind == "diag":
        args = (x, y, c(model.Z), c(model.log_ell_z), xs.cpu(), s, noise, c(model.prior_c), c(model.prior_os),
                c(model.prior_lam))
        mean, cov = sgpr_gibbs_predict_cov(*args)
        assert rel(torch.diagonal(cov), o.sgpr_gibbs_predict(*args)[1]) < 1e-12
        return mean, cov
    return o.st_predict(x, y, c(model.Z), c(model.log_ell_z), xs.cpu(), c(model.hyp_t()), s, noise, c(model.prior_c),
                        c(model.prior_os), c(model.prior_lam), literal=False)


# digit path: diag M = 128 / 256, st M = 64 / 128 (W = 128 / 256); FP64 path: widths not a multiple of 128 (diag M = 96,
# st M = 50: W = 100) and use_i8 = False.  The temporal Kzz of the spatio-temporal model is ill conditioned; M = 50 keeps it
# as well conditioned as test_sgpr_predict_gpu.py needs it for the 1e-8 comparisons with the oracle
CASES = [("diag", 128, True), ("diag", 256, True), ("diag", 96, True), ("diag", 128, False),
         ("st", 64, True), ("st", 128, True), ("st", 50, True), ("st", 64, False)]


# ---------------------------------------------------------------------------------------------------------------------
# construction and exactness
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,M,use_i8", CASES)
def test_draws_equal_the_fp64_construction(kind, M, use_i8):
    model, x, y = problem(kind, M, seed=M + 1, use_i8=use_i8)
    post = model.posterior(x.cuda(), y.cuda(), chunk=256)
    assert post.digits == (use_i8 and post.width % 128 == 0)
    xs = rows_for(kind, 700, seed=M, spread=1.1)
    S, seed, chunk = 40, 4321, 256
    n, W = xs.shape[0], post.width
    K, P, V = features(post, xs), p_factor(model), post.V
    E = torch.stack([normals(W, seed, s << 32) for s in range(S)], 1)  # (W, S)
    xi = torch.stack([normals(n, seed, (1 << 63) + (s << 48)) for s in range(S)])
    r, qsize = residual(post, K, P)
    KW = (K @ (V.T @ E)).T
    scale = (K.abs() @ (V.abs().T @ E.abs())).T
    mean = post.predictive(xs, chunk=chunk).mean  # the mean term of the draws is the predictive mean, bitwise
    noise = post.noise
    for with_noise in (False, True):
        got = post.sample(xs, S, seed=seed, noise=with_noise, chunk=chunk)
        assert got.shape == (S, n) and torch.isfinite(got).all()
        var = r + noise if with_noise else r
        sd = torch.sqrt(var)
        want = mean + KW + sd * xi
        # K V^T E: the rounding of the digit (or FP64) product relative to sum_j |K_ij| (|V|^T |E|)_js.  r cancels: it is exact
        # to 1e-14 of the size of the terms of |P k|^2, which sqrt divides by 2 sqrt(r) (or takes the root of, near 0)
        dr = 1e-14 * qsize
        dsd = torch.minimum(dr / (2 * sd).clamp_min(1e-300), torch.sqrt(dr)) + 1e-14 * sd
        bound = 1e-12 * scale + dsd * xi.abs() + 1e-15 * mean.abs()
        err = (got - want).abs()
        assert (err <= bound).all(), (err / bound).max().item()


@pytest.mark.parametrize("kind,M,use_i8", [CASES[0], CASES[2], CASES[4], CASES[6]])
def test_covariance_is_the_joint_predictive_of_the_reference(kind, M, use_i8):
    model, x, y = problem(kind, M, seed=M, n=700, use_i8=use_i8)
    post = model.posterior(x.cuda(), y.cuda(), chunk=256)
    xs = rows_for(kind, 500, seed=M + 3)
    K, P = features(post, xs), p_factor(model)
    r, qsize = residual(post, K, P)
    Rk = K @ post.V.T  # (n, W): rows (V k)^T
    cov = Rk @ Rk.T + torch.diag(r)
    mean_o, cov_o = oracle_cov(kind, model, x, y, xs)
    e = rel(cov, cov_o)
    print("%s M=%d: joint covariance %.2e" % (kind, M, e))
    assert e < 1e-8
    pred = post.predictive(xs)
    # r + |V k|^2 is var_f, to the rounding of the row norms: predictive() forms them from digit planes (or FP64 GEMMs), here
    # they are FP64 products of the re-derived P and of V.  Both are exact to a small multiple of eps times the bound
    # |k|^2 |P|_F^2 (|k|^2 |V|_F^2) on the size of their terms; the temporal P of the spatio-temporal model makes that bound
    # large against var_f, so the error is measured against it rather than against var_f
    vsize = (K ** 2).sum(1) * (post.V ** 2).sum()
    err = (r + (Rk * Rk).sum(1) - pred.var).abs()
    bound = 1e-13 * (qsize + vsize) + 1e-15 * pred.var
    print("%s M=%d: r + |V k|^2 - var_f %.2e of var_f, %.2e of the bound (bound %.2e of var_f)" % (
        kind, M, rel(r + (Rk * Rk).sum(1), pred.var), (err / bound).max().item(), (bound / pred.var).max().item()))
    assert (err <= bound).all(), (err / bound).max().item()
    # that bound is loose for the spatio-temporal model (up to several var_f); relative to var_f the identity holds to 4e-11
    # there (st M = 64, from the conditioning of P_t) and to 1e-12 or better elsewhere
    assert rel(r + (Rk * Rk).sum(1), pred.var) < 1e-9
    assert rel(pred.mean, mean_o) < 1e-8


# ---------------------------------------------------------------------------------------------------------------------
# moments of many draws
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,M", [("diag", 128), ("st", 64)])
def test_moments_of_many_draws(kind, M):
    model, x, y = problem(kind, M, seed=41)
    post = model.posterior(x.cuda(), y.cuda(), chunk=256)
    x0 = model.Z[5].detach()  # at an inducing point the residual r is small: the correlated part V k dominates
    offs = torch.tensor([0.0, 0.01, 0.03, 0.1, 0.3], device="cuda")
    step = torch.zeros(x0.shape[0], device="cuda")
    step[-2:] = 1.0  # move in space (the Gibbs columns), at a fixed time for the spatio-temporal model
    xs = torch.cat([x0 + offs[:, None] * step, rows_for(kind, 45, seed=43)]).contiguous()
    n = xs.shape[0]
    draws = torch.cat([post.sample(xs, 1024, seed=100 + k) for k in range(8)])  # (8192, n)
    N = draws.shape[0]
    mean, cov = (t.cuda() for t in oracle_cov(kind, model, x, y, xs))
    var = torch.diagonal(cov)
    avg = draws.mean(0)
    assert ((avg - mean).abs() <= 6 * torch.sqrt(var / N)).all()
    dev = draws - avg
    emp = dev.T @ dev / (N - 1)
    band = 6 * torch.sqrt((var[:, None] * var[None, :] + cov ** 2) / (N - 1))  # sd of a sample covariance
    assert ((emp - cov).abs() <= band).all(), ((emp - cov).abs() / band).max().item()
    corr = cov[0, 1] / torch.sqrt(cov[0, 0] * cov[1, 1])
    assert corr > 0.5  # nearby rows are strongly correlated: the fields are coherent, not independent marginals
    # a weighted "basin total" a^T f over all n rows: its sample variance against a^T Cov a
    a = torch.rand(n, generator=torch.Generator().manual_seed(5)).cuda()
    tot = draws @ a
    want = a @ cov @ a
    assert abs(tot.var().item() - want.item()) <= 6 * want.item() * math.sqrt(2.0 / (N - 1))


# ---------------------------------------------------------------------------------------------------------------------
# invariances
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,M,use_i8", [CASES[1], CASES[2], CASES[5], CASES[7]])
def test_seeds_sample_counts_row_offsets_and_chunks(kind, M, use_i8):
    # W <= 256 here: npgp_dgemm forms W^T = E^T V without splitting its inner dimension, so the draws are bitwise functions
    # of (seed, s, row) wherever the mean is
    model, x, y = problem(kind, M, seed=17, n=700, use_i8=use_i8)
    post = model.posterior(x.cuda(), y.cuda(), chunk=256)
    xs = rows_for(kind, 700, seed=19)
    chunk = 256
    a = post.sample(xs, 64, seed=5, chunk=chunk)
    assert torch.equal(a, post.sample(xs, 64, seed=5, chunk=chunk))
    assert not (post.sample(xs, 64, seed=6, chunk=chunk) == a).any()
    assert torch.equal(post.sample(xs, 16, seed=5, chunk=chunk), a[:16])
    assert torch.equal(post.sample(xs, 100, seed=5, chunk=chunk)[:64], a)  # 128 padded rows of W^T instead of 64
    # two calls with row offsets: the rows of one call.  The diagonal model's digit path adds its mean from K u partials whose
    # column split depends on the chunk's row count; nothing else does.  So bitwise wherever the two chunkings give the same mean
    h = 300  # not a chunk boundary
    two = torch.cat([post.sample(xs[:h], 64, seed=5, chunk=chunk),
                     post.sample(xs[h:], 64, seed=5, row_offset=h, chunk=chunk)], 1)
    mean_a = post.predictive(xs, chunk=chunk).mean
    mean_h = torch.cat([post.predictive(xs[:h], chunk=chunk).mean, post.predictive(xs[h:], chunk=chunk).mean])
    same = mean_a == mean_h
    assert same.float().mean() > 0.5
    assert torch.equal(two[:, same], a[:, same]) and rel(two, a) <= 1e-13
    assert rel(post.sample(xs, 64, seed=5, chunk=4096), a) <= 1e-12


@pytest.mark.parametrize("kind", ["diag", "st"])
def test_posterior_from_two_emulated_ranks_gives_the_same_draws(kind):
    model, x, y = diag_problem(800, 128, 2, seed=4) if kind == "diag" else st_problem(800, 64, seed=4)
    x, y = x.cuda(), y.cuda()
    xs = x[:300] * 0.97
    full = model.posterior(x, y, chunk=256).sample(xs, 64, seed=5)
    got = []
    model.posterior(x[400:], y[400:], chunk=256, n_total=800, all_reduce=lambda t: got.append(t.clone()))
    post = model.posterior(x[:400], y[:400], chunk=256, n_total=800, all_reduce=lambda t: t.add_(got[0]))
    e = rel(post.sample(xs, 64, seed=5), full)
    print("%s: two ranks %.2e" % (kind, e))
    assert e <= 1e-10


def test_empty_rows():
    model, x, y = problem("diag", 128, seed=3, n=400)
    post = model.posterior(x.cuda(), y.cuda())
    out = post.sample(torch.zeros(0, 2, device="cuda"), 7)
    assert out.shape == (7, 0)


# ---------------------------------------------------------------------------------------------------------------------
# the finishing kernel and the generator
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb_t,add_noise", [(0, False), (3, True), (3, False)])
def test_finish_matches_formula(nb_t, add_noise):
    from nonstationary_precip_b200 import ops
    n, nb_s, S, Sp, ldo, seed, row0 = 1000, 4, 40, 64, 1037, 77, 123456
    g = torch.Generator().manual_seed(nb_t + 10 * add_noise)
    s, noise, os_t = torch.tensor(0.7).cuda(), torch.tensor(0.03).cuda(), torch.tensor(7.5).cuda()
    qn = torch.rand(nb_t + nb_s, n, generator=g) * 0.3
    qn[nb_t:, :100] *= 5.0  # these rows' Gibbs clamp is active
    if nb_t:
        qn[:nb_t, 100:200] = torch.rand(nb_t, 100, generator=g) * 4.0
    qn = qn.cuda()
    mean = torch.randn(n, generator=g).cuda()
    F = torch.randn(n, Sp, generator=g).cuda()
    F[:, S:] = float("nan")  # padding columns: never read
    out = torch.full((S, ldo), float("nan"), device="cuda")
    ops.sgpr_sample_finish(mean, qn, nb_t, F, S, s, noise, out[:, :n], os_t=os_t if nb_t else None, add_noise=add_noise,
                           seed=seed, row0=row0)
    r = s * (1 - qn[nb_t:].sum(0)).clamp_min(0)
    if nb_t:
        r = r + (os_t - qn[:nb_t].sum(0)).clamp_min(0)
    if add_noise:
        r = r + noise
    xi = torch.stack([normals(n, seed, (1 << 63) + (k << 48) + row0) for k in range(S)])
    want = mean + F[:, :S].T + torch.sqrt(r) * xi
    assert torch.isfinite(out[:, :n]).all() and out[:, n:].isnan().all()  # nothing beyond n in each row of out
    assert rel(out[:, :n], want) < 1e-14


def test_sample_normals_match_the_regenerated_normals():
    from nonstationary_precip_b200 import ops
    W, S, seed = 160, 70, 99
    Et = torch.full((128, W), float("nan"), device="cuda")
    ops.sample_normals(W, S, seed, Et)
    want = torch.stack([normals(W, seed, s << 32) for s in range(S)])
    assert torch.equal(Et[:S], want) and bool((Et[S:] == 0).all())


# ---------------------------------------------------------------------------------------------------------------------
# snapshot, predictive after sampling, host sync
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["diag", "st"])
def test_snapshot_and_predictive_are_unaffected(kind):
    model, x, y = problem(kind, 128 if kind == "diag" else 64, seed=6, n=600)
    x, y = x.cuda(), y.cuda()
    post = model.posterior(x, y)
    xs = x[:200] + 0.02
    pred0 = post.predictive(xs)
    before = post.sample(xs, 32, seed=3)
    pred1 = post.predictive(xs)
    assert torch.equal(pred0.mean, pred1.mean) and torch.equal(pred0.var, pred1.var)
    model.neg_objective_and_grad(x, y, chunk=256)
    with torch.no_grad():
        for p in model.parameters():
            if p.grad is not None:
                p -= 0.05 * p.grad
    assert torch.equal(post.sample(xs, 32, seed=3), before)
    assert not torch.equal(model.posterior(x, y).sample(xs, 32, seed=3), before)


@pytest.mark.parametrize("kind,M,use_i8", [CASES[0], CASES[2], CASES[4], CASES[6]])
def test_sample_does_not_synchronise(kind, M, use_i8):
    model, x, y = problem(kind, M, seed=8, n=500, use_i8=use_i8)
    post = model.posterior(x.cuda(), y.cuda())
    xs = x.cuda() + 0.01
    post.sample(xs[:10], 8, chunk=128)  # warm-up outside the check (allocator, module loading)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        post.sample(xs, 70, seed=2, noise=True, row_offset=12, chunk=128)
    finally:
        torch.cuda.set_sync_debug_mode("default")
