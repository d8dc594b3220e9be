"""Posterior snapshots of the Gibbs GPs of the spatial experiment (DiagonalExactGP.posterior, DiagonalSparseGP.posterior):
the exact GP's marginals and field against the oracle's dense predictive on the digit and FP64 paths, its draws against
mean + K_U V^T E + sqrt(r + 1e-4) xi formed in FP64 from regenerated normals, the covariance of the draws against the dense
joint (equal diagonal, off-diagonal difference = the Nystrom residual, smaller with knots), the moments of many draws, the
invariances of the keys, the snapshot and no-host-sync properties, the sparse model's snapshot against its own predict(),
the finishing kernel npgp_exact_predict_finish against its formula, and the map of experiments/spatial_exp.py."""
import math

import numpy as np
import pytest
import torch

from oracle import gibbs_oracle as o
from test_sgpr_predict_gpu import check_metrics, rel
from test_sgpr_sample_gpu import normals

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)

S_OUT, NOISE = 0.644, 0.011  # the experiment's fixed outputscale and noise
C, OS, LAM = math.log(0.3), 1.0, 1.3  # the experiment's prior


def make_prior(D):
    from nonstationary_precip_b200.models.gibbs_kernels import LogNormalPriorProcess
    prior = LogNormalPriorProcess(input_dim=D).cuda().double()
    prior.covar_module.outputscale = OS * torch.ones_like(prior.covar_module.outputscale)
    prior.covar_module.base_kernel.lengthscale = LAM * torch.ones_like(prior.covar_module.base_kernel.lengthscale)
    prior.mean_module.constant = torch.nn.Parameter(C * torch.ones_like(prior.mean_module.constant))
    for p in prior.parameters():
        p.requires_grad = False
    return prior


def hypers(D):
    return torch.full((D,), C), torch.full((D,), OS), torch.full((D, D), LAM)


def exact_problem(n, D, seed, use_i8=True):
    """A DiagonalExactGP with the experiment's outputscale, noise and prior: x in [-1, 1]^D, y = sin(3 x_0) + noise."""
    from nonstationary_precip_b200.gp_base import GaussianLikelihood
    from nonstationary_precip_b200.models.nonstationary_models import DiagonalExactGP
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, D, generator=g) * 2 - 1
    y = torch.sin(3 * x[:, 0]) + 0.1 * torch.randn(n, generator=g)
    model = DiagonalExactGP(x.cuda(), y.cuda(), GaussianLikelihood().cuda().double(), make_prior(D), num_dim=D)
    model = model.cuda().double()
    model.likelihood.noise = NOISE
    model.covar_module.outputscale = S_OUT
    with torch.no_grad():  # short lengthscales keep K_XX (the knots' Gram matrix) far from singular: the draws take j = 0
        model.log_ell_train_x.copy_(math.log(0.1) + 0.2 * torch.randn(D, n, generator=g))
    model.eval()
    model.use_i8 = use_i8
    return model, x, y


def oracle(model, x, y, xs):
    le = model.log_ell_train_x.detach().cpu()
    return o.exact_gp_predict(x, y, le, xs.cpu(), torch.tensor(S_OUT), torch.tensor(NOISE), *hypers(x.shape[1]))


def rows_in(D, n, seed, spread=1.4):
    g = torch.Generator().manual_seed(seed)
    return ((torch.rand(n, D, generator=g) * 2 - 1) * spread).cuda()  # spread > 1: rows outside the data too


def grid_knots(G, D=2, lim=1.0):
    a = torch.linspace(-lim, lim, G)
    return torch.stack(torch.meshgrid(*([a] * D), indexing="ij"), -1).reshape(-1, D).cuda()


@torch.no_grad()
def draw_parts(post, n_u, xs):
    """FP64 parts of the draws from the snapshot's columns: K_U (rows, Wp), P_U = chol(K_UU)^-1 padded, the residual
    r = s max(1 - |P_U k|^2, 0) and a bound on the rounding of the snapshot's r."""
    from nonstationary_precip_b200 import functional as F, ops
    ell = post.predictive(xs, field=True).field
    K = ops.gibbs_diag_fwd(xs, ell, post.Z, post.ell_z)
    U, eu = post.Z[:n_u].contiguous(), post.ell_z[:, :n_u].contiguous()
    _, PU, info = F.chol_inv(F.gibbs_diag(U, eu, U, eu))
    assert int(info) == 0  # j = 0
    P = torch.zeros(post.width, post.width, device="cuda")
    P[:n_u, :n_u] = PU
    G = K @ P.T
    r = post.s * (1 - (G ** 2).sum(1)).clamp_min(0)
    # rounding of |P_U k|^2: 1e-14 of the size |k|^2 |P_U|_F^2 of its terms, plus, on the digit path, the digits of k, which
    # are exact to about 2^-56 of their bound 1 rather than of |k|: an absolute 1e-16 per entry
    e = 1e-16 * P.abs().sum(1).norm()
    dr = post.s * (1e-14 * (K ** 2).sum(1) * (P ** 2).sum() + 2 * e * G.norm(dim=1) + e * e)
    return K, P, r, dr


# ---------------------------------------------------------------------------------------------------------------------
# marginals against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,D", [(316, 2), (1, 2), (127, 1), (128, 3), (129, 2), (1000, 3), (1000, 1)])
def test_predictive_matches_oracle_on_both_paths(n, D):
    model, x, y = exact_problem(n, D, seed=n + D)
    xs = rows_in(D, 433, seed=n)
    ys = torch.sin(3 * xs[:, 0])
    mean_o, sigma = oracle(model, x, y, xs)
    var_o = torch.diagonal(sigma)
    preds = []
    for use_i8 in (True, False):
        model.use_i8 = use_i8
        post = model.posterior()
        assert post.digits == use_i8 and post.width % 128 == 0
        pred = post.predictive(xs, ys, field=True, chunk=200)
        em, ev = rel(pred.mean, mean_o), rel(pred.var, var_o)
        print("n=%d D=%d i8=%d: mean %.2e var %.2e" % (n, D, use_i8, em, ev))
        assert em < 1e-8 and ev < 1e-8
        fld = o.field_interp_diag(xs.cpu(), x, torch.exp(model.log_ell_train_x.detach().cpu()), *hypers(D))
        assert rel(pred.field, fld) < 1e-8
        check_metrics(pred, ys, post.noise)
        preds.append(pred)
    a, b = preds
    # the mean k^T u cancels: the two paths agree to a small multiple of 1e-11 of the size sum_j |k_j| |u_j| of its terms,
    # where the digits of k are exact to about 2^-56 of their bound 1 rather than of |k_j| (the 1e-3 sum_j |u_j| term: rows
    # far from the data).  Measured on a B200 over three runs, which differ in the last bits at n = 1000: the mean to at most
    # 1.6e-11 of max |mean| and 1.2e-11 of the terms at n = 1000 (1e-14 below), var to at most 9.3e-12 of max var
    from nonstationary_precip_b200 import ops
    K = ops.gibbs_diag_fwd(xs, a.field, post.Z, post.ell_z)
    size = K.abs() @ post.u.abs() + 1e-3 * post.u.abs().sum()
    print("n=%d D=%d: digit - FP64 mean %.2e of max |mean|, %.2e of the terms; var %.2e" % (
        n, D, rel(a.mean, b.mean), ((a.mean - b.mean).abs() / size).max().item(), rel(a.var, b.var)))
    assert ((a.mean - b.mean).abs() <= 5e-11 * size).all() and rel(a.var, b.var) < 2e-11


@pytest.mark.parametrize("use_i8", [True, False])
def test_predictive_does_not_depend_on_knots(use_i8):
    model, x, y = exact_problem(316, 2, seed=2, use_i8=use_i8)
    xs = rows_in(2, 700, seed=3)
    a = model.posterior().predictive(xs, chunk=256)
    for knots in (grid_knots(16), rows_in(2, 300, seed=4)):  # width 640 / 640 instead of 384
        post = model.posterior(knots=knots)
        assert post.width == 640
        b = post.predictive(xs, chunk=256)
        assert rel(b.mean, a.mean) < 1e-12 and rel(b.var, a.var) < 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# draws: construction, covariance, moments
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m,use_i8", [(316, 0, True), (316, 100, True), (129, 0, False), (127, 64, False)])
def test_draws_equal_the_fp64_construction(n, m, use_i8):
    model, x, y = exact_problem(n, 2, seed=n + m, use_i8=use_i8)
    post = model.posterior(knots=rows_in(2, m, seed=9, spread=1.0) if m else None)
    xs = rows_in(2, 600, seed=m + 1)
    S, seed, chunk = 40, 4321, 256
    rows, W = xs.shape[0], post.width
    K, P, r, dr = draw_parts(post, n + m, xs)
    E = torch.stack([normals(W, seed, s << 32) for s in range(S)], 1)  # (W, S)
    xi = torch.stack([normals(rows, seed, (1 << 63) + (s << 48)) for s in range(S)])
    V = post.V
    KW = (K @ (V.T @ E)).T
    # K V^T E: rounding relative to sum_j |K_ij| (|V|^T |E|)_js, plus the digits of K (absolute, see draw_parts)
    scale = (K.abs() @ (V.abs().T @ E.abs())).T + 1e-3 * (V.abs().T @ E.abs()).sum(0)[:, None]
    mean = post.predictive(xs, chunk=chunk).mean
    for with_noise in (False, True):
        got = post.sample(xs, S, seed=seed, noise=with_noise, chunk=chunk)
        assert got.shape == (S, rows) and torch.isfinite(got).all()
        sd = torch.sqrt(r + 1e-4 + (post.noise if with_noise else 0.0))
        want = mean + KW + sd * xi
        dsd = torch.minimum(dr / (2 * sd), torch.sqrt(dr)) + 1e-14 * sd
        bound = 1e-12 * scale + dsd * xi.abs() + 1e-15 * mean.abs()
        err = (got - want).abs()
        assert (err <= bound).all(), (err / bound).max().item()


def test_covariance_against_the_dense_joint_and_the_nystrom_residual():
    from nonstationary_precip_b200 import functional as F
    model, x, y = exact_problem(316, 2, seed=11)
    xs = rows_in(2, 300, seed=12, spread=1.1)
    _, sigma = oracle(model, x, y, xs)
    sigma = sigma.cuda()
    off = ~torch.eye(xs.shape[0], dtype=torch.bool, device="cuda")
    gaps = []
    for knots in (None, grid_knots(16, lim=1.1)):
        post = model.posterior(knots=knots)
        n_u = 316 + (0 if knots is None else knots.shape[0])
        K, P, r, _ = draw_parts(post, n_u, xs)
        Rk = K @ post.V.T
        cov = Rk @ Rk.T + torch.diag(r + 1e-4)
        ed = rel(torch.diagonal(cov), torch.diagonal(sigma))
        # the Nystrom residual s (k(x, x') - k_U^T K_UU^-1 k_U'), off the diagonal
        ell = post.predictive(xs, field=True).field
        G = K @ P.T
        nys = post.s * (F.gibbs_diag(xs, ell, xs, ell) - G @ G.T)
        en = rel((sigma - cov)[off], nys[off])
        gap = (sigma - cov)[off].abs().max().item()
        print("knots %s: diag %.2e, residual identity %.2e, max off-diagonal gap %.3e" % (
            None if knots is None else knots.shape[0], ed, en, gap))
        assert ed < 1e-8
        assert ((sigma - cov)[off] - nys[off]).abs().max() < 1e-8 * sigma.abs().max()
        gaps.append(gap)
    assert gaps[1] < 0.5 * gaps[0]  # a grid of knots makes the residual smaller


def test_moments_of_many_draws():
    model, x, y = exact_problem(316, 2, seed=21)
    post = model.posterior()
    xs = torch.cat([x[:5].cuda() + 0.02, rows_in(2, 40, seed=22)]).contiguous()
    draws = torch.cat([post.sample(xs, 1024, seed=100 + k) for k in range(8)])  # (8192, n)
    N = draws.shape[0]
    K, P, r, _ = draw_parts(post, 316, xs)
    Rk = K @ post.V.T
    cov = Rk @ Rk.T + torch.diag(r + 1e-4)
    mean_o, sigma = oracle(model, x, y, xs)
    mean_o, var = mean_o.cuda(), torch.diagonal(sigma).cuda()
    avg = draws.mean(0)
    assert ((avg - mean_o).abs() <= 6 * torch.sqrt(var / N)).all()
    dev = draws - avg
    emp = dev.T @ dev / (N - 1)
    band = 6 * torch.sqrt((var[:, None] * var[None, :] + cov ** 2) / (N - 1))
    assert ((emp - cov).abs() <= band).all(), ((emp - cov).abs() / band).max().item()
    assert (torch.diagonal(emp) - var).abs().max() <= 6 * (var * math.sqrt(2.0 / (N - 1))).max()


# ---------------------------------------------------------------------------------------------------------------------
# invariances, snapshot, host sync
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_i8", [True, False])
def test_seeds_sample_counts_row_offsets_chunks_and_shards(use_i8):
    model, x, y = exact_problem(316, 2, seed=17, use_i8=use_i8)
    post = model.posterior(knots=grid_knots(8))
    xs = rows_in(2, 700, seed=19)
    ys = torch.sin(3 * xs[:, 0])
    chunk = 256
    a = post.sample(xs, 64, seed=5, chunk=chunk)
    assert torch.equal(a, post.sample(xs, 64, seed=5, chunk=chunk))
    assert not (post.sample(xs, 64, seed=6, chunk=chunk) == a).any()
    assert torch.equal(post.sample(xs, 16, seed=5, chunk=chunk), a[:16])
    assert torch.equal(post.sample(xs, 100, seed=5, chunk=chunk)[:64], a)
    h = 300  # two emulated ranks, each with its global row offset: the rows of one call
    two = torch.cat([post.sample(xs[:h], 64, seed=5, chunk=chunk),
                     post.sample(xs[h:], 64, seed=5, row_offset=h, chunk=chunk)], 1)
    assert rel(two, a) <= 1e-13
    assert rel(post.sample(xs, 64, seed=5, chunk=4096), a) <= 1e-12
    # noise=True adds the noise variance to the residual and nothing else
    b = post.sample(xs, 64, seed=5, noise=True, chunk=chunk)
    mean = post.predictive(xs, chunk=chunk).mean
    K, P, r, _ = draw_parts(post, 316 + 64, xs)
    xi = torch.stack([normals(xs.shape[0], 5, (1 << 63) + (s << 48)) for s in range(64)])
    want = (a - mean) + (torch.sqrt(r + 1e-4 + post.noise) - torch.sqrt(r + 1e-4)) * xi
    assert rel(b - mean, want) < 1e-9  # r enters through 1 / sd: its rounding is amplified
    # the predictive's sums over two shards add up to the full sums
    full = post.predictive(xs, ys, chunk=chunk)
    p1, p2 = post.predictive(xs[:h], ys[:h], chunk=chunk), post.predictive(xs[h:], ys[h:], chunk=chunk)
    assert rel(p1.sums + p2.sums, full.sums) < 1e-12
    assert rel(torch.cat([p1.var, p2.var]), full.var) < 1e-13


def test_snapshot_is_unaffected_by_later_updates():
    model, x, y = exact_problem(316, 2, seed=6)
    post = model.posterior(knots=grid_knots(6))
    xs = rows_in(2, 200, seed=7)
    pred0, draws0 = post.predictive(xs, field=True), post.sample(xs, 32, seed=3)
    with torch.no_grad():
        model.log_ell_train_x += 0.1
        model.covar_module.outputscale = 0.9
        model.likelihood.noise = 0.02
    pred1 = post.predictive(xs, field=True)
    assert torch.equal(pred0.mean, pred1.mean) and torch.equal(pred0.var, pred1.var)
    assert torch.equal(pred0.field, pred1.field) and torch.equal(post.sample(xs, 32, seed=3), draws0)
    assert not torch.equal(model.posterior(knots=grid_knots(6)).sample(xs, 32, seed=3), draws0)


@pytest.mark.parametrize("use_i8", [True, False])
def test_chunk_loop_does_not_synchronise(use_i8):
    model, x, y = exact_problem(316, 2, seed=8, use_i8=use_i8)
    post = model.posterior()
    xs = rows_in(2, 500, seed=9)
    ys = torch.sin(3 * xs[:, 0])
    post.predictive(xs[:10], ys[:10], field=True, chunk=128)  # warm-up outside the check
    post.sample(xs[:10], 8, chunk=128)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        post.predictive(xs, ys, field=True, chunk=128)
        post.sample(xs, 70, seed=2, noise=True, row_offset=12, chunk=128)
    finally:
        torch.cuda.set_sync_debug_mode("default")


def test_jitter_that_reaches_tau_is_an_error(monkeypatch):
    from nonstationary_precip_b200 import functional as F
    model, x, y = exact_problem(128, 2, seed=30)
    chol_inv = F.chol_inv

    def knots_need_jitter(A):  # K_UU (128 + 20 columns, unit diagonal) does not factor without jitter; all else does
        L, P, info = chol_inv(A)
        return L, P, (info + 1 if A.shape[0] == 148 and abs(float(A[0, 0]) - 1.0) < 1e-12 else info)
    monkeypatch.setattr(F, "chol_inv", knots_need_jitter)
    knots = rows_in(2, 20, seed=31)
    model.posterior(knots=knots)  # tau = 0.011 / 0.644: the jitter 1e-8 is below it
    model.covar_module.outputscale = 1e7  # tau ~ 1e-9, below the ladder's first jitter
    with pytest.raises(ValueError, match="jitter"):
        model.posterior(knots=knots)


# ---------------------------------------------------------------------------------------------------------------------
# the reference-shaped sparse model
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [64, 128])  # FP64 path, digit path
def test_sparse_model_posterior_matches_its_predict(M):
    from nonstationary_precip_b200 import functional as F
    from nonstationary_precip_b200.gp_base import GaussianLikelihood
    from nonstationary_precip_b200.models.nonstationary_models import DiagonalSparseGP
    g = torch.Generator().manual_seed(M)
    n, D = 500, 2
    x = torch.rand(n, D, generator=g) * 2 - 1
    y = torch.sin(3 * x[:, 0]) + 0.1 * torch.randn(n, generator=g)
    z = x[torch.randperm(n, generator=g)[:M]].clone()
    model = DiagonalSparseGP(x.cuda(), y.cuda(), GaussianLikelihood().cuda().double(), make_prior(D), z.cuda(),
                             num_dim=D).cuda().double()
    model.likelihood.noise = 0.05
    model.covar_module.outputscale = 0.8
    with torch.no_grad():
        model.log_ell_z += 0.2 * torch.randn(D, M, generator=g).cuda()
    model.eval()
    post = model.posterior()
    assert post.digits == (M % 128 == 0)
    xs = rows_in(D, 300, seed=M + 1, spread=1.1)
    pred = post.predictive(xs, field=True)
    with torch.no_grad():
        ref = model.predict(xs)
    mean_o, var_o = o.sgpr_gibbs_predict(x, y, z, model.log_ell_z.detach().cpu(), xs.cpu(), torch.tensor(0.8),
                                         torch.tensor(0.05), *hypers(D))
    assert rel(pred.mean, mean_o) < 1e-8 and rel(pred.var, var_o) < 1e-8
    assert rel(pred.mean, ref.mean) < 1e-8 and rel(pred.var, torch.diagonal(ref.covariance_matrix)) < 1e-8
    # the draws' covariance (V k)^T (V k') + delta r is predict()'s joint
    with torch.no_grad():
        ell_z = torch.exp(model.log_ell_z)
        Zc = model.covar_module.base_kernel.inducing_points
        _, P = F.psd_safe_chol_inv(F.gibbs_diag(Zc, ell_z, Zc, ell_z))
        K = F.gibbs_diag(xs, pred.field, Zc, ell_z)
    Rk = K @ post.V.T
    r = post.s * (1 - ((K @ P.T) ** 2).sum(1)).clamp_min(0)
    assert rel(Rk @ Rk.T + torch.diag(r), ref.covariance_matrix) < 1e-8


# ---------------------------------------------------------------------------------------------------------------------
# the finishing kernel
# ---------------------------------------------------------------------------------------------------------------------
def test_exact_finish_matches_formula():
    from nonstationary_precip_b200 import ops
    n, nb, add_var = 1000, 5, 1e-4
    g = torch.Generator().manual_seed(1)
    s, noise = torch.tensor(0.644).cuda(), torch.tensor(0.011).cuda()
    qn = torch.rand(nb, n, generator=g) * 0.2
    qn[:, :100] *= 2.0  # these rows' clamp is active
    qn = qn.cuda()
    mean, y = torch.randn(n, generator=g).cuda(), torch.randn(n, generator=g).cuda()
    var, var_y, lpd = (torch.empty(n, device="cuda") for _ in range(3))
    sums = torch.zeros(3, device="cuda")
    work = ops.sgpr_predict_workspace(n, "cuda")
    for _ in range(2):  # sums accumulate; the kernel leaves its ticket at 0 for the next call
        ops.exact_predict_finish(qn, s, noise, add_var, var, mean=mean, y=y, var_y=var_y, lpd=lpd, sums=sums, work=work)
    want = s * (1 - qn.sum(0)).clamp_min(0) + add_var
    assert bool(((1 - qn.sum(0)) < 0).any())
    assert rel(var, want) < 1e-14
    assert torch.equal(var_y, var + noise)
    r = y - mean
    wl = -0.5 * (math.log(2 * math.pi) + torch.log(want + noise) + r * r / (want + noise))
    assert rel(lpd, wl) < 1e-13
    assert rel(sums, 2 * torch.stack([(r * r).sum(), -wl.sum(), torch.tensor(float(n), device="cuda")])) < 1e-12
    assert int(work[:4].view(torch.int32).item()) == 0
    only = torch.empty(n, device="cuda")  # var_f alone: no y, no sums
    ops.exact_predict_finish(qn, s, noise, add_var, only)
    assert torch.equal(only, var)


# ---------------------------------------------------------------------------------------------------------------------
# the experiment's map
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("inference", ["exact", "sparse"])
def test_spatial_exp_writes_the_map(inference, tmp_path):
    from experiments import spatial_exp as se
    out = str(tmp_path / "map.npz")
    args = se.parse_args(["--n_iter", "3", "--splits", "1", "--inference", inference, "--M", "64", "--log_every", "2",
                          "--map_grid", "64", "--map_samples", "4", "--map_out", out])
    x, y = se.load_khyber_data()
    se.run_split(0, x, y, args, torch.device("cuda"), log=lambda *_: None)
    m = np.load(out)
    assert m["mean"].shape == (64, 64) and m["var_y"].shape == (64, 64) and m["ell"].shape == (2, 64, 64)
    assert m["samples"].shape == (4, 64, 64) and m["lon"].shape == (64,) and m["lat"].shape == (64,)
    assert all(np.isfinite(m[k]).all() for k in m.files) and (m["var_y"] > 0).all() and (m["ell"] > 0).all()
    assert m["lon"][0] >= x[:, 0].min().item() - 1e-9 and m["lon"][-1] <= x[:, 0].max().item() + 1e-9
    # the map's mean is the predictive mean in the original units: within the range of the data, give or take
    assert abs(m["mean"].mean() - y.mean().item()) < 3 * y.std().item()
