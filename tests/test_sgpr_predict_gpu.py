"""Streamed prediction of the SGPR models (sgpr.py: posterior().predictive()) against the oracle's dense SGPR predictives,
the triangular row-norm kernel (npgp_o8_trinorm_digits) against exact products of its planes and against the q-only
row-quadratic pass, the finishing kernel against its formula, the test metrics against their closed forms, and the
determinism, snapshot and no-host-sync properties of the predictive."""
import math

import pytest
import torch

from oracle import gibbs_oracle as o

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


def rel(a, b):
    a, b = a.detach().cpu(), b.detach().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


# ---------------------------------------------------------------------------------------------------------------------
# models and oracles
# ---------------------------------------------------------------------------------------------------------------------
def diag_problem(n, M, D, seed):
    from nonstationary_precip_b200.sgpr import SGPRGibbsStream
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, D, generator=g) * 2 - 1
    y = torch.sin(3 * x[:, 0]) + 0.1 * torch.randn(n, generator=g)
    Z = x[torch.randperm(n, generator=g)[:M]].clone()
    le = math.log(0.3) + 0.2 * torch.randn(D, M, generator=g)
    c, os_, lam = torch.full((D,), math.log(0.3)), torch.ones(D), torch.full((D, D), 1.3)
    model = SGPRGibbsStream(Z.cuda(), le.cuda(), c.cuda(), os_.cuda(), lam.cuda(), outputscale=0.8, noise=0.05)
    return model, x, y


def diag_oracle(model, x, y, xs):
    c = lambda t: t.detach().cpu()  # noqa: E731
    s = torch.nn.functional.softplus(c(model.raw_outputscale)).reshape(())
    noise = (1e-4 + torch.nn.functional.softplus(c(model.raw_noise))).reshape(())
    return o.sgpr_gibbs_predict(x, y, c(model.Z), c(model.log_ell_z), xs, s, noise, c(model.prior_c), c(model.prior_os),
                                c(model.prior_lam))


def st_problem(n, M, seed):
    from nonstationary_precip_b200.sgpr import SGPRSpatioTemporalStream
    g = torch.Generator().manual_seed(seed)
    x = torch.cat([torch.rand(n, 1, generator=g) * 6 - 3, torch.rand(n, 2, generator=g) * 2 - 1], 1)
    y = torch.sin(2 * math.pi * x[:, 0] / 1.7) * torch.exp(-(x[:, 1:] ** 2).sum(-1)) + 0.1 * torch.randn(n, generator=g)
    Z = x[torch.randperm(n, generator=g)[:M]].clone()
    le = math.log(0.4) + 0.2 * torch.randn(2, M, generator=g)
    c, os_, lam = torch.full((2,), math.log(0.4)), torch.ones(2), torch.full((2, 2), 1.3)
    hyp0 = (0.12, 0.8, 1.7, 7.6)  # a short temporal lengthscale keeps the temporal Kzz well conditioned
    model = SGPRSpatioTemporalStream(Z.cuda(), le.cuda(), c.cuda(), os_.cuda(), lam.cuda(), hyp_t=hyp0, outputscale_s=0.8,
                                     noise=0.05)
    return model, x, y


def st_oracle(model, x, y, xs):
    c = lambda t: t.detach().cpu()  # noqa: E731
    sp = torch.nn.functional.softplus
    hyp = c(model.hyp_t())
    mean, cov = o.st_predict(x, y, c(model.Z), c(model.log_ell_z), xs, hyp, sp(c(model.raw_outputscale)).reshape(()),
                             (1e-4 + sp(c(model.raw_noise))).reshape(()), c(model.prior_c), c(model.prior_os),
                             c(model.prior_lam), literal=False)
    return mean, torch.diagonal(cov)


def check_metrics(pred, ys, noise):
    from nonstationary_precip_b200.utils import metrics
    assert torch.equal(pred.var_y, pred.var + noise)  # var_y = var_f + noise exactly
    r = ys - pred.mean
    lpd = -0.5 * (math.log(2 * math.pi) + torch.log(pred.var_y) + r * r / pred.var_y)
    assert rel(pred.lpd, lpd) < 1e-13
    want = torch.stack([(r * r).sum(), -lpd.sum(), torch.tensor(float(len(ys)), device=ys.device)])
    assert rel(pred.sums, want) < 1e-12 and pred.sums[2].item() == len(ys)
    n = pred.sums[2]
    assert abs(math.sqrt(pred.sums[0].item() / n.item()) - metrics.rmse(pred.mean, ys, 1.0).item()) < 1e-12
    nlpd = metrics.negative_log_predictive_density(ys, pred.mean, pred.var_y).item()
    assert abs(pred.sums[1].item() / n.item() - nlpd) < 1e-12 * max(1.0, abs(nlpd))


# ---------------------------------------------------------------------------------------------------------------------
# end to end against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,D,n_test,chunk", [(128, 1, 517, 128), (256, 2, 700, 333), (128, 3, 1030, 4096),
                                              (48, 2, 301, 100), (130, 3, 640, 256)])  # M % 128 == 0: digit planes
def test_diag_predictive_matches_oracle(M, D, n_test, chunk):
    model, x, y = diag_problem(900, M, D, seed=M + D)
    g = torch.Generator().manual_seed(7)
    xs = torch.rand(n_test, D, generator=g) * 2.2 - 1.1  # some rows outside the data: the clamp becomes inactive / active
    ys = torch.sin(3 * xs[:, 0])
    post = model.posterior(x.cuda(), y.cuda(), chunk=256)
    assert post.digits == (M % 128 == 0)
    pred = post.predictive(xs.cuda(), ys.cuda(), field=True, chunk=chunk)
    mean, var = diag_oracle(model, x, y, xs)
    em, ev = rel(pred.mean, mean), rel(pred.var, var)
    print("diag M=%d D=%d: mean %.2e var %.2e" % (M, D, em, ev))
    assert em < 1e-8 and ev < 1e-8
    ell_z = torch.exp(model.log_ell_z.detach().cpu())
    fld = o.field_interp_diag(xs, model.Z.detach().cpu(), ell_z, model.prior_c.cpu(), model.prior_os.cpu(),
                              model.prior_lam.cpu())
    assert rel(pred.field, fld) < 1e-8
    noise = (1e-4 + torch.nn.functional.softplus(model.raw_noise.detach())).reshape(())
    check_metrics(pred, ys.cuda(), noise)


def test_diag_digit_and_fp64_paths_agree():
    model, x, y = diag_problem(800, 128, 2, seed=5)
    xs = (torch.rand(999, 2) * 2 - 1).cuda()
    a = model.posterior(x.cuda(), y.cuda()).predictive(xs, chunk=300)
    model.use_i8 = False
    post = model.posterior(x.cuda(), y.cuda())
    assert not post.digits
    b = post.predictive(xs, chunk=300)
    assert rel(a.mean, b.mean) < 1e-11 and rel(a.var, b.var) < 1e-11


@pytest.mark.parametrize("M,n_test,chunk", [(64, 611, 256), (50, 420, 128)])  # 2M = 128: digit planes; 100: FP64
def test_spatio_temporal_predictive_matches_oracle(M, n_test, chunk):
    model, x, y = st_problem(700, M, seed=M)
    g = torch.Generator().manual_seed(9)
    xs = torch.cat([torch.rand(n_test, 1, generator=g) * 6 - 3, torch.rand(n_test, 2, generator=g) * 2 - 1], 1)
    ys = torch.sin(2 * math.pi * xs[:, 0] / 1.7)
    post = model.posterior(x.cuda(), y.cuda(), chunk=256)
    assert post.digits == ((2 * M) % 128 == 0)
    pred = post.predictive(xs.cuda(), ys.cuda(), field=True, chunk=chunk)
    mean, var = st_oracle(model, x, y, xs)
    em, ev = rel(pred.mean, mean), rel(pred.var, var)
    print("st M=%d: mean %.2e var %.2e" % (M, em, ev))
    assert em < 1e-8 and ev < 1e-8
    noise = (1e-4 + torch.nn.functional.softplus(model.raw_noise.detach())).reshape(())
    check_metrics(pred, ys.cuda(), noise)
    assert pred.field.shape == (2, n_test)


# ---------------------------------------------------------------------------------------------------------------------
# the triangular row-norm kernel
# ---------------------------------------------------------------------------------------------------------------------
def _planes(X, block_rows):
    from nonstationary_precip_b200 import ops
    R, Kd = X.shape
    d = torch.empty(ops.digits_bytes(R, Kd, block_rows), dtype=torch.uint8, device="cuda")
    e = torch.empty((R + block_rows - 1) // block_rows * block_rows, dtype=torch.int32, device="cuda")
    ops.o8_slice_rows(X, block_rows, d, e)
    return d, e


def _ints(X, e):
    """The integers the planes hold: y = rint(x 2^(54 - e)) per row (decoded value y 2^(e - 54))."""
    e = e[:X.shape[0]].cpu().to(torch.float64)
    return torch.round(X.cpu() * torch.exp2(54 - e)[:, None]).to(torch.int64), e


def _exact_product(Ya, Yb):
    """Ya Yb^T for |Y| <= 2^54 through 27-bit halves (each int64 product sum is exact), combined in FP64."""
    sh = lambda Y: (Y >> 27, Y & ((1 << 27) - 1))  # noqa: E731
    ah, al = sh(Ya)
    bh, bl = sh(Yb)
    f = lambda t: t.to(torch.float64)  # noqa: E731
    return f(ah @ bh.T) * 2.0 ** 54 + (f(ah @ bl.T) + f(al @ bh.T)) * 2.0 ** 27 + f(al @ bl.T)


def _tri_operand(N, Ms, g):
    B = torch.randn(N, N, generator=g).tril()
    if Ms:
        B[Ms:, :Ms] = 0.0
    return B


@pytest.mark.parametrize("n,N,Ms,per_row", [(300, 256, 0, True), (128, 128, 0, False), (517, 384, 128, True),
                                            (64, 256, 128, True)])
def test_trinorm_matches_exact_product_and_rowquad(n, N, Ms, per_row):
    from nonstationary_precip_b200 import ops
    g = torch.Generator().manual_seed(n + N)
    Ad = torch.rand(n, N, generator=g) * (torch.rand(n, 1, generator=g) * 4 if per_row else 1.0)
    if not per_row:
        Ad[:, 0] = 1.0  # every row's exponent is then the matrix-wide one of the scale bound 1
    Bm = _tri_operand(N, Ms, g)
    A, B = Ad.cuda(), Bm.cuda()
    a_d, a_e = _planes(A, 128)
    a_scale = None if per_row else torch.ones((), device="cuda")
    if not per_row:
        assert bool((a_e[:n] == 1).all())
    b_d, b_e = _planes(B, 64)
    q = torch.full((N // 64, n + 5), float("nan"), device="cuda")
    ops.o8_trinorm_digits(n, N, N, a_d, a_scale, b_d, b_e, q, Ms=Ms, a_expo=a_e if per_row else None)
    # exact reference from the integers of the planes
    Ya, ea = _ints(A, a_e)
    Yb, eb = _ints(B, b_e)
    T = _exact_product(Ya, Yb) * torch.exp2(ea - 108)[:, None] * torch.exp2(eb)[None, :]
    want = (T * T).reshape(n, N // 64, 64).sum(-1).T
    Aq = Ya.to(torch.float64) * torch.exp2(ea - 54)[:, None]
    Bq = Yb.to(torch.float64) * torch.exp2(eb - 54)[:, None]
    bound = (Aq.norm(dim=1)[None, :] ** 2) * (Bq.norm(dim=1) ** 2).reshape(N // 64, 64).sum(-1)[:, None]
    err = ((q[:, :n].cpu() - want).abs() / bound).max().item()
    print("trinorm n=%d N=%d Ms=%d: %.2e of |A||B|" % (n, N, Ms, err))
    assert err <= 1e-14
    assert bool(torch.isnan(q[:, n:]).all())  # nothing past n is written
    # the q-only row-quadratic pass against P^T P gives the same |B a|^2
    C = (B.T @ B).contiguous()
    c_d, c_e = _planes(C, 64)
    qp = torch.empty(N // 64, n, device="cuda")
    ops.o8_rowquad_digits(n, N, a_d, a_scale, c_d, c_e, None, q_part=qp, a_expo=a_e if per_row else None)
    assert rel(q[:, :n].sum(0), qp.sum(0)) < 1e-12


@pytest.mark.parametrize("Ms", [0, 128])
def test_trinorm_never_reads_the_skipped_k_steps(Ms):
    from nonstationary_precip_b200 import ops
    n, N = 333, 256
    g = torch.Generator().manual_seed(Ms + 1)
    A = (torch.rand(n, N, generator=g) * torch.rand(n, 1, generator=g)).cuda()
    a_d, a_e = _planes(A, 128)
    b_d, b_e = _planes(_tri_operand(N, Ms, g).cuda(), 64)
    q0 = torch.empty(N // 64, n, device="cuda")
    ops.o8_trinorm_digits(n, N, N, a_d, None, b_d, b_e, q0, Ms=Ms, a_expo=a_e)
    # B planes: [row block rb][k-step ks][7 digits x 2 halves x 64 rows x 16 bytes]; fill the k-steps the kernel skips
    nks = N // 32
    st = b_d.view(N // 64, nks, 7 * 2 * 64 * 16)
    junk = torch.randint(0, 256, st.shape, generator=g, dtype=torch.uint8).cuda()
    for rb in range(N // 64):
        lo = Ms // 32 if Ms and 64 * rb >= Ms else 0
        st[rb, 2 * (rb + 1):] = junk[rb, 2 * (rb + 1):]  # past the diagonal block
        st[rb, :lo] = junk[rb, :lo]                      # the zero quadrant of the split
    q1 = torch.empty_like(q0)
    ops.o8_trinorm_digits(n, N, N, a_d, None, b_d, b_e, q1, Ms=Ms, a_expo=a_e)
    assert torch.equal(q0, q1)


# ---------------------------------------------------------------------------------------------------------------------
# the finishing kernel
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb_t", [0, 3])
def test_finish_matches_formula(nb_t):
    from nonstationary_precip_b200 import ops
    n, nb_s, nb_v = 1000, 4, 7
    g = torch.Generator().manual_seed(nb_t)
    s, noise, os_t = torch.tensor(0.7), torch.tensor(0.03), torch.tensor(7.5)
    qn = torch.rand(nb_t + nb_s, n, generator=g) * 0.3
    qn[nb_t:, :100] *= 5.0  # these rows' Gibbs clamp is active
    if nb_t:
        qn[:nb_t, 100:200] = torch.rand(nb_t, 100, generator=g) * 4.0  # temporal clamp active on most of these
    qv = torch.rand(nb_v, n, generator=g) * 0.1
    mean, y = torch.randn(n, generator=g), torch.randn(n, generator=g)
    dev = lambda t: t.cuda().contiguous()  # noqa: E731
    var, var_y, lpd = (torch.empty(n, device="cuda") for _ in range(3))
    sums = torch.zeros(3, device="cuda")
    work = ops.sgpr_predict_workspace(n, "cuda")
    for _ in range(2):  # sums accumulate; the kernel leaves its ticket at 0 for the next call
        ops.sgpr_predict_finish(dev(qn), nb_t, dev(qv), dev(s), dev(noise), var, os_t=dev(os_t) if nb_t else None,
                                mean=dev(mean), y=dev(y), var_y=var_y, lpd=lpd, sums=sums, work=work)
    want = s * (1 - qn[nb_t:].sum(0)).clamp_min(0) + qv.sum(0)
    if nb_t:
        want = want + (os_t - qn[:nb_t].sum(0)).clamp_min(0)
        assert bool(((os_t - qn[:nb_t].sum(0)) < 0).any())
    assert bool(((1 - qn[nb_t:].sum(0)) < 0).any())
    assert rel(var, want) < 1e-14
    assert torch.equal(var_y, var + noise.cuda())
    r = y - mean
    wl = -0.5 * (math.log(2 * math.pi) + torch.log(want + noise) + r * r / (want + noise))
    assert rel(lpd, wl) < 1e-13
    assert rel(sums, 2 * torch.stack([(r * r).sum(), -wl.sum(), torch.tensor(float(n))])) < 1e-12
    assert int(work[:4].view(torch.int32).item()) == 0


# ---------------------------------------------------------------------------------------------------------------------
# determinism, sharding, snapshot, host sync
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,M", [("diag", 256), ("st", 64), ("diag", 48)])
def test_predictive_is_deterministic_and_chunking_invariant(kind, M):
    model, x, y = diag_problem(700, M, 2, seed=3) if kind == "diag" else st_problem(700, M, seed=3)
    post = model.posterior(x.cuda(), y.cuda(), chunk=200)
    xs = x[:600].cuda() + 0.01
    ys = y[:600].cuda()
    a = post.predictive(xs, ys, chunk=256)
    b = post.predictive(xs, ys, chunk=256)
    for f in ("mean", "var", "var_y", "lpd", "sums"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    # rows split at a chunk boundary across two calls concatenate to the bits of one call
    c1, c2 = post.predictive(xs[:512], chunk=256), post.predictive(xs[512:], chunk=256)
    assert torch.equal(torch.cat([c1.mean, c2.mean]), a.mean) and torch.equal(torch.cat([c1.var, c2.var]), a.var)
    big = post.predictive(xs, ys, chunk=4096)
    assert rel(big.mean, a.mean) < 1e-12 and rel(big.var, a.var) < 1e-12 and rel(big.sums, a.sums) < 1e-12


@pytest.mark.parametrize("kind", ["diag", "st"])
def test_posterior_from_two_emulated_ranks_matches_one(kind):
    model, x, y = diag_problem(800, 128, 2, seed=4) if kind == "diag" else st_problem(800, 64, seed=4)
    x, y = x.cuda(), y.cuda()
    xs = x[:300] * 0.97
    full = model.posterior(x, y, chunk=256).predictive(xs)
    halves = [(x[:400], y[:400]), (x[400:], y[400:])]
    got = []
    model.posterior(*halves[1], chunk=256, n_total=800, all_reduce=lambda t: got.append(t.clone()))
    post = model.posterior(*halves[0], chunk=256, n_total=800, all_reduce=lambda t: t.add_(got[0]))
    two = post.predictive(xs)
    assert rel(two.mean, full.mean) < 1e-10 and rel(two.var, full.var) < 1e-10


@pytest.mark.parametrize("kind", ["diag", "st"])
def test_posterior_is_a_snapshot(kind):
    model, x, y = diag_problem(600, 128, 2, seed=6) if kind == "diag" else st_problem(600, 64, seed=6)
    x, y = x.cuda(), y.cuda()
    post = model.posterior(x, y)
    xs = x[:200] + 0.02
    before = post.predictive(xs)
    model.neg_objective_and_grad(x, y, chunk=256)
    with torch.no_grad():
        for p in model.parameters():
            if p.grad is not None:
                p -= 0.05 * p.grad
    after = post.predictive(xs)
    assert torch.equal(before.mean, after.mean) and torch.equal(before.var, after.var)
    assert not torch.equal(model.posterior(x, y).predictive(xs).mean, before.mean)


@pytest.mark.parametrize("kind,M", [("diag", 128), ("st", 64), ("diag", 48), ("st", 50)])
def test_predictive_does_not_synchronise(kind, M):
    model, x, y = diag_problem(500, M, 2, seed=8) if kind == "diag" else st_problem(500, M, seed=8)
    post = model.posterior(x.cuda(), y.cuda())
    xs, ys = x.cuda() + 0.01, y.cuda()
    post.predictive(xs[:10], ys[:10], chunk=128)  # warm-up outside the check (allocator, module loading)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        post.predictive(xs, ys, field=True, chunk=128)
    finally:
        torch.cuda.set_sync_debug_mode("default")
