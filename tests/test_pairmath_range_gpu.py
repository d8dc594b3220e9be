"""The per-pair arithmetic of csrc/pairmath.cuh (table-driven exp_neg, fast_rsqrt / fast_rcp, closed-form 2x2 / 3x3
determinants and adjugates) through every kernel that uses it, at every dimension the C API accepts, entry by entry against
an extended-precision evaluation of the reference's own formulas (oracle/gibbs_oracle.py), over the whole exponent range and
with non-finite inputs.

Tolerances follow the conditioning of each entry instead of one global max: an entry far below the largest one (K ~ 1e-200, a
small row of a gradient) is checked at its own scale.  For K the bound is |K - K_ref| <= c eps (1 + Q_ij) |K_ref| with Q_ij
the exponent argument and c = C_PAIR(D) = 8 (D + 2); a gradient entry is bounded by c eps times the sum over the reduced
axis of |G_ij| |dK_ij/dtheta| (1 + Q_ij), |dK/dtheta| taken term by term, plus the rounding of that sum."""
import math
import os
import re

import mpmath
import numpy as np
import pytest
import torch

from oracle import gibbs_oracle as o

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)

LD = np.longdouble
assert np.finfo(LD).eps < 2.0 ** -60, "the reference needs an extended-precision long double (64-bit mantissa)"
EPS = 2.0 ** -53
EXP_FLOOR = 3.4e-308          # exp_neg clamps its argument at -708: exp(-708) = 3.3e-308 stands in for the tail
SUBNORMAL_SLACK = 2.0 ** -1070  # products that end below DBL_MIN lose relative precision
SCALE = 0.644


def C_PAIR(D):
    return 8 * (D + 2)


def ops():
    from nonstationary_precip_b200 import ops as _ops
    return _ops


def ld(t):
    return t.detach().cpu().numpy().astype(LD)


def f64(a):
    return torch.from_numpy(np.asarray(a, dtype=np.float64))


def sum_slack(n):
    """Rounding of an n-term FP64 sum relative to the sum of the absolute terms (tile partials + atomics)."""
    return 4.0 * math.sqrt(n) * EPS


# ------------------------------------------------------------------------------------------------------- 1. exp_neg
def exp_neg_device(x):
    """exp_neg(-0.5 fl(x^2)) per entry of x, through the d = nb = nv = 1 field kernel with lam = os = V = 1, one column z = 0,
    no bias, no exp: the kernel forms q = fma(x, x, 0) and adds one product k * 1 to zero."""
    one = torch.ones(1, 1, device="cuda")
    out = ops().rbf_matvec_fwd(x.reshape(-1, 1).cuda(), torch.zeros(1, 1, device="cuda"), one, torch.ones(1, device="cuda"),
                               one.reshape(1, 1, 1), bias=None, apply_exp=False)
    return out.reshape(-1).cpu()


def test_exp_neg_every_table_interval_and_the_clamp():
    rng = np.random.default_rng(0)
    ln2_256 = math.log(2.0) / 256
    # both ends of every table interval j = 0..255, at several octaves k, and a dense sweep of [-720, 0]
    ks = np.array([0, -1, -2, -37, -500, -1000, -1021])
    js = np.arange(256)
    centres = (256 * ks[:, None] + js[None, :]).reshape(-1) * ln2_256
    ends = np.concatenate([centres - 0.5 * ln2_256 * (1 - 1e-12), centres + 0.5 * ln2_256 * (1 - 1e-12)])
    args = np.concatenate([-np.linspace(0.0, 720.0, 100001), -rng.uniform(0, 720, 20000), ends, [0.0, -1e-300, -708.0]])
    args = args[args <= 0]
    x = np.sqrt(-2.0 * args)
    a = -0.5 * (x * x)  # the argument the kernel sees: x*x rounded once, the halving is exact
    got = exp_neg_device(torch.from_numpy(x)).numpy()
    mpmath.mp.prec = 113
    ref = np.array([float(mpmath.exp(mpmath.mpf(float(v)))) for v in a])
    inside = a >= -708.0
    ulps = np.abs(got[inside] - ref[inside]) / np.spacing(ref[inside])
    assert ulps.max() <= 3.0, (ulps.max(), a[inside][ulps.argmax()])
    assert (got[~inside] >= 0).all() and (got[~inside] <= EXP_FLOOR).all()
    assert got[a == 0.0].tolist() == [1.0] * int((a == 0.0).sum())


def test_exp_neg_non_finite_arguments():
    x = torch.tensor([float("nan"), float("inf"), -float("inf"), 1.0])
    got = exp_neg_device(x)
    assert math.isnan(got[0])
    assert 0.0 <= got[1] <= EXP_FLOOR and 0.0 <= got[2] <= EXP_FLOOR  # exp(-inf) = 0 up to the clamp
    assert abs(got[3] - math.exp(-0.5)) <= 2 * EPS


# ----------------------------------------------------------------------------------------------- 2. diagonal Gibbs
def diag_inputs(n1, n2, D, seed):
    """Lengthscale ratios up to 1e3 either way, distances that put Q over [0, 700] and past the underflow edge, and rows of x1
    that coincide with columns of x2 (same point, same lengthscales: Q = 0 exactly, K = scale)."""
    g = torch.Generator().manual_seed(seed)
    e1 = torch.exp(torch.empty(D, n1).uniform_(-3.45, 3.45, generator=g))  # 10^(+-1.5)
    e2 = torch.exp(torch.empty(D, n2).uniform_(-3.45, 3.45, generator=g))
    spread1 = torch.exp(torch.empty(n1, 1).uniform_(-4.0, 3.5, generator=g))
    spread2 = torch.exp(torch.empty(n2, 1).uniform_(-4.0, 3.5, generator=g))
    x1 = (torch.rand(n1, D, generator=g) * 2 - 1) * spread1
    x2 = (torch.rand(n2, D, generator=g) * 2 - 1) * spread2
    nc = min(n1, n2) // 3 if min(n1, n2) > 1 else 1
    x1[:nc] = x2[:nc]
    e1[:, :nc] = e2[:, :nc]
    return x1, e1, x2, e2


def diag_reference(x1, e1, x2, e2):
    """Per-pair pieces of scale * GibbsKernel in long double, written as oracle.gibbs_diag_K writes it."""
    a, b = ld(e1).T[:, None, :], ld(e2).T[None, :, :]       # (n1,1,D), (1,n2,D)
    S = a * a + b * b
    dl = ld(x1)[:, None, :] - ld(x2)[None, :, :]
    pref = np.prod(np.sqrt(2 * a * b / S), axis=-1)
    Q = np.sum(dl * dl / S, axis=-1)
    K = LD(SCALE) * pref * np.exp(-Q)
    return dict(a=a, b=b, S=S, dl=dl, pref=pref, Q=Q, K=K)


def check_K(K, r, D):
    K = K.cpu().numpy().astype(LD)
    Kref, Q = r["K"], r["Q"]
    err = np.abs(K - Kref)
    tol = C_PAIR(D) * EPS * (1 + Q) * np.abs(Kref) + SUBNORMAL_SLACK
    tail = Q > 707.0  # argument past the clamp: any value in [0, scale * prefactor * exp(-708)]
    ok = (err <= tol) | (tail & (K >= 0) & (K <= LD(SCALE) * r["pref"] * LD(EXP_FLOOR) * (1 + 1e-12)))
    assert ok.all(), ("K", int((~ok).sum()), float((err / np.maximum(tol, 1e-300)).max()))


def check_reduced(got, ref, scale, D, n_red, what, floor=0.0):
    """|got - ref| <= (c eps + sum rounding) scale + floor; floor: what the pairs past exp_neg's clamp may contribute in
    full (their K is exp(-708) times the prefactor instead of ~0), with the same weights as in scale."""
    got = np.asarray(got.detach().cpu().numpy(), dtype=LD)
    tol = (C_PAIR(D) * EPS + sum_slack(n_red)) * scale + floor + SUBNORMAL_SLACK
    bad = ~(np.abs(got - ref) <= tol)  # a NaN in got or in the reference fails too
    assert not bad.any(), (what, int(bad.sum()), float((np.abs(got - ref) / np.maximum(tol, 1e-300)).max()))


# Forms of the upstream gradient G_ij = rowscale_i T_ij + rowvec_i colvec_j that the backward kernels take: formed in memory,
# composed inside the kernel (the C step's data term), rowscale only, and the rank-one part alone with G = None (the C
# step's -beta alpha^T through the lengthscale field's covariance when the prior term is off).  Values: the keyword
# arguments each form passes.
G_FORMS = dict(formed=("G",), composed=("T", "rowscale", "rowvec", "colvec"), rowscale=("T", "rowscale"),
               rankone=("rowvec", "colvec"))


def g_form_args(how, G, T, rs, rv, cv):
    """Keyword arguments of ops().gibbs_*_bwd for one form of G (CUDA tensors; T goes in the G slot)."""
    t = dict(G=G, T=T, rowscale=rs, rowvec=rv, colvec=cv)
    return {("G" if k == "T" else k): t[k].cuda() for k in G_FORMS[how]}


def g_form_ref(how, T, rs, rv, cv):
    """(G, |G| term by term) in long double for one form.  The formed G is the FP64 rounding of the composed one: the
    C_PAIR eps of the bound covers the difference."""
    T, rs, rv, cv = ld(T), ld(rs), ld(rv), ld(cv)
    if how == "rankone":
        T = 0 * T
    if how == "rowscale":
        rv = 0 * rv
    return (rs[:, None] * T + rv[:, None] * cv[None, :],
            np.abs(rs)[:, None] * np.abs(T) + np.abs(rv)[:, None] * np.abs(cv)[None, :])


DIAG_SHAPES = [(1, 1), (33, 257), (300, 1023), (1, 257)]


@pytest.mark.parametrize("D", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("n1,n2", DIAG_SHAPES)
def test_gibbs_diag_entrywise_every_dimension(D, n1, n2):
    x1, e1, x2, e2 = diag_inputs(n1, n2, D, seed=100 * D + n1 + n2)
    r = diag_reference(x1, e1, x2, e2)
    if n1 * n2 > 1000:  # the problem really spans the exponent range
        Q = r["Q"]
        assert (Q == 0).sum() > 0 and ((Q > 1) & (Q < 100)).any() and ((Q > 100) & (Q < 700)).any() and (Q > 708).any()
    g = torch.Generator().manual_seed(D + n1)
    u = torch.randn(n2, generator=g)
    s = torch.tensor(SCALE, device="cuda")
    K, Ku = ops().gibbs_diag_fwd(x1.cuda(), e1.cuda(), x2.cuda(), e2.cuda(), s, u=u.cuda())
    check_K(K, r, D)
    coincide = (r["Q"] == 0) & (r["pref"] == 1)
    assert (np.abs(K.cpu().numpy()[coincide] - SCALE) <= C_PAIR(D) * EPS * SCALE).all()
    Kw = (1 + r["Q"]) * np.abs(r["K"])                                    # weight of the rounding of each pair
    Kf = np.where(r["Q"] > 700, LD(SCALE) * r["pref"] * LD(EXP_FLOOR), 0)  # pairs past the clamp, in full
    check_reduced(Ku, r["K"] @ ld(u), Kw @ np.abs(ld(u)), D, n2, "K u", floor=Kf @ np.abs(ld(u)))

    # backward: G_ij = rowscale_i T_ij + rowvec_i colvec_j, in each of the forms of G_FORMS
    T, rs, rv, cv = torch.randn(n1, n2, generator=g), torch.randn(n1, generator=g), torch.randn(n1, generator=g), torch.randn(n2, generator=g)
    G = rs[:, None] * T + rv[:, None] * cv[None, :]
    args = (x1.cuda(), e1.cuda(), x2.cuda(), e2.cuda(), s)
    for how in G_FORMS:
        res = ops().gibbs_diag_bwd(*args, **g_form_args(how, G, T, rs, rv, cv), need_dx1=True, need_dx2=True, need_dscale=True)
        want, scale, floor, red = diag_bwd_reference(r, *g_form_ref(how, T, rs, rv, cv))
        for k in want:
            check_reduced(res[k], want[k], scale[k], D, red[k], (how, k), floor=floor[k])


def diag_bwd_reference(r, Gl, Ga):
    """Gradients of sum_ij G_ij K_ij for the pieces r of diag_reference and G = Gl, with check_reduced's rounding scale and
    clamp floor for |G| <= Ga term by term, and the length of each reduction."""
    a, b, S, dl, Kr = r["a"], r["b"], r["S"], r["dl"], r["K"][..., None]
    n1, n2 = r["K"].shape
    # d log K / d l1 = 1/(2 a) - a/S + 2 a dl^2/S^2 (SURVEY Appendix A.4), same for l2 with b; d log K / d x1 = -2 dl / S
    t_a = [1 / (2 * a) + 0 * b, -a / S, 2 * a * dl * dl / (S * S)]
    t_b = [1 / (2 * b) + 0 * a, -b / S, 2 * b * dl * dl / (S * S)]
    dx = -2 * dl / S
    Kw = ((1 + r["Q"]) * np.abs(r["K"]))[..., None]                              # weight of the rounding of each pair
    Kf = np.where(r["Q"] > 700, LD(SCALE) * r["pref"] * LD(EXP_FLOOR), 0)[..., None]  # pairs past the clamp, in full
    want = dict(d_ell1=np.einsum("ij,ijd->di", Gl, Kr * sum(t_a)), d_ell2=np.einsum("ij,ijd->dj", Gl, Kr * sum(t_b)),
                d_x1=np.einsum("ij,ijd->id", Gl, Kr * dx), d_x2=np.einsum("ij,ijd->jd", Gl, -Kr * dx),
                d_scale=np.sum(Gl * r["K"]) / LD(SCALE))
    absd = dict(d_ell1=("ij,ijd->di", sum(np.abs(t) for t in t_a)), d_ell2=("ij,ijd->dj", sum(np.abs(t) for t in t_b)),
                d_x1=("ij,ijd->id", np.abs(dx)), d_x2=("ij,ijd->jd", np.abs(dx)), d_scale=("ij,ijd->", 1 / LD(SCALE)))
    scale = {k: np.einsum(e, Ga, Kw * t) for k, (e, t) in absd.items()}
    floor = {k: np.einsum(e, Ga, Kf * t) for k, (e, t) in absd.items()}
    red = dict(d_ell1=n2, d_x1=n2, d_ell2=n1, d_x2=n1, d_scale=n1 * n2)
    return want, scale, floor, red


# -------------------------------------------------------------------------------------------- 3. full-matrix Gibbs
def rot(d, g):
    q, _ = torch.linalg.qr(torch.randn(d, d, generator=g))
    return q


def full_inputs(n1, n2, d, seed, near_singular):
    """Packed Sigmas.  near_singular: every Sigma shares one rotation R and has eigenvalues (a, ..., a 1e-8 u), so that
    At = S_i + S_j has cond up to ~1e8; otherwise Sigma(h) from a non-diagonal D."""
    g = torch.Generator().manual_seed(seed)
    x1 = torch.rand(n1, d, generator=g) * 2 - 1
    x2 = torch.rand(n2, d, generator=g) * 2 - 1
    if near_singular:
        R = rot(d, g)

        def sig(n):
            lam = torch.exp(torch.empty(n, d).uniform_(-1, 1, generator=g))
            lam[:, -1] *= 1e-8 * (0.5 + torch.rand(n, generator=g))
            return R @ torch.diag_embed(lam) @ R.T
        S1, S2 = sig(n1), sig(n2)
    else:
        Dm = 0.7 * torch.eye(d) + 0.25 * torch.randn(d, d, generator=g)
        Dm = 0.5 * (Dm + Dm.T)  # D o D must be symmetric
        S1 = o.sigma_from_H(torch.randn(n1, d, generator=g), Dm)
        S2 = o.sigma_from_H(torch.randn(n2, d, generator=g), Dm)
        for S in (S1, S2):  # with a non-diagonal D a few draws of h (about 1 in 10^4) give an indefinite Sigma: use others
            pd = torch.linalg.eigvalsh(S)[:, 0] > 0
            S[~pd] = S[pd][:int((~pd).sum())]
    return x1, S1, x2, S2


def _det_inv_ld(A):
    """det and inverse of (..., d, d) long-double matrices, d = 2 or 3, by cofactors (exact to the long double's rounding)."""
    d = A.shape[-1]
    if d == 2:
        det = A[..., 0, 0] * A[..., 1, 1] - A[..., 0, 1] * A[..., 1, 0]
        adj = np.stack([np.stack([A[..., 1, 1], -A[..., 0, 1]], -1), np.stack([-A[..., 1, 0], A[..., 0, 0]], -1)], -2)
    else:
        c = lambda i, j: (A[..., (i + 1) % 3, (j + 1) % 3] * A[..., (i + 2) % 3, (j + 2) % 3]
                          - A[..., (i + 1) % 3, (j + 2) % 3] * A[..., (i + 2) % 3, (j + 1) % 3])
        cof = np.stack([np.stack([c(i, j) for j in range(3)], -1) for i in range(3)], -2)
        det = np.sum(A[..., 0, :] * cof[..., 0, :], -1)
        adj = np.swapaxes(cof, -1, -2)
    return det, adj / det[..., None, None]


def full_reference(x1, S1, x2, S2, jitter):
    """oracle.gibbs_full_K's formulas in long double: prefactor det(S_i)^1/4 det(S_j)^1/4 det(A)^-1/2, Q = dl^T w with
    w = (A + jit I)^-1 dl, A = (S_i + S_j)/2; also A^-1 (no jitter), S_i^-1 and S_j^-1 for the backward."""
    d = x1.shape[1]
    S1l, S2l = ld(S1), ld(S2)
    A = LD(0.5) * (S1l[:, None] + S2l[None, :])
    detA, Ainv = _det_inv_ld(A)
    _, inv = _det_inv_ld(A + LD(jitter) * np.eye(d, dtype=LD))
    det1, S1inv = _det_inv_ld(S1l)
    det2, S2inv = _det_inv_ld(S2l)
    dl = ld(x1)[:, None, :] - ld(x2)[None, :, :]
    w = np.einsum("ijab,ijb->ija", inv, dl)
    Q = np.einsum("ija,ija->ij", dl, w)
    pref = (det1 ** LD(0.25))[:, None] * (det2 ** LD(0.25))[None, :] / np.sqrt(detA)
    At = (S1[:, None] + S2[None, :]).numpy()
    ev = np.linalg.eigvalsh(At)
    cond = ev[..., -1] / ev[..., 0]
    ev1, ev2 = np.linalg.eigvalsh(S1.numpy()), np.linalg.eigvalsh(S2.numpy())
    cond_s = np.maximum((ev1[:, -1] / ev1[:, 0])[:, None], (ev2[:, -1] / ev2[:, 0])[None, :])
    return dict(K=LD(SCALE) * pref * np.exp(-Q), Q=Q, pref=pref, cond=np.maximum(cond, cond_s), w=w, Ainv=Ainv,
                S1inv=S1inv, S2inv=S2inv)


def check_full_K(K, r, d):
    """Closed-form determinant and adjugate: relative error <= c eps cond(At); Q inherits it times (1 + Q)."""
    got = K.cpu().numpy().astype(LD)
    tol = C_PAIR(d) * EPS * r["cond"] * (1 + r["Q"]) * np.abs(r["K"]) + SUBNORMAL_SLACK
    tail = r["Q"] > 707.0
    ok = (np.abs(got - r["K"]) <= tol) | (tail & (got >= 0) & (got <= LD(SCALE) * r["pref"] * LD(EXP_FLOOR) * 1.0001))
    assert ok.all(), (int((~ok).sum()), float((np.abs(got - r["K"]) / tol).max()))


def full_bwd_reference(r, Gl, Ga):
    """Gradients of sum_ij G_ij K_ij for the pieces r of full_reference and G = Gl, as the kernel returns them (entries of
    the symmetric matrix dL/dSigma, packed upper), with g_ij = G_ij K_ij:
        dL/dS_i = sum_j g_ij (1/4 S_i^-1 - 1/4 A_ij^-1 + 1/2 w_ij w_ij^T),  dL/dS_j likewise with S_j^-1,
        dL/dx_i = -2 sum_j g_ij w_ij,  dL/dx_j = 2 sum_i g_ij w_ij,  dL/ds = sum_ij g_ij / s;
    and check_reduced's rounding scale (the same sums of absolute terms with |G| <= Ga and the forward's weight
    cond (1 + Q) |K|) and clamp floor, and the length of each reduction."""
    d = r["w"].shape[-1]
    n1, n2 = r["K"].shape
    iu = np.triu_indices(d)
    pk = lambda M: M[..., iu[0], iu[1]]
    w = r["w"]
    ww, Ai = pk(w[..., :, None] * w[..., None, :]), pk(r["Ainv"])
    s1, s2 = LD(0.25) * pk(r["S1inv"]), LD(0.25) * pk(r["S2inv"])

    def sums(g, pair, s1, s2, w):
        return dict(d_S1=np.einsum("ij,ijp->ip", g, pair) + s1 * g.sum(1)[:, None],
                    d_S2=np.einsum("ij,ijp->jp", g, pair) + s2 * g.sum(0)[:, None],
                    d_x1=-2 * np.einsum("ij,ija->ia", g, w), d_x2=2 * np.einsum("ij,ija->ja", g, w), d_scale=g.sum() / LD(SCALE))

    want = sums(Gl * r["K"], LD(0.5) * ww - LD(0.25) * Ai, s1, s2, w)
    pair_abs = LD(0.5) * np.abs(ww) + LD(0.25) * np.abs(Ai)
    weight = r["cond"] * (1 + r["Q"]) * np.abs(r["K"])
    clamp = np.where(r["Q"] > 700, LD(SCALE) * r["pref"] * LD(EXP_FLOOR), 0)
    scale = {k: np.abs(v) for k, v in sums(Ga * weight, pair_abs, np.abs(s1), np.abs(s2), np.abs(w)).items()}
    floor = {k: np.abs(v) for k, v in sums(Ga * clamp, pair_abs, np.abs(s1), np.abs(s2), np.abs(w)).items()}
    red = dict(d_S1=n2, d_x1=n2, d_S2=n1, d_x2=n1, d_scale=n1 * n2)
    return want, scale, floor, red


def full_case(n1, n2, d, near_singular, seed):
    x1, S1, x2, S2 = full_inputs(n1, n2, d, seed=seed, near_singular=near_singular)
    if near_singular:
        x1 = x1 * 2e-3  # keep Q moderate along the nearly flat direction
        x2 = x2 * 2e-3
    return x1, S1, x2, S2


def full_args(x1, S1, x2, S2, jitter):
    return (x1.cuda(), ops().sym_pack(S1.cuda()), x2.cuda(), ops().sym_pack(S2.cuda()), jitter,
            torch.tensor(SCALE).cuda())


@pytest.mark.parametrize("d", [2, 3])
@pytest.mark.parametrize("near_singular", [False, True])
@pytest.mark.parametrize("jitter", [1e-5, 1e-3, 0.0])
def test_gibbs_full_entrywise_conditioning(d, near_singular, jitter):
    n1, n2 = 65, 300
    x1, S1, x2, S2 = full_case(n1, n2, d, near_singular, seed=10 * d + int(near_singular))
    r = full_reference(x1, S1, x2, S2, jitter)
    if near_singular:
        assert r["cond"].max() > 1e7
    check_full_K(ops().gibbs_full_fwd(*full_args(x1, S1, x2, S2, jitter)), r, d)


def full_bwd_problem(n1, n2, d, near_singular, jitter, seed):
    """full_case with its reference and an upstream gradient (T, rowscale, rowvec, colvec) and its formed G."""
    x1, S1, x2, S2 = full_case(n1, n2, d, near_singular, seed)
    r = full_reference(x1, S1, x2, S2, jitter)
    g = torch.Generator().manual_seed(seed + 1000)
    T, rs, rv, cv = torch.randn(n1, n2, generator=g), torch.randn(n1, generator=g), torch.randn(n1, generator=g), torch.randn(n2, generator=g)
    return (x1, S1, x2, S2), r, (rs[:, None] * T + rv[:, None] * cv[None, :], T, rs, rv, cv)


def check_full_bwd(res, r, how, T, rs, rv, cv, d):
    want, scale, floor, red = full_bwd_reference(r, *g_form_ref(how, T, rs, rv, cv))
    for k in want:
        if res[k] is not None:
            check_reduced(res[k], want[k], scale[k], d, red[k], (how, k), floor=floor[k])


@pytest.mark.parametrize("d", [2, 3])
@pytest.mark.parametrize("near_singular", [False, True])
@pytest.mark.parametrize("jitter,n1,n2", [(1e-5, 65, 300), (1e-3, 65, 300), (0.0, 65, 300), (1e-5, 1, 1), (1e-5, 33, 257)])
def test_gibbs_full_bwd_entrywise(d, near_singular, jitter, n1, n2):
    """All five outputs of the full-matrix backward, every entry at its own scale, for each form of G; the same inputs as
    the forward test above (near-singular Sigmas: cond(At) up to ~1e8)."""
    xs, r, (G, T, rs, rv, cv) = full_bwd_problem(n1, n2, d, near_singular, jitter, seed=10 * d + int(near_singular))
    args = full_args(*xs, jitter)
    for how in G_FORMS:
        res = ops().gibbs_full_bwd(*args, **g_form_args(how, G, T, rs, rv, cv), need_dx1=True, need_dx2=True, need_dscale=True)
        assert all(res[k] is not None for k in ("d_x1", "d_x2", "d_scale"))
        check_full_bwd(res, r, how, T, rs, rv, cv, d)


@pytest.mark.parametrize("d", [2, 3])
def test_gibbs_full_bwd_every_instantiation_and_unaligned_G(d):
    """The four (d_x1, d_x2) instantiations of the kernel, each with and without d_scale (the C step's data term requests
    d_x2 only, and nothing but d_S when the inducing points are frozen); then a formed G that starts 8 bytes past a 16-byte
    boundary, with an odd row length: the launcher has to pick the scalar G loads by itself."""
    n1, n2 = 33, 257
    xs, r, (G, T, rs, rv, cv) = full_bwd_problem(n1, n2, d, False, 1e-5, seed=50 + d)
    args = full_args(*xs, 1e-5)
    for dx1 in (False, True):
        for dx2 in (False, True):
            for dscale in (False, True):
                res = ops().gibbs_full_bwd(*args, **g_form_args("composed", G, T, rs, rv, cv), need_dx1=dx1, need_dx2=dx2,
                                           need_dscale=dscale)
                assert [res[k] is not None for k in ("d_x1", "d_x2", "d_scale")] == [dx1, dx2, dscale]
                check_full_bwd(res, r, "composed", T, rs, rv, cv, d)
    buf = torch.empty(n1 * n2 + 1).cuda()
    Gu = buf[1:].view(n1, n2)
    Gu.copy_(G.cuda())
    assert Gu.data_ptr() % 16 == 8 and Gu.is_contiguous()
    res = ops().gibbs_full_bwd(*args, G=Gu, need_dx1=True, need_dx2=True, need_dscale=True)
    check_full_bwd(res, r, "formed", T, rs, rv, cv, d)


@pytest.mark.parametrize("kind", ["full", "diag"])
def test_gibbs_bwd_aliased_self_pair(kind):
    """The Kzz backward of the C step and of the DSVI layer: K(Z, Z) with one x and one Sigma / lengthscale buffer on both
    sides and one d_Sigma / d_ell and one d_x buffer in both output slots, so that every entry gathers its row and its
    column sums.  M = 1024: the step's 4 column tiles.  The reference is the sum of the two slots' reference gradients."""
    from nonstationary_precip_b200._lib import check, lib, ptr, stream
    M, d, jitter = 1024, 3, 1e-5
    g = torch.Generator().manual_seed(61)
    R = torch.randn(M, M, generator=g)
    G = 0.5 * (R + R.T)
    Gl, Gc = ld(G), G.cuda()
    s = torch.tensor(SCALE, device="cuda")
    ds = torch.zeros((), device="cuda")
    if kind == "full":
        x, S, _, _ = full_inputs(M, 1, d, seed=62, near_singular=False)
        Sp = ops().sym_pack(S.cuda())
        dS, dx = torch.zeros(M, d * (d + 1) // 2, device="cuda"), torch.zeros(M, d, device="cuda")
        xc = x.cuda()
        check(lib().npgp_gibbs_full_bwd(d, M, M, ptr(xc), ptr(Sp), ptr(xc), ptr(Sp), jitter, ptr(s), ptr(Gc), M, None,
                                        None, None, ptr(dS), ptr(dx), ptr(dS), ptr(dx), ptr(ds), stream()), "npgp_gibbs_full_bwd")
        want, scale, floor, _ = full_bwd_reference(full_reference(x, S, x, S, jitter), Gl, np.abs(Gl))
        pairs = dict(d_S=(dS, "d_S1", "d_S2"), d_x=(dx, "d_x1", "d_x2"))
    else:
        x, e, _, _ = diag_inputs(M, 1, d, seed=63)
        xc, ec = x.cuda(), e.cuda()
        de, dx = torch.zeros(d, M, device="cuda"), torch.zeros(M, d, device="cuda")
        check(lib().npgp_gibbs_diag_bwd(d, M, M, ptr(xc), ptr(ec), ptr(xc), ptr(ec), ptr(s), ptr(Gc), M, None, None,
                                        None, ptr(de), ptr(dx), ptr(de), ptr(dx), ptr(ds), stream()), "npgp_gibbs_diag_bwd")
        want, scale, floor, _ = diag_bwd_reference(diag_reference(x, e, x, e), Gl, np.abs(Gl))
        pairs = dict(d_ell=(de, "d_ell1", "d_ell2"), d_x=(dx, "d_x1", "d_x2"))
    for name, (got, a, b) in pairs.items():
        check_reduced(got, want[a] + want[b], scale[a] + scale[b], d, 2 * M, name, floor=floor[a] + floor[b])
    check_reduced(ds, want["d_scale"], scale["d_scale"], d, M * M, "d_scale", floor=floor["d_scale"])


# ---- both Gibbs kernels at the benchmark's shape: several staged chunks of kTI rows per CTA
BENCH_N1, BENCH_N2 = 65536, 1024  # B and M of the 1-GPU benchmark (BASELINE config 2)


def _csrc(name):
    with open(os.path.join(os.path.dirname(__file__), "..", "nonstationary_precip_b200", "csrc", name)) as f:
        return f.read()


def rows_per_cta(n1, col_tiles, waves_target):
    """pick_rows_per_cta of csrc/common.cuh, with its constants read from the source."""
    common = _csrc("common.cuh")
    sms = int(re.search(r"kNumSMs\s*=\s*(\d+)", common).group(1))
    kti = int(re.search(r"kTI\s*=\s*(\d+)", common).group(1))
    row_ctas = -(-sms * waves_target // col_tiles)
    rpc = -(-n1 // row_ctas)
    return max(kti, -(-rpc // kti) * kti), kti


def launch_waves(src):
    """Wave targets (forward, backward) that gibbs_{full,diag}.cu pass to pick_rows_per_cta."""
    waves = [int(w) for w in re.findall(r"pick_rows_per_cta\(n1, col_tiles, (\d+)\)", _csrc(src))]
    assert len(waves) == 2, "expected one forward and one backward launcher"
    return waves


def bench_split(kind, n1, n2):
    """((forward rows per CTA, kTI), (backward rows per CTA, kTI)) of gibbs_{kind}.cu at n1 x n2: both launchers tile the
    columns 256 at a time (128 threads x 2 columns)."""
    return [rows_per_cta(n1, -(-n2 // 256), w) for w in launch_waves("gibbs_%s.cu" % kind)]


def bench_rows(n1, fwd_rpc, bwd_rpc, kti, seed):
    """First and last row of every CTA under both splits, both sides of every chunk boundary inside three CTAs of each
    split (first, middle, last full one), the whole ragged last CTA, and random rows."""
    rows = set()
    for rpc in (fwd_rpc, bwd_rpc):
        starts = list(range(0, n1, rpc))
        for r0 in starts:
            rows |= {r0, min(r0 + rpc, n1) - 1}
        full = [r0 for r0 in starts if r0 + rpc <= n1]
        for r0 in (full[0], full[len(full) // 2], full[-1]):
            for c in range(kti, rpc, kti):
                rows |= {r0 + c - 1, r0 + c}
        rows |= set(range(starts[-1], n1))
    rows |= set(np.random.default_rng(seed).choice(n1, 64, replace=False).tolist())
    return torch.tensor(sorted(rows))


def bench_cols(n2, seed):
    fixed = [0, 1, 254, 255, 256, 257, 511, 512, n2 - 2, n2 - 1]
    rest = np.setdiff1d(np.arange(n2), fixed)
    return torch.tensor(sorted(fixed + np.random.default_rng(seed).choice(rest, 6, replace=False).tolist()))


def check_bench_shape(kind, n1, n2):
    """Forward (K entry by entry on the sampled rows, all columns, and K u) and the backward as the C step calls it
    (composed G, d_x2 and d_scale, no d_x1; then once more with d_x1): row outputs on the sampled rows, whose reference runs
    over the whole row, column outputs on the sampled columns, whose reference runs over all n1 rows, and d_scale against
    an FP64 sum of G o K with the kernel's own K (pinned entry by entry on the sampled rows)."""
    D, jitter = 3, 1e-5
    full = kind == "full"
    g = torch.Generator().manual_seed(7)
    if full:
        x1, S1, x2, S2 = full_inputs(n1, n2, D, seed=81, near_singular=False)
        args = full_args(x1, S1, x2, S2, jitter)
        fwd, bwd = ops().gibbs_full_fwd, ops().gibbs_full_bwd
        ref = lambda rows, cols: full_reference(x1[rows], S1[rows], x2[cols], S2[cols], jitter)
        bwd_ref, check_k = full_bwd_reference, lambda K, r: check_full_K(K, r, D)
        row_keys, col_keys = ("d_S1", "d_x1"), ("d_S2", "d_x2")
        pick = dict(d_S1=lambda t, i: t[i], d_x1=lambda t, i: t[i], d_S2=lambda t, j: t[j], d_x2=lambda t, j: t[j])
    else:
        x1, e1, x2, e2 = diag_inputs(n1, n2, D, seed=82)
        args = (x1.cuda(), e1.cuda(), x2.cuda(), e2.cuda(), torch.tensor(SCALE).cuda())
        fwd, bwd = ops().gibbs_diag_fwd, ops().gibbs_diag_bwd
        ref = lambda rows, cols: diag_reference(x1[rows], e1[:, rows], x2[cols], e2[:, cols])
        bwd_ref, check_k = diag_bwd_reference, lambda K, r: check_K(K, r, D)
        row_keys, col_keys = ("d_ell1", "d_x1"), ("d_ell2", "d_x2")
        pick = dict(d_ell1=lambda t, i: t[:, i], d_x1=lambda t, i: t[i], d_ell2=lambda t, j: t[:, j], d_x2=lambda t, j: t[j])
    (fwd_rpc, kti), (bwd_rpc, _) = bench_split(kind, n1, n2)
    rows, cols = bench_rows(n1, fwd_rpc, bwd_rpc, kti, seed=5), bench_cols(n2, seed=6)
    u = torch.randn(n2, generator=g)
    T, rs, rv, cv = torch.randn(n1, n2, generator=g), torch.randn(n1, generator=g), torch.randn(n1, generator=g), torch.randn(n2, generator=g)

    # forward
    K, Ku = fwd(*args, u=u.cuda())
    rr = ref(rows, torch.arange(n2))
    check_k(K[rows.cuda()], rr)
    weight = (rr["cond"] if full else 1) * (1 + rr["Q"]) * np.abs(rr["K"])
    clamp = np.where(rr["Q"] > 700, LD(SCALE) * rr["pref"] * LD(EXP_FLOOR), 0)
    check_reduced(Ku[rows.cuda()], rr["K"] @ ld(u), weight @ np.abs(ld(u)), D, n2, "K u", floor=clamp @ np.abs(ld(u)))

    # backward, C-step form
    Tc, rsc, rvc, cvc = T.cuda(), rs.cuda(), rv.cuda(), cv.cuda()
    gabs = (rsc.abs()[:, None] * Tc.abs() + rvc.abs()[:, None] * cvc.abs()[None, :]) * K.abs()
    want_ds = ((rsc[:, None] * Tc + rvc[:, None] * cvc[None, :]) * K).sum() / SCALE
    scale_ds = gabs.sum().item() / SCALE
    del gabs
    rc = ref(torch.arange(n1), cols)
    want_r, scale_r, floor_r, red_r = bwd_ref(rr, *g_form_ref("composed", T[rows], rs[rows], rv[rows], cv))
    want_c, scale_c, floor_c, red_c = bwd_ref(rc, *g_form_ref("composed", T[:, cols], rs, rv, cv[cols]))
    for dx1 in (False, True):
        res = bwd(*args, G=Tc, rowscale=rsc, rowvec=rvc, colvec=cvc, need_dx1=dx1, need_dx2=True, need_dscale=True)
        assert (res["d_x1"] is not None) == dx1
        for k in row_keys:
            if res[k] is not None:
                check_reduced(pick[k](res[k], rows.cuda()), want_r[k], scale_r[k], D, red_r[k], ("rows", dx1, k), floor=floor_r[k])
        for k in col_keys:
            check_reduced(pick[k](res[k], cols.cuda()), want_c[k], scale_c[k], D, red_c[k], ("cols", dx1, k), floor=floor_c[k])
        tol = (C_PAIR(D) * EPS + sum_slack(n1 * n2)) * scale_ds
        assert abs(res["d_scale"].item() - want_ds.item()) <= tol, ("d_scale", dx1)


@pytest.mark.parametrize("kind", ["full", "diag"])
def test_gibbs_bench_shape_every_cta_and_chunk(kind):
    """n1 = 65536 rows against n2 = 1024 columns, the shape of the benchmark's step: pick_rows_per_cta gives each CTA 128
    rows in the forward and 224 in the backward, so the chunk loop, the G prefetch queue across chunk boundaries and the
    row reducer's flushes of later chunks all run, and the last backward CTA is ragged.  No smaller test reaches past the
    first chunk."""
    (fwd_rpc, kti), (bwd_rpc, _) = bench_split(kind, BENCH_N1, BENCH_N2)
    assert fwd_rpc > kti and bwd_rpc > kti, "the benchmark's shape no longer runs several chunks per CTA"
    check_bench_shape(kind, BENCH_N1, BENCH_N2)


@pytest.mark.parametrize("d", [2, 3])
def test_gibbs_full_sigma_from_h_off_diagonal_D_gradients(d):
    """Forward and backward through sigma_from_h with a non-diagonal D: the off-diagonal entries of dD are checked too."""
    g = torch.Generator().manual_seed(40 + d)
    n1, n2 = 45, 258
    x1, x2 = torch.rand(n1, d, generator=g) * 2 - 1, torch.rand(n2, d, generator=g) * 2 - 1
    H1, H2 = torch.randn(n1, d, generator=g), torch.randn(n2, d, generator=g)
    Dm = 0.8 * torch.eye(d) + 0.2 * torch.randn(d, d, generator=g)
    Dm = 0.5 * (Dm + Dm.T)
    s = torch.tensor(SCALE)
    G = torch.randn(n1, n2, generator=g)
    c = [t.clone().requires_grad_(True) for t in (x1, H1, x2, H2, Dm, s)]
    Kc = c[5] * o.gibbs_full_K(c[0], c[2], o.sigma_from_H(c[1], c[4]), o.sigma_from_H(c[3], c[4]))
    (Kc * G).sum().backward()
    gg = [t.clone().cuda().requires_grad_(True) for t in (x1, H1, x2, H2, Dm, s)]
    Kg = ops().gibbs_full(gg[0], ops().sigma_from_h(gg[1], gg[4]), gg[2], ops().sigma_from_h(gg[3], gg[4]), gg[5])
    (Kg * G.cuda()).sum().backward()
    assert ((Kg.detach().cpu() - Kc.detach()).abs() <= 1e-13 * Kc.detach().abs()).all()
    for name, a, b in zip(("x1", "H1", "x2", "H2", "scale"), gg[:4] + gg[5:], c[:4] + c[5:]):
        assert (a.grad.cpu() - b.grad).abs().max() <= 1e-9 * b.grad.abs().max(), name
    off = ~torch.eye(d, dtype=torch.bool)
    assert (c[4].grad[off].abs() > 1e-3 * c[4].grad.abs().max()).all()  # the off-diagonal dD is exercised
    assert ((gg[4].grad.cpu() - c[4].grad).abs() <= 1e-9 * c[4].grad.abs()).all()  # entry by entry


# ------------------------------------------------------------------------------------------------ 4. digit emitters
def _digits_bound_check(K, digits, n, M):
    from test_digits_gpu import decode_planes
    e = math.frexp(SCALE * 1.0000000001)[1]
    Kd = decode_planes(digits, n, M) * 2.0 ** (e - 54)
    assert (Kd[:n] - K).abs().max().item() <= 2.0 ** (e - 55) + 4e-16
    assert (Kd[n:] == 0).all()


@pytest.mark.parametrize("D", [1, 2, 3, 4, 5, 6])
def test_gibbs_diag_digits_every_dimension(D):
    n, M = 300, 256
    x1, e1, x2, e2 = diag_inputs(n, M, D, seed=7 + D)
    u = torch.randn(M, generator=torch.Generator().manual_seed(D))
    s = torch.tensor([SCALE], device="cuda")
    args = [t.cuda() for t in (x1, e1, x2, e2)]
    K, Ku = ops().gibbs_diag_fwd(*args, s, u=u.cuda())
    digits = torch.empty(ops().digits_bytes(n, M, 128), dtype=torch.uint8, device="cuda")
    parts = torch.full((ops().gibbs_digits_splits(n, M), n), float("nan"), device="cuda")
    ops().gibbs_diag_fwd_digits(*args, s, digits, u=u.cuda(), Ku_part=parts)
    _digits_bound_check(K, digits, n, M)
    assert ((parts.sum(0) - Ku).abs() <= 1e-13 * (K.abs() @ u.cuda().abs())).all()


@pytest.mark.parametrize("d", [2, 3])
def test_gibbs_full_digits_off_diagonal_D(d):
    n, M = 200, 128
    x1, S1, x2, S2 = full_inputs(n, M, d, seed=70 + d, near_singular=False)
    s = torch.tensor([SCALE], device="cuda")
    args = [x1.cuda(), ops().sym_pack(S1.cuda()), x2.cuda(), ops().sym_pack(S2.cuda())]
    K = ops().gibbs_full_fwd(*args, 1e-5, s)
    digits = torch.empty(ops().digits_bytes(n, M, 128), dtype=torch.uint8, device="cuda")
    ops().gibbs_full_fwd_digits(*args, 1e-5, s, digits)
    _digits_bound_check(K, digits, n, M)


# ------------------------------------------------------------------------------------------ 5. field interpolation
FIELD_CONFIGS = [(1, 1, 1), (2, 1, 1), (3, 1, 1), (3, 2, 1), (4, 4, 1), (5, 5, 1), (6, 6, 1)]


def field_reference(x, z, lam, os_, V, bias):
    xs = ld(x)[None, :, None, :] / ld(lam)[:, None, None, :]   # (nb, n, 1, d)
    zs = ld(z)[None, None, :, :] / ld(lam)[:, None, None, :]   # (nb, 1, m, d)
    df = xs - zs
    Q = LD(0.5) * np.sum(df * df, -1)                          # (nb, n, m)
    Qabs = LD(0.5) * np.sum((np.abs(xs) + np.abs(zs)) ** 2, -1)  # the pre-scaled difference cancels: its rounding scale
    k = ld(os_)[:, None, None] * np.exp(-Q)
    return dict(Q=Q, Qabs=Qabs, k=k, df=df, out=ld(bias)[:, None, None] + k @ ld(V))


@pytest.mark.parametrize("d,nb,nv", FIELD_CONFIGS)
@pytest.mark.parametrize("n,m", [(77, 203), (300, 1000)])
def test_field_every_dispatched_configuration(d, nb, nv, n, m):
    g = torch.Generator().manual_seed(n + m + 10 * d + nb)
    x, z = torch.rand(n, d, generator=g) * 2 - 1, torch.rand(m, d, generator=g) * 2 - 1
    x[:5] = z[:5]  # coincident points: k = os exactly
    lam, os_ = 0.3 + torch.rand(nb, d, generator=g), 0.5 + torch.rand(nb, generator=g)
    V, bias, W = torch.randn(nb, m, nv, generator=g), torch.randn(nb, generator=g), torch.randn(nb, n, nv, generator=g)
    r = field_reference(x, z, lam, os_, V, bias)
    c = C_PAIR(d)
    kscale = (np.abs(r["k"]) + ld(os_)[:, None, None] * LD(EXP_FLOOR)) * (1 + r["Qabs"])
    fscale = kscale @ np.abs(ld(V)) + np.abs(ld(bias))[:, None, None]
    args = (x.cuda(), z.cuda(), lam.cuda(), os_.cuda(), V.cuda())
    out = ops().rbf_matvec_fwd(*args, bias=bias.cuda())
    check_reduced(out, r["out"], fscale, d, m, "out")
    out_e = ops().rbf_matvec_fwd(*args, bias=bias.cuda(), apply_exp=True).cpu().numpy().astype(LD)
    tol_e = np.exp(r["out"]) * ((c * EPS + sum_slack(m)) * fscale + 4 * EPS)
    assert (np.abs(out_e - np.exp(r["out"])) <= tol_e).all()
    dV, dz = ops().rbf_matvec_bwd(*args, W.cuda())
    Wl = ld(W)
    want_dV = np.einsum("bnm,bnc->bmc", r["k"], Wl)
    check_reduced(dV, want_dV, np.einsum("bnm,bnc->bmc", kscale, np.abs(Wl)), d, n, "dV")
    # dz_ja = sum_b sum_i sum_c W_bic V_bjc k_bij (x_ia - z_ja) / lam_ba^2
    gv = np.einsum("bnc,bmc->bnm", Wl, ld(V))
    il = 1 / ld(lam)[:, None, None, :]
    want_dz = np.einsum("bnm,bnmd->md", gv * r["k"], r["df"] * il)
    gva = np.einsum("bnc,bmc->bnm", np.abs(Wl), np.abs(ld(V)))
    scale_dz = np.einsum("bnm,bnmd->md", gva * kscale, (np.abs(r["df"]) + np.sqrt(2 * r["Qabs"])[..., None]) * il)
    check_reduced(dz, want_dz, scale_dz, d, n * nb, "dz")


# ------------------------------------------------------------------------------------------------------- 6. DSVI
def dsvi_problem(n, M, d, seed):
    g = torch.Generator().manual_seed(seed)
    span = {1: 10.0, 3: 1.0, 6: 1.0}[d]
    Z = (torch.rand(M, d, generator=g) * 2 - 1) * span
    if d == 1:  # a jittered grid: random points on a line come too close for a well-conditioned Kzz
        Z = torch.linspace(-span, span, M).unsqueeze(1) + 0.02 * span / M * torch.randn(M, 1, generator=g)
    X = (torch.rand(n, d, generator=g) * 2 - 1) * span
    # lengthscale below the typical inducing-point spacing: Kzz well conditioned, so the two Cholesky routes agree to ~1e-12
    ls = torch.full((d,), {1: 0.08, 3: 0.15, 6: 0.3}[d]) * (0.8 + 0.4 * torch.rand(d, generator=g))
    os_ = torch.tensor([0.9])
    m = 0.5 * torch.randn(M, generator=g)
    Ls = 0.7 * torch.eye(M) + 0.05 * torch.tril(torch.randn(M, M, generator=g))
    return X, Z, ls, os_, m, Ls


@pytest.mark.parametrize("d", [1, 3, 6])
@pytest.mark.parametrize("n,M", [(700, 98), (4100, 128)])
def test_dsvi_layer_every_dimension(d, n, M):
    """M even but not a multiple of 64 (FP64 row-quadratic path) and M = 128 with n >= 4096 (int8 T = K C and SYRK)."""
    X, Z, ls, os_, m, Ls = dsvi_problem(n, M, d, seed=d + M)
    Kzz = o.rbf_ard_K(Z, Z, ls, os_) + 1e-6 * torch.eye(M)
    assert torch.linalg.cond(Kzz) < 1e3, "test problem must be well conditioned"
    g = torch.Generator().manual_seed(3)
    a, b = torch.randn(n, generator=g), torch.randn(n, generator=g)
    c = [t.clone().requires_grad_(True) for t in (X, Z, ls, os_, m, Ls)]
    mo, vo = o.dgp_layer_marginals(c[0], c[1], c[4], c[5], c[3], c[2], jitter_zz=1e-6)
    ((mo * a).sum() + (vo * b).sum()).backward()
    gg = [t.clone().cuda().requires_grad_(True) for t in (X, Z, ls, os_, m, Ls)]
    mg, vg, info = ops().dsvi_layer(*gg, jitter=1e-6)
    assert int(info) == 0
    ((mg * a.cuda()).sum() + (vg * b.cuda()).sum()).backward()
    rel = lambda p, q: ((p.detach().cpu() - q.detach()).abs().max() / q.detach().abs().max()).item()
    assert rel(mg, mo) < 1e-10 and rel(vg, vo) < 1e-10
    for name, p, q in zip(("X", "Z", "ls", "os", "m", "Ls"), gg, c):
        want = torch.tril(q.grad) if name == "Ls" else q.grad
        assert rel(p.grad, want) < 1e-10, name


# ------------------------------------------------------------------------------------------- 7. SVGP variant 0
def variant0_problem(d, B, M, seed, device="cuda"):
    """make_problem's diagonal variant at any d (it reads x[:, 1], so it cannot build d = 1); the lengthscale grows with d
    so that K(x, Z) is not negligible in 6 dimensions, and in 1-D the inducing points sit on a jittered grid over a wider
    domain so that Kzz stays well conditioned."""
    g = torch.Generator().manual_seed(173 + seed)
    span = 8.0 if d == 1 else 1.0
    ell0 = 0.1 if d == 1 else 0.3 * math.sqrt(d / 2)
    x = (torch.rand(B, d, generator=g) * 2 - 1) * span
    y = torch.sin(3 * x[:, 0] / span) + 0.5 * torch.cos(5 * x[:, -1] / span) + 0.1 * torch.randn(B, generator=g)
    Z = (torch.rand(M, d, generator=g) * 2 - 1) * span
    if d == 1:  # a jittered grid: random points on a line come too close for a well-conditioned Kzz
        Z = torch.linspace(-span, span, M).unsqueeze(1) + 0.1 * span / M * torch.randn(M, 1, generator=g)
    m = 0.3 * torch.randn(M, generator=g)
    Ls = torch.eye(M) * 0.8 + 0.05 * torch.tril(torch.randn(M, M, generator=g))
    kw = dict(m=m, Ls=Ls, outputscale=0.644, noise=0.011,
              log_ell_z=math.log(ell0) + 0.1 * torch.randn(d, M, generator=g), prior_c=torch.full((d,), math.log(ell0)),
              prior_os=torch.ones(d), prior_lam=torch.full((d, d), 1.3))
    mv = lambda t: t.to(device) if torch.is_tensor(t) else t
    return mv(x), mv(y), mv(Z), {k: mv(v) for k, v in kw.items()}, 4 * B


@pytest.mark.parametrize("d", [1, 4, 6])
def test_svgp_variant0_every_dimension(d):
    import sys
    import os
    sys.path.insert(0, os.path.dirname(__file__))
    from svgp_cases import oracle_loss_and_grads
    from nonstationary_precip_b200.svgp import SVGPGibbs
    B, M = 400, 128
    x, y, Z, p, N = variant0_problem(d, B, M, seed=d)
    mc, mp = SVGPGibbs("diag", Z, N, **p), SVGPGibbs("diag", Z, N, **p)
    mc.use_c_engine()
    lc, lp = mc.loss_and_grad(x, y), mp.loss_and_grad(x, y)
    assert int(mc.last["info"]) == 0 and mc.check_status() == 0
    want_loss, want = oracle_loss_and_grads("diag", x, y, Z, p, N)
    rel = lambda a, b: ((a.detach().cpu() - b.detach().cpu()).abs().max() / b.detach().cpu().abs().max().clamp_min(1e-300)).item()
    assert abs(lc.item() - want_loss.item()) < 1e-9 * abs(want_loss.item())
    assert abs(lc.item() - lp.item()) < 1e-8 * abs(lp.item())
    for name, gw in want.items():
        assert rel(mc.g[name], gw) < 1e-6, name
        assert rel(mp.g[name], gw) < 1e-6, name
    # prediction against the oracle, then one draw
    from test_svgp_predict_gpu import oracle_predict
    xs = variant0_problem(d, 300, M, seed=d + 50)[0]
    r = mc.predictive(xs)
    mean_o, var_o = oracle_predict(mc, xs, p)
    assert rel(r.mean, mean_o) <= 1e-8 and rel(r.var, var_o) <= 1e-8
    draws = mc.sample(xs, 8, seed=5)
    assert draws.shape == (8, 300) and torch.isfinite(draws).all()


# -------------------------------------------------------------------------------------------- 8. NaN and Inf
NAN_ROW, NAN_DIM = 17, 0


def _with_nan(x):
    y = x.clone()
    y[NAN_ROW, NAN_DIM] = float("nan")
    return y


def _rows_nan_others_equal(a, b, row_dim=0, rtol=None):
    """Row NAN_ROW of a is NaN throughout; every other row equals b bitwise, or, for sums that FP64 atomics add in a
    run-dependent order (rtol given), to rtol times the largest entry."""
    a, b = a.movedim(row_dim, 0).cpu(), b.movedim(row_dim, 0).cpu()
    keep = torch.ones(a.shape[0], dtype=torch.bool)
    keep[NAN_ROW] = False
    assert torch.isnan(a[NAN_ROW]).all(), "the row with the missing coordinate must be NaN throughout"
    if rtol is None:
        assert torch.equal(a[keep], b[keep]), "every other row must be bitwise unchanged"
    else:
        assert ((a[keep] - b[keep]).abs() <= rtol * b[keep].abs().max()).all(), "every other row must be unchanged"


@pytest.mark.parametrize("D", [1, 3, 6])
def test_nan_coordinate_poisons_its_row_diag(D):
    x1, e1, x2, e2 = diag_inputs(60, 256, D, seed=D)
    s = torch.tensor([SCALE], device="cuda")
    u = torch.randn(256, device="cuda")
    K0, Ku0 = ops().gibbs_diag_fwd(x1.cuda(), e1.cuda(), x2.cuda(), e2.cuda(), s, u=u)
    K1, Ku1 = ops().gibbs_diag_fwd(_with_nan(x1).cuda(), e1.cuda(), x2.cuda(), e2.cuda(), s, u=u)
    _rows_nan_others_equal(K1, K0)
    _rows_nan_others_equal(Ku1, Ku0, rtol=1e-14)
    # the digit path: a NaN has no fixed-point digits, but the fused K u partials of that row are NaN (the predictive mean,
    # hence the loss, goes NaN) and no other row changes
    n, M = 60, 256
    outs = []
    for xx in (x1, _with_nan(x1)):
        digits = torch.empty(ops().digits_bytes(n, M, 128), dtype=torch.uint8, device="cuda")
        parts = torch.empty(ops().gibbs_digits_splits(n, M), n, device="cuda")
        ops().gibbs_diag_fwd_digits(xx.cuda(), e1.cuda(), x2.cuda(), e2.cuda(), s, digits, u=u, Ku_part=parts)
        from test_digits_gpu import decode_planes
        outs.append((decode_planes(digits, n, M)[:n], parts))
    _rows_nan_others_equal(outs[1][1], outs[0][1], row_dim=1)
    keep = torch.ones(n, dtype=torch.bool)
    keep[NAN_ROW] = False
    assert torch.equal(outs[1][0][keep.cuda()], outs[0][0][keep.cuda()])


@pytest.mark.parametrize("d", [2, 3])
def test_nan_coordinate_poisons_its_row_full(d):
    x1, S1, x2, S2 = full_inputs(60, 128, d, seed=d, near_singular=False)
    s = torch.tensor([SCALE], device="cuda")
    S1p, S2p = ops().sym_pack(S1.cuda()), ops().sym_pack(S2.cuda())
    K0 = ops().gibbs_full_fwd(x1.cuda(), S1p, x2.cuda(), S2p, 1e-5, s)
    K1 = ops().gibbs_full_fwd(_with_nan(x1).cuda(), S1p, x2.cuda(), S2p, 1e-5, s)
    _rows_nan_others_equal(K1, K0)


def test_nan_coordinate_poisons_its_row_field_and_dsvi():
    g = torch.Generator().manual_seed(9)
    for d, nb in ((2, 1), (3, 3), (6, 6)):
        x, z = torch.rand(60, d, generator=g), torch.rand(203, d, generator=g)
        lam, os_ = 0.5 + torch.rand(nb, d, generator=g), torch.ones(nb)
        V, bias = torch.randn(nb, 203, 1, generator=g), torch.randn(nb, generator=g)
        args = lambda xx: (xx.cuda(), z.cuda(), lam.cuda(), os_.cuda(), V.cuda())
        for apply_exp in (False, True):  # ell(x) = exp(c + ...): a NaN must not come out as a lengthscale
            o0 = ops().rbf_matvec_fwd(*args(x), bias=bias.cuda(), apply_exp=apply_exp)
            o1 = ops().rbf_matvec_fwd(*args(_with_nan(x)), bias=bias.cuda(), apply_exp=apply_exp)
            _rows_nan_others_equal(o1, o0, row_dim=1)
    X, Z, ls, os_, m, Ls = dsvi_problem(300, 98, 3, seed=1)
    r0 = ops().dsvi_layer(*[t.cuda() for t in (X, Z, ls, os_, m, Ls)])
    r1 = ops().dsvi_layer(*[t.cuda() for t in (_with_nan(X), Z, ls, os_, m, Ls)])
    _rows_nan_others_equal(r1[0], r0[0], rtol=1e-14)
    _rows_nan_others_equal(r1[1], r0[1], rtol=1e-14)


def test_nan_row_norm_gives_nan_sgpr_variance():
    n = 300
    g = torch.Generator().manual_seed(4)
    qn = (0.1 * torch.rand(3, n, generator=g)).cuda()
    qv = (0.01 * torch.rand(2, n, generator=g)).cuda()
    s, noise, os_t = (torch.tensor([v], device="cuda") for v in (0.644, 0.01, 0.5))
    qn1 = qn.clone()
    qn1[2, NAN_ROW] = float("nan")   # a Gibbs block
    qn1[0, NAN_ROW + 1] = float("nan")  # the temporal block
    v0 = ops().sgpr_predict_finish(qn, 1, qv, s, noise, torch.empty(n, device="cuda"), os_t=os_t)
    v1 = ops().sgpr_predict_finish(qn1, 1, qv, s, noise, torch.empty(n, device="cuda"), os_t=os_t)
    want = (0.5 - qn[0]).clamp_min(0) + 0.644 * (1 - qn[1] - qn[2]).clamp_min(0) + qv.sum(0)
    assert ((v0 - want).abs() <= 4 * EPS * want.abs()).all()
    assert torch.isnan(v1[NAN_ROW]) and torch.isnan(v1[NAN_ROW + 1])
    keep = torch.ones(n, dtype=torch.bool, device="cuda")
    keep[NAN_ROW:NAN_ROW + 2] = False
    assert torch.equal(v1[keep], v0[keep])


def test_nan_coordinate_stops_the_guarded_c_step():
    from nonstationary_precip_b200.svgp import SVGPGibbs
    x, y, Z, p, N = variant0_problem(3, 512, 128, seed=11)
    mc = SVGPGibbs("diag", Z, N, **p)
    mc.use_c_engine()
    mc.train_step(x, y, lr=0.01)
    assert mc.check_status() == 0
    before = [t.clone() for t in (mc.theta, mc.adam_m, mc.adam_v, mc.step_dev)]
    mc.train_step(_with_nan(x), y, lr=0.01)
    assert mc.check_status() & 2, "a NaN in the data must set the non-finite-loss bit"
    for t, b in zip((mc.theta, mc.adam_m, mc.adam_v, mc.step_dev), before):
        assert torch.equal(t, b)


def test_infinite_coordinate_gives_zero_covariance():
    """A point at +-inf against finite points: K = 0 (exp(-inf)), as the reference gives, up to exp_neg's clamp."""
    for D in (1, 3, 6):
        x1, e1, x2, e2 = diag_inputs(40, 128, D, seed=D + 20)
        x1[3, 0], x1[5, D - 1] = float("inf"), -float("inf")
        K = ops().gibbs_diag_fwd(x1.cuda(), e1.cuda(), x2.cuda(), e2.cuda(), torch.tensor([SCALE], device="cuda")).cpu()
        assert torch.isfinite(K).all()
        assert (K[[3, 5]] >= 0).all() and (K[[3, 5]] <= SCALE * EXP_FLOOR).all()
    x, z = torch.rand(40, 3), torch.rand(203, 3)
    x[3, 1] = float("inf")
    V, bias = torch.randn(3, 203, 1), torch.randn(3)
    out = ops().rbf_matvec_fwd(x.cuda(), z.cuda(), torch.ones(3, 3, device="cuda"), torch.ones(3, device="cuda"), V.cuda(),
                               bias=bias.cuda()).cpu()
    assert ((out[:, 3, 0] - bias).abs() <= V.abs().sum(1)[:, 0] * EXP_FLOOR).all()
