"""Digit-plane path of the SVGP step (csrc/gibbs_digits.cu + csrc/oz8.cu): the Gibbs kernels emitted as 7-byte fixed-point
digits, the row-quadratic product and the MN-major SYRK that consume them, the deterministic partial reductions.
Checked against the FP64 tile kernels / FP64 products and, through them, the oracle (test_ops_gpu.py pins those)."""
import math
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))
from oz8_ref import decode_planes, encode_a_planes, encode_b_planes  # noqa: E402

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


def gibbs_inputs(variant, n, M, d, seed):
    from nonstationary_precip_b200 import ops
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(n, d, generator=g) * 2 - 1).cuda()
    z = (torch.rand(M, d, generator=g) * 2 - 1).cuda()
    if variant == "diag":
        f1 = torch.exp(0.3 * torch.randn(d, n, generator=g) - 1.0).cuda()
        f2 = torch.exp(0.3 * torch.randn(d, M, generator=g) - 1.0).cuda()
    else:
        Dm = torch.diag(0.8 + torch.rand(d, generator=g)).cuda()
        f1 = ops.sigma_from_h_fwd(torch.randn(n, d, generator=g).cuda(), Dm)
        f2 = ops.sigma_from_h_fwd(torch.randn(M, d, generator=g).cuda(), Dm)
    s = torch.tensor([0.644], device="cuda")
    u = torch.randn(M, generator=g).cuda()
    return x, f1, z, f2, s, u


def fwd_both(variant, x, f1, z, f2, s, u):
    from nonstationary_precip_b200 import ops
    n, M = x.shape[0], z.shape[0]
    digits = torch.empty(ops.digits_bytes(n, M, 128), dtype=torch.uint8, device="cuda")
    parts = torch.full((ops.gibbs_digits_splits(n, M), n), float("nan"), device="cuda")
    if variant == "diag":
        K, Ku = ops.gibbs_diag_fwd(x, f1, z, f2, s, u=u)
        ops.gibbs_diag_fwd_digits(x, f1, z, f2, s, digits, u=u, Ku_part=parts)
    else:
        K, Ku = ops.gibbs_full_fwd(x, f1, z, f2, 1e-5, s, u=u)
        ops.gibbs_full_fwd_digits(x, f1, z, f2, 1e-5, s, digits, u=u, Ku_part=parts)
    return K, Ku, digits, parts


@pytest.mark.parametrize("variant,n,M,d", [("full", 1, 128, 3), ("full", 300, 128, 2), ("full", 1000, 256, 3),
                                            ("diag", 129, 128, 3), ("diag", 777, 384, 2), ("full", 4100, 1024, 3)])
def test_gibbs_digits_equal_fp64_kernel(variant, n, M, d):
    x, f1, z, f2, s, u = gibbs_inputs(variant, n, M, d, seed=n + M)
    K, Ku, digits, parts = fwd_both(variant, x, f1, z, f2, s, u)
    e = math.frexp(0.644 * 1.0000000001)[1]
    Kd = decode_planes(digits, n, M) * 2.0 ** (e - 54)
    # fixed point with 54 fractional bits below 2^e: absolute error <= 2^(e-55) (+ the two kernels' own last-bit differences)
    assert (Kd[:n] - K).abs().max().item() <= 2.0 ** (e - 55) + 4e-16
    assert (Kd[n:] == 0).all()  # padded rows: zero digits (they enter the SYRK's contraction)
    assert ((parts.sum(0) - Ku).abs().max() / Ku.abs().max()).item() < 1e-13


@pytest.mark.parametrize("variant,n,M", [("full", 300, 128), ("full", 4100, 1024), ("diag", 2000, 256)])
def test_rowquad_and_syrk_from_digits(variant, n, M):
    from nonstationary_precip_b200 import ops
    x, f1, z, f2, s, u = gibbs_inputs(variant, n, M, 3, seed=7 * n + M)
    K, Ku, digits, parts = fwd_both(variant, x, f1, z, f2, s, u)
    g = torch.Generator().manual_seed(3)
    A = torch.randn(M, M, generator=g).cuda()
    C = A @ A.T / M - 0.3 * torch.eye(M, device="cuda")
    C = 0.5 * (C + C.T)
    gvec = torch.randn(n, generator=g).cuda()
    Cd = torch.empty(ops.digits_bytes(M, M, 64), dtype=torch.uint8, device="cuda")
    cexp = torch.empty(M, dtype=torch.int32, device="cuda")
    ops.o8_slice_rows(C, 64, Cd, cexp)
    T = torch.full((n, M), float("nan"), device="cuda")
    q_part = torch.full((M // 64, n), float("nan"), device="cuda")
    du_part = torch.full(((n + 127) // 128, M), float("nan"), device="cuda")
    ops.o8_rowquad_digits(n, M, digits, s, Cd, cexp, T, q_part=q_part, gvec=gvec, du_part=du_part)
    # The tensor cores contract the fixed-point K held in the planes: compare against that operand (decoded on the host side;
    # test_gibbs_digits_equal_fp64_kernel pins it to the FP64 kernel within the plane quantum), so the only differences left are
    # the FP64 roundings of the reference products (~sqrt(M) eps |K||C|) and the final rounding of the exact integer sums.
    e = math.frexp(0.644 * 1.0000000001)[1]
    K = decode_planes(digits, n, M)[:n] * 2.0 ** (e - 54)
    scale = K.abs() @ C.abs()
    # digit products with p + q >= 7 are dropped: <= 6 * 2^-54 * 2^(e + f_j) per contraction entry with random signs (balanced
    # digits): sigma = sqrt(6 M) / 3 in that unit; the bound below is > 10 sigma (2^f_j <= 2 max_k |C_kj|)
    trunc = 16 * math.sqrt(M) * 2.0 ** -54 * 2.0 ** e * 2 * C.abs().max(0).values[None, :]
    T0, q0 = ops.rowquad(K, C)
    assert ((T - T0).abs() <= 1e-14 * scale + trunc).all()
    q_bound = 1e-14 * (scale * K.abs()).sum(1) + (trunc * K.abs()).sum(1) + 2.0 ** -52 * T0.abs().sum(1)
    assert ((q_part.sum(0) - q0).abs() <= q_bound).all()
    du = ops.o8_sum_partials(du_part)
    assert ((du - K.T @ gvec).abs() <= 1e-14 * (K.abs().T @ gvec.abs())).all()
    # deterministic: a second run is bitwise identical
    T2, q2, du2 = torch.empty_like(T), torch.empty_like(q_part), torch.empty_like(du_part)
    ops.o8_rowquad_digits(n, M, digits, s, Cd, cexp, T2, q_part=q2, gvec=gvec, du_part=du2)
    assert torch.equal(T, T2) and torch.equal(q_part, q2) and torch.equal(du_part, du2)
    # SYRK from the same planes, read MN-major
    part = torch.empty(max(1, ops.o8_syrk_part_bytes(n, M) // 8), device="cuda")
    w0 = torch.tensor([-0.37], device="cuda")
    got = ops.o8_syrk_digits(n, M, digits, s, part, w0=w0, alpha=2.0)
    want = -0.74 * (K.T @ K)
    syrk_bound = 0.74 * (1e-14 * (K.abs().T @ K.abs()) + 16 * math.sqrt(n) * 2.0 ** -54 * 4.0 ** e)
    assert ((got - want).abs() <= syrk_bound).all()
    assert torch.equal(got, got.T)
    assert torch.equal(got, ops.o8_syrk_digits(n, M, digits, s, part, w0=w0, alpha=2.0))
    # rows of weight zero are taken out again
    skip = torch.tensor([5, n - 1, n // 2], dtype=torch.int32, device="cuda")[:min(3, n)]
    cnt = torch.tensor([skip.numel()], dtype=torch.int32, device="cuda")
    rows = torch.zeros(n, dtype=torch.int32, device="cuda")
    rows[:skip.numel()] = skip
    got2 = ops.o8_syrk_digits(n, M, digits, s, part, w0=w0, alpha=2.0, skip_count=cnt, skip_rows=rows)
    wv = torch.ones(n, device="cuda")
    wv[skip.long()] = 0.0
    want2 = -0.74 * (K.T @ (wv[:, None] * K))
    assert ((got2 - want2).abs() <= syrk_bound).all()


def test_non_finite_input_poisons_the_row_not_the_digits():
    """ADVICE r1: the slicer turned NaN / Inf into finite digits.  Now the row's exponent is marked and the result is NaN."""
    from nonstationary_precip_b200 import ops
    g = torch.Generator().manual_seed(2)
    K = torch.rand(300, 128, generator=g).cuda()
    C = torch.eye(128, device="cuda")
    K[17, 5] = float("nan")
    K[40, 9] = float("inf")
    T, q = ops.rowquad_i8(K, C)
    assert torch.isnan(T[17]).all() and torch.isnan(T[40]).all()
    ok = torch.ones(300, dtype=torch.bool, device="cuda")
    ok[17] = ok[40] = False
    assert torch.isfinite(T[ok]).all() and (T[ok] - K[ok]).abs().max().item() < 1e-15
    S = ops.syrk_i8(K)
    assert torch.isnan(S[5]).all() and torch.isnan(S[:, 9]).all()


def test_gauss_ell_parts_matches_atomic_version_and_lists_clamped_rows():
    from nonstationary_precip_b200 import ops
    g = torch.Generator().manual_seed(4)
    n = 5000
    y, mu = torch.randn(n, generator=g).cuda(), torch.randn(n, generator=g).cuda()
    q_part = (0.01 * torch.randn(16, n, generator=g)).cuda()
    q_part[:, 123] = -10.0  # forces v < min_var: clamped
    q_part[:, 4000] = -10.0
    s, noise = torch.tensor([0.644], device="cuda"), torch.tensor([0.0111], device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    rows = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    acc, gmu, gv, var = ops.gauss_ell_parts(y, mu, q_part, s, noise, wscale=1.0 / n, want_var=True, skip_count=cnt, skip_rows=rows)
    acc0, gmu0, gv0, var0 = ops.gauss_ell(y, mu, q_part.sum(0), s, noise, wscale=1.0 / n, want_var=True)
    assert ((acc[:3] - acc0).abs() / acc0.abs()).max().item() < 1e-13
    assert torch.allclose(gmu, gmu0, rtol=1e-15, atol=0) and torch.equal(gv, gv0) and torch.allclose(var, var0, rtol=1e-14)
    assert abs(acc[3].item() - (-0.5 / n / 0.0111)) < 1e-18
    assert int(cnt) == 2 and sorted(rows[:2].tolist()) == [123, 4000]
    acc2, *_ = ops.gauss_ell_parts(y, mu, q_part, s, noise, wscale=1.0 / n)
    assert torch.equal(acc, acc2)  # two-stage reductions: bitwise reproducible


@pytest.mark.parametrize("variant", ["full", "diag"])
def test_svgp_step_with_clamped_rows_matches_dmma_path(variant):
    """A clamped predictive variance (gradient zero for that row) goes through the skip list of the int8 SYRK."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from svgp_cases import make_problem
    from nonstationary_precip_b200.svgp import SVGPGibbs
    x, y, Z, p, N = make_problem(variant, device="cuda", B=600, M=128, d=3, seed=31)
    p["Ls"] = 1e-4 * torch.eye(128, device="cuda")  # S ~ 0: the whitened variance s - k^T Kzz^-1 k goes (numerically) negative
    outs = []
    for impl in ("dmma", "i8"):
        # a NEGATIVE diagonal jitter pushes the variance of the rows closest to the inducing points below min_variance:
        # 248 of 600 rows (full) / 260 of 600 (diag) clamp (counted with the CPU emulator)
        model = SVGPGibbs(variant, Z, N, jitter_xx=-0.01 if variant == "full" else -0.1, **p)
        model.rowquad_impl = impl
        loss = model.loss_and_grad(x, y)
        outs.append((loss.item(), model.grad.clone(), model))
    (l0, g0, m0), (l1, g1, m1) = outs
    n_clamped = int(m1._i8_bufs[600]["skip_count"])
    assert 100 < n_clamped < 500, "test problem must clamp some rows and keep some"
    assert abs(l0 - l1) < 1e-10 * abs(l0)
    assert (g0 - g1).abs().max().item() < 1e-7 * g0.abs().max().item()


# ---- digit-level diagnostics: hand-made planes, exact integer reference ----------------------------------------------
@pytest.mark.parametrize("n,M", [(128, 64), (256, 128)])
def test_every_digit_product_is_exact(n, M):
    """A carries only digit p, C only digit q: T must be exactly 2^(-12-8(p+q)) A_p C_q^T for the 28 kept products and 0 for
    the dropped ones; then all digits at once against the integer sum.  Isolates a wrong product / accumulator / hazard."""
    from nonstationary_precip_b200 import ops
    g = torch.Generator().manual_seed(n + M)
    DA = torch.randint(-128, 128, (7, n, M), generator=g, dtype=torch.int8)
    DC = torch.randint(-128, 128, (7, M, M), generator=g, dtype=torch.int8)
    ea = torch.zeros(n, dtype=torch.int32, device="cuda")
    ec = torch.zeros(M, dtype=torch.int32, device="cuda")
    T = torch.empty(n, M, device="cuda")
    bad = []
    for p in range(7):
        for q in range(7):
            A1, C1 = torch.zeros_like(DA), torch.zeros_like(DC)
            A1[p], C1[q] = DA[p], DC[q]
            ops.o8_rowquad_digits(n, M, encode_a_planes(A1).cuda(), None, encode_b_planes(C1).cuda(), ec, T, a_expo=ea)
            want = (DA[p].long() @ DC[q].long().T).double() * 2.0 ** (-12 - 8 * (p + q)) if p + q <= 6 else torch.zeros(n, M)
            if not torch.equal(T.cpu(), want):
                bad.append((p, q, (T.cpu() - want).abs().max().item() / max(want.abs().max().item(), 1e-300)))
    assert not bad, bad
    ops.o8_rowquad_digits(n, M, encode_a_planes(DA).cuda(), None, encode_b_planes(DC).cuda(), ec, T, a_expo=ea)
    want = torch.zeros(n, M)
    for p in range(7):
        for q in range(7 - p):
            want += (DA[p].long() @ DC[q].long().T).double() * 2.0 ** (-12 - 8 * (p + q))
    assert ((T.cpu() - want).abs().max() / want.abs().max()).item() < 1e-15
