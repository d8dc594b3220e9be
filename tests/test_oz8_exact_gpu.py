"""The int8 digit contractions of csrc/oz8.cu against their exact integer arithmetic (tests/oz8_ref.py), bit for bit.

T = K C (npgp_o8_rowquad_digits), T = A B^T (npgp_o8_gemm_digits) and the digit SYRK K^T K (npgp_o8_syrk_digits) compute
integer digit products exactly and round once per recombination, so their outputs are fully specified: the reference
recomputes every G_t with exact FP64 GEMMs, recombines and scales it as the epilogue does and, for the SYRK, adds the
per-segment partials in the finishing kernel's order over the same work split (ported from O8SegIter / o8_syrk_shape).
The FP64 sums formed by the kernels in their own order (row dot, column sums, triangular row norms) are checked against
the bitwise-exact T with gamma_k bounds on the sums of absolute terms.  The slicers must decode to rint(x 2^(54 - e))."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))
import oz8_ref as R  # noqa: E402

pytestmark = pytest.mark.gpu
torch.set_default_dtype(torch.float64)


def ops():
    from nonstationary_precip_b200 import ops as o
    return o


def scaled_rows(n, M, g, spread=40):
    """FP64 rows of random sign and magnitude with row maxima spread over 2^+-spread (per-row exponents differ)."""
    K = torch.randn(n, M, generator=g, dtype=torch.float64)
    K *= torch.pow(2.0, torch.randint(-spread, spread + 1, (n, 1), generator=g).double())
    return K.cuda()


def symmetric(M, g):
    A = torch.randn(M, M, generator=g, dtype=torch.float64)
    d = torch.pow(2.0, torch.randint(-6, 7, (M,), generator=g).double())
    C = d[:, None] * (A + A.T) * d[None, :]
    return C.cuda()


def slice_rows(X, block_rows):
    o = ops()
    R_, Kd = X.shape
    buf = torch.empty(o.digits_bytes(R_, Kd, block_rows), dtype=torch.uint8, device="cuda")
    ex = torch.empty((R_ + block_rows - 1) // block_rows * block_rows, dtype=torch.int32, device="cuda")
    o.o8_slice_rows(X, block_rows, buf, ex)
    return buf, ex


def decoded(buf, ex, rows, Kd, block_rows):
    """The FP64 values the planes hold: y 2^(e - 54) (exact)."""
    D = R.a_digits(buf, rows, Kd) if block_rows == 128 else R.b_digits(buf, rows, Kd)
    return R.digits_value(D[:, :rows]).double() * R.scale_or_nan(ex[:rows], -R.FRAC)[:, None]


# ---- T = K C and the row dot / column sums ----------------------------------------------------------------------------
ROWS = [1, 127, 129, 148 * 128, 148 * 128 + 1, 65536, 65536 + 37]
COLS = [64, 192, 1024, 2048]


@pytest.mark.parametrize("M", COLS)
@pytest.mark.parametrize("n", ROWS)
def test_rowquad_T_is_bitwise_the_exact_recombination(n, M):
    """Per-row exponents (o8_slice_rows): T bitwise; q partials, du partials against T within gamma bounds; the q-only pass
    (T NULL) gives bitwise the q of the T pass."""
    o = ops()
    g = torch.Generator().manual_seed(n * 7 + M)
    K, C = scaled_rows(n, M, g), symmetric(M, g)
    gvec = torch.randn(n, generator=g, dtype=torch.float64).cuda()
    As, ea = slice_rows(K, 128)
    Cs, ec = slice_rows(C, 64)
    T = torch.full((n, M), float("nan"), device="cuda")
    q = torch.full((M // 64, n), float("nan"), device="cuda")
    du = torch.full(((n + 127) // 128, M), float("nan"), device="cuda")
    o.o8_rowquad_digits(n, M, As, None, Cs, ec, T, q_part=q, gvec=gvec, du_part=du, a_expo=ea)
    want = R.gemm_reference(R.a_digits(As, n, M)[:, :n], ea[:n], R.b_digits(Cs, M, M), ec)
    assert torch.equal(T, want), (T - want).abs().max().item()
    Kq = decoded(As, ea, n, M, 128)  # the K the kernel rebuilds from the planes for the row dot
    TK = (T * Kq).view(n, M // 64, 64)
    q_ref = TK.sum(-1).T
    # kernel: two fma chains of 32 and one add (gamma_33); reference: 64 products and their sum (gamma_65)
    assert ((q - q_ref).abs() <= (R.gamma(33) + R.gamma(65)) * TK.abs().sum(-1).T).all()
    q2 = torch.full_like(q, float("nan"))
    o.o8_rowquad_digits(n, M, As, None, Cs, ec, None, q_part=q2, a_expo=ea)
    assert torch.equal(q, q2)
    npad = (n + 127) // 128 * 128
    gK = torch.zeros(npad, M, device="cuda")
    gK[:n] = gvec[:, None] * Kq
    gK = gK.view(npad // 128, 128, M)
    # kernel: two fma chains of 64 and one add (gamma_65); reference: 128 products and their sum (gamma_129)
    assert ((du - gK.sum(1)).abs() <= (R.gamma(65) + R.gamma(129)) * gK.abs().sum(1)).all()


@pytest.mark.parametrize("n,M", [(129, 192), (148 * 128 + 1, 1024), (65536 + 37, 1024)])
def test_rowquad_matrix_wide_scale_of_the_gibbs_digits(n, M):
    """A from the Gibbs digit kernel (one exponent for the matrix, from the device scalar outputscale)."""
    o = ops()
    g = torch.Generator().manual_seed(n + M)
    x = (torch.rand(n, 3, generator=g, dtype=torch.float64) * 2 - 1).cuda()
    z = (torch.rand(M, 3, generator=g, dtype=torch.float64) * 2 - 1).cuda()
    f1 = torch.exp(0.3 * torch.randn(3, n, generator=g, dtype=torch.float64) - 1.0).cuda()
    f2 = torch.exp(0.3 * torch.randn(3, M, generator=g, dtype=torch.float64) - 1.0).cuda()
    s = torch.tensor([0.644], dtype=torch.float64, device="cuda")
    As = torch.empty(o.digits_bytes(n, M, 128), dtype=torch.uint8, device="cuda")
    o.gibbs_diag_fwd_digits(x, f1, z, f2, s, As)
    Cs, ec = slice_rows(symmetric(M, g), 64)
    T = torch.full((n, M), float("nan"), device="cuda")
    q = torch.full((M // 64, n), float("nan"), device="cuda")
    o.o8_rowquad_digits(n, M, As, s, Cs, ec, T, q_part=q)
    e = R.exponent_of_scale(0.644)
    ea = torch.full((n,), e, dtype=torch.int32, device="cuda")
    assert torch.equal(T, R.gemm_reference(R.a_digits(As, n, M)[:, :n], ea, R.b_digits(Cs, M, M), ec))
    q2 = torch.full_like(q, float("nan"))
    o.o8_rowquad_digits(n, M, As, s, Cs, ec, None, q_part=q2)
    assert torch.equal(q, q2)


@pytest.mark.parametrize("n,N,Kd", [(1, 64, 2048), (129, 2048, 64), (148 * 128 + 1, 192, 1024), (65536 + 37, 64, 192),
                                    (300, 1024, 16384)])
def test_gemm_digits_bitwise(n, N, Kd):
    o = ops()
    g = torch.Generator().manual_seed(n + N + Kd)
    As, ea = slice_rows(scaled_rows(n, Kd, g), 128)
    Bs, eb = slice_rows(scaled_rows(N, Kd, g, spread=8), 64)
    T = torch.full((n, N), float("nan"), device="cuda")
    o.o8_gemm_digits(n, N, Kd, As, None, Bs, eb, T, a_expo=ea)
    assert torch.equal(T, R.gemm_reference(R.a_digits(As, n, Kd)[:, :n], ea[:n], R.b_digits(Bs, N, Kd), eb))


@pytest.mark.parametrize("da,db", [(-128, -128), (127, 127), (-128, 127)])
def test_worst_case_digits_over_16384_long_contractions(da, db):
    """Every digit at its extreme over Kd = 16384: |G_6| = 7 * 16384 * 2^14 = 0.875 * 2^31 (all -128).  Both entry points,
    T = A B^T (N != Kd) and T = K C (N = Kd = 16384), must still be the exact recombination."""
    o = ops()
    Kd, n, N = 16384, 256, 128
    ea = torch.zeros(n, dtype=torch.int32, device="cuda")
    eb = torch.zeros(Kd, dtype=torch.int32, device="cuda")
    As = torch.full((o.digits_bytes(n, Kd, 128),), da & 0xFF, dtype=torch.uint8, device="cuda")  # constant planes
    DA = torch.full((7, 1, Kd), da, dtype=torch.int8, device="cuda")
    DB = torch.full((7, 64, Kd), db, dtype=torch.int8, device="cuda")
    G = R.digit_products(DA, DB)
    assert G.abs().max().item() == 7 * Kd * abs(da * db)
    want_row = R.gemm_reference(DA, ea[:1], DB, eb[:64])[0, 0].item()
    Bs = torch.full((o.digits_bytes(N, Kd, 64),), db & 0xFF, dtype=torch.uint8, device="cuda")
    T = torch.full((n, N), float("nan"), device="cuda")
    o.o8_gemm_digits(n, N, Kd, As, None, Bs, eb, T, a_expo=ea)
    assert (T == want_row).all(), (T - want_row).abs().max().item()
    Cs = torch.full((o.digits_bytes(Kd, Kd, 64),), db & 0xFF, dtype=torch.uint8, device="cuda")
    T = torch.full((n, Kd), float("nan"), device="cuda")
    o.o8_rowquad_digits(n, Kd, As, None, Cs, eb, T, a_expo=ea)
    assert (T == want_row).all(), (T - want_row).abs().max().item()


@pytest.mark.parametrize("n,Kd,Ms", [(129, 1024, 0), (148 * 128 + 1, 1024, 384), (1000, 2048, 1536)])
def test_trinorm_against_the_exact_product(n, Kd, Ms):
    """Row norms over column blocks of A L^T, L lower triangular (block diagonal split at Ms): the kernel skips the zero
    k-steps, the reference contracts over all of them."""
    o = ops()
    g = torch.Generator().manual_seed(n + Kd + Ms)
    L = torch.tril(torch.randn(Kd, Kd, generator=g, dtype=torch.float64))
    if Ms:
        L[Ms:, :Ms] = 0.0
    As, ea = slice_rows(scaled_rows(n, Kd, g), 128)
    Ls, el = slice_rows(L.cuda(), 64)
    q = torch.full((Kd // 64, n), float("nan"), device="cuda")
    o.o8_trinorm_digits(n, Kd, Kd, As, None, Ls, el, q, Ms=Ms, a_expo=ea)
    T = R.gemm_reference(R.a_digits(As, n, Kd)[:, :n], ea[:n], R.b_digits(Ls, Kd, Kd), el)
    T2 = (T * T).view(n, Kd // 64, 64).sum(-1).T
    # T of the kernel is bitwise T of the reference; both sum 64 squares (gamma_64 each, the squares included)
    assert ((q - T2).abs() <= 2 * R.gamma(65) * T2).all()


# ---- the digit SYRK, bitwise over its work split --------------------------------------------------------------------
def random_planes(n, M, g, fill=None):
    """(7, npad, M) int8 digits (random, or all `fill`) with zero padded rows, and their A-type planes."""
    npad = (n + 127) // 128 * 128
    if fill is None:
        D = torch.randint(-128, 128, (7, npad, M), generator=g, dtype=torch.int8).cuda()
    else:
        D = torch.full((7, npad, M), fill, dtype=torch.int8, device="cuda")
    D[:, n:] = 0
    return D, R.encode_a_planes(D)


def plan_case(plan):
    """The situations of the work split a plan exercises."""
    nt, nks, spc, G, full = plan["n_tiles"], plan["nks"], plan["spc"], plan["n_cta"], plan["full"]
    rem = plan["n_items"] - full * G
    per_item, crosses, phantom_idle = {}, False, False
    totalB = rem * spc
    LB = -(-totalB // G) if totalB else 0
    for c in range(G):
        segs = R.cta_segments(nt, nks, spc, c, G)[full:]
        items = {(t, k0 // spc) for t, k0, _ in segs}
        crosses |= len(items) > 1
        for it in items:
            per_item[it] = per_item.get(it, 0) + 1
        phantom_idle |= min(c * LB + LB, totalB) > c * LB and not segs
    return dict(few=plan["n_items"] < R.NUM_SMS, no_remainder=plan["n_items"] >= R.NUM_SMS and rem == 0,
                spread3=max(per_item.values(), default=0) >= 3, crosses=crosses, phantom_idle=phantom_idle,
                full_chunk=spc == R.MAX_SEG)


SYRK_CASES = [  # (n, M, digits, situation the shape must produce)
    (4100, 1024, None, "few"),
    (1, 128, None, "few"),
    (119168, 128, None, "no_remainder"),
    (30000, 1024, None, "spread3"),
    (30000, 1024, None, "crosses"),
    (21760, 1024, None, "phantom_idle"),
    (120832, 128, None, "phantom_idle"),
    (65536, 1024, "gibbs", "spread3"),
    (16384, 4096, -128, "full_chunk"),
    (16384 + 128, 4096, 127, "crosses"),
]


@pytest.mark.parametrize("n,M,fill,case", SYRK_CASES)
def test_syrk_digits_bitwise_over_its_work_split(n, M, fill, case):
    o = ops()
    plan = R.syrk_plan(n, M)
    assert plan_case(plan)[case], (case, plan_case(plan))
    assert o.o8_syrk_part_bytes(n, M) == plan["n_cta"] * plan["slots"] * 128 * 64 * 8  # the ported shape is the library's
    g = torch.Generator().manual_seed(n + M)
    if fill == "gibbs":
        x = (torch.rand(n, 3, generator=g, dtype=torch.float64) * 2 - 1).cuda()
        z = (torch.rand(M, 3, generator=g, dtype=torch.float64) * 2 - 1).cuda()
        f1 = torch.exp(0.3 * torch.randn(3, n, generator=g, dtype=torch.float64) - 1.0).cuda()
        f2 = torch.exp(0.3 * torch.randn(3, M, generator=g, dtype=torch.float64) - 1.0).cuda()
        scale = 0.644
        planes = torch.empty(o.digits_bytes(n, M, 128), dtype=torch.uint8, device="cuda")
        o.gibbs_diag_fwd_digits(x, f1, z, f2, torch.tensor([scale], device="cuda"), planes)
        D = R.a_digits(planes, n, M)
    else:
        scale = 1.0
        D, planes = random_planes(n, M, g, fill)
    s = torch.tensor([scale], dtype=torch.float64, device="cuda")
    part = torch.empty(o.o8_syrk_part_bytes(n, M) // 8, dtype=torch.float64, device="cuda")
    w0 = torch.tensor([-0.37], dtype=torch.float64, device="cuda")
    got = o.o8_syrk_digits(n, M, planes, s, part, w0=w0, alpha=2.0)
    want = R.syrk_reference(D, R.exponent_of_scale(scale), plan, M, alpha=2.0, w0=-0.37)
    assert torch.equal(got, want), (got - want).abs().max().item()


# ---- rows of weight zero ---------------------------------------------------------------------------------------------
def run_skip(n, M, planes, s, part, rows):
    rows = torch.as_tensor(rows, dtype=torch.int32).cuda()
    cnt = torch.tensor([rows.numel()], dtype=torch.int32, device="cuda")
    buf = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    buf[:rows.numel()] = rows
    return ops().o8_syrk_digits(n, M, planes, s, part, alpha=0.5, skip_count=cnt, skip_rows=buf)


@pytest.mark.parametrize("n,M,which", [(30000, 1024, "edges"), (30000, 256, "half"), (4100, 1024, "half")])
def test_syrk_skip_rows_exact_and_independent_of_list_order(n, M, which):
    """The correction is the exact sum of the listed rows' digit products: bitwise the reference, and the same bits for
    any order of the list (the SVGP step fills it through atomics)."""
    o = ops()
    plan = R.syrk_plan(n, M)
    g = torch.Generator().manual_seed(n + M + len(which))
    D, planes = random_planes(n, M, g)
    s = torch.tensor([1.0], dtype=torch.float64, device="cuda")
    part = torch.empty(o.o8_syrk_part_bytes(n, M) // 8, dtype=torch.float64, device="cuda")
    if which == "edges":  # chunk edges, row-block edges, first and last rows
        cuts = [32 * k for k in range(plan["spc"], plan["nks"], plan["spc"])]
        rows = sorted({r for c in cuts + [128, 256, 128 * (n // 128)] for r in (c - 1, c) if 0 <= r < n} | {0, n - 1})
    else:
        rows = torch.randperm(n, generator=g)[:n // 2].sort().values.tolist()
    got = run_skip(n, M, planes, s, part, rows)
    perm = [rows[i] for i in torch.randperm(len(rows), generator=g).tolist()]
    again = run_skip(n, M, planes, s, part, perm)
    assert torch.equal(got, again), (got - again).abs().max().item()
    want = R.syrk_reference(D, R.exponent_of_scale(1.0), plan, M, alpha=0.5, skip=rows)
    assert torch.equal(got, want), (got - want).abs().max().item()


def test_clamped_rows_of_gauss_ell_parts_give_the_same_syrk_in_any_order():
    """gauss_ell_parts appends clamped rows through atomicAdd; the SYRK over its list and over the sorted list agree bitwise."""
    o = ops()
    n, M = 20000, 512
    g = torch.Generator().manual_seed(11)
    D, planes = random_planes(n, M, g)
    y, mu = torch.randn(n, generator=g).cuda(), torch.randn(n, generator=g).cuda()
    q_part = (0.01 * torch.randn(8, n, generator=g)).cuda()
    clamp = torch.rand(n, generator=g) < 0.4
    q_part[:, clamp.cuda()] = -10.0
    kd, noise = torch.tensor([0.644], device="cuda"), torch.tensor([0.0111], device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    rows = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    o.gauss_ell_parts(y, mu, q_part, kd, noise, wscale=1.0 / n, skip_count=cnt, skip_rows=rows)
    k = int(cnt)
    assert k == int(clamp.sum())
    s = torch.tensor([1.0], dtype=torch.float64, device="cuda")
    part = torch.empty(o.o8_syrk_part_bytes(n, M) // 8, dtype=torch.float64, device="cuda")
    got = o.o8_syrk_digits(n, M, planes, s, part, skip_count=cnt, skip_rows=rows)
    srt = rows.clone()
    srt[:k] = rows[:k].sort().values
    rev = srt.clone()
    rev[:k] = srt[:k].flip(0)
    for other in (srt, rev):
        again = o.o8_syrk_digits(n, M, planes, s, part, skip_count=cnt, skip_rows=other)
        assert torch.equal(got, again), (got - again).abs().max().item()
    want = R.syrk_reference(D, R.exponent_of_scale(1.0), R.syrk_plan(n, M), M, skip=srt[:k].tolist())
    assert torch.equal(got, want)


# ---- slicers ---------------------------------------------------------------------------------------------------------
def edge_rows(R_, Kd, g):
    """Rows of every kind the slicers treat specially, then random rows of spread exponents."""
    X = torch.randn(R_, Kd, generator=g, dtype=torch.float64)
    X *= torch.pow(2.0, torch.randint(-60, 61, (R_, 1), generator=g).double())
    X[0] = 0.0                                                       # all zero
    X[1, 3] = 4.0                                                    # row maximum an exact power of two
    X[1] = X[1].clamp(-4.0, 4.0)
    X[2] = -X[2].abs()                                               # negative only, maximum at a power of two
    X[2, -1] = -2.0 ** -20
    X[2] = X[2].clamp(min=-2.0 ** -20)
    X[3] = torch.randn(Kd, generator=g, dtype=torch.float64) * 2.0 ** -1060   # subnormal
    X[4] = torch.randn(Kd, generator=g, dtype=torch.float64) * 2.0 ** -980    # normal, below 2^-961: exponent clamps
    X[5, 1] = float("nan")
    X[6, Kd - 1] = float("-inf")
    X[7] = torch.where(torch.arange(Kd) % 2 == 0, 2.0 ** 1000, -(2.0 ** -1000))  # huge and tiny in one row
    return X


def check_sliced(X, D, ex, pad_rows):
    """D (7, rows, Kd) digits, ex exponents of the first rows of X: y = rint(x 2^(54 - e)), poisoned rows zero, padding
    zero; rows clamped at EMIN keep the absolute bound 2^(EMIN - 55)."""
    R_ = X.shape[0]
    m = X.abs().max(1).values
    e = torch.frexp(m)[1].to(torch.int64)
    e = torch.where(m > 0, e, torch.zeros_like(e)).clamp(min=R.EMIN)
    poison = ~torch.isfinite(X).all(1)
    e = torch.where(poison, torch.full_like(e, R.POISON), e)
    assert torch.equal(ex[:R_].to(torch.int64), e)
    y = R.digits_value(D)
    ok = ~poison
    want = torch.round(X[ok] * R.pow2(R.FRAC - e[ok])[:, None])
    assert torch.equal(y[:R_][ok].double(), want)  # |y| <= 2^54 and y is x scaled: exact as a double
    assert (y[:R_][poison] == 0).all()
    assert (D[:, R_:R_ + pad_rows] == 0).all()
    tiny = ok & (e == R.EMIN)
    if tiny.any():
        back = y[:R_][tiny].double() * 2.0 ** (R.EMIN - R.FRAC)
        assert ((back - X[tiny]).abs() <= 2.0 ** (R.EMIN - 55)).all()


@pytest.mark.parametrize("block_rows", [128, 64])
@pytest.mark.parametrize("R_,Kd", [(37, 32), (200, 16384), (1000, 96)])
def test_slice_rows_decodes_to_the_rounded_fixed_point(R_, Kd, block_rows):
    g = torch.Generator().manual_seed(R_ + Kd + block_rows)
    X = edge_rows(R_, Kd, g).cuda()
    buf, ex = slice_rows(X, block_rows)
    rpad = (R_ + block_rows - 1) // block_rows * block_rows
    D = R.a_digits(buf, R_, Kd) if block_rows == 128 else R.b_digits(buf, R_, Kd)
    check_sliced(X, D, ex, rpad - R_)
    assert (ex[R_:] == 0).all()


@pytest.mark.parametrize("n,M", [(33, 256), (16384 + 37, 128)])
def test_slice_t_decodes_to_the_rounded_fixed_point(n, M):
    """The transposed slicer of npgp_syrk_i8 (per-column exponents), read back from the workspace."""
    o = ops()
    g = torch.Generator().manual_seed(n + M)
    X = edge_rows(M, n, g).T.contiguous().cuda()   # column j of X = row j of the edge cases
    ws = o.I8Workspace()
    o.syrk_i8(X, workspace=ws)
    torch.cuda.synchronize()
    buf = ws._bufs[("syrk", n, M)]
    npad = (n + 127) // 128 * 128
    D = R.a_digits(buf, M, npad)                    # operand rows = columns of X, contraction along the rows of X
    ex = buf[npad * M * 7 + 8 * M:].view(torch.int32)[:M]
    check_sliced(X.T.contiguous(), D[:, :, :n], ex, 0)
    assert (D[:, :, n:] == 0).all()
