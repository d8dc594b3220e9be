"""Exact reference of the byte-digit int8 contractions (csrc/oz8.cuh, csrc/oz8.cu), shared by the digit-plane tests.

An operand entry is y = rint(x 2^(54-e)) = sum_p a_p 2^(48-8p), seven signed digits a_p.  The kernels form, per output entry,
G_t = sum_{p+q=t} (A_p B_q^T) for t = 0..6 exactly in int32, recombine hi = G_0 2^24 + G_1 2^16 + G_2 2^8 + G_3 and
lo = G_4 2^16 + G_5 2^8 + G_6 as 64-bit integers into fma(double(lo), 2^-24, double(hi)) (o8_recombine), then apply
power-of-two scales.  Everything here reproduces that arithmetic operation by operation: the G_t come from FP64 GEMMs, which
are exact because every partial sum is an integer below 7 * 16384 * 2^14 < 2^53, and fma(lo, 2^-24, hi) is the plain sum
double(hi) + double(lo) 2^-24 since the product by 2^-24 is exact."""
import torch

NS = 7          # digits per entry
POISON = 1 << 20
EMIN = -960
FRAC = 54
NUM_SMS = 148   # kNumSMs of csrc/common.cuh: the SYRK's work split does not depend on the card
MAX_SEG = 512   # O8_MAX_SEG of csrc/oz8.cu


# ---- plane layouts (csrc/oz8.cuh) ------------------------------------------------------------------------------------
def decode_planes(digits, n, M):
    """Inverse of the A-type row layout of csrc/oz8.cuh: int8 planes -> integer-valued double matrix (npad, M), without the
    power-of-two scale.  Layout: [row block][digit][k-step][16-byte half][8-row group][row in group][16 bytes]."""
    npad = (n + 127) // 128 * 128
    nks = M // 32
    d = digits[:npad * M * 7].view(torch.int8).view(npad // 128, 7, nks, 2, 16, 8, 16).to(torch.int64)
    y = d[:, 0]
    for p in range(1, 7):
        y = y * 256 + d[:, p]  # seven signed digits
    # y: [rb, ks, cj, m8, r8, k16] -> rows rb*128 + m8*8 + r8, cols ks*32 + cj*16 + k16
    return y.permute(0, 3, 4, 1, 2, 5).reshape(npad, M).double()


def encode_a_planes(D):
    """D: (7, npad, M) int8 digits -> uint8 buffer in the A-type row layout [rb][p][ks][cj][m8][r8][k16]."""
    _, npad, M = D.shape
    nks = M // 32
    t = D.view(7, npad // 128, 16, 8, nks, 2, 16)      # [p, rb, m8, r8, ks, cj, k16]
    return t.permute(1, 0, 4, 5, 2, 3, 6).contiguous().view(torch.uint8).reshape(-1)


def encode_b_planes(D):
    """D: (7, Mr, Kd) int8 digits of the B operand (row blocks of 64) -> [cb][ks][p][cj][m8][r8][k16]."""
    _, Mr, Kd = D.shape
    nks = Kd // 32
    t = D.view(7, Mr // 64, 8, 8, nks, 2, 16)          # [p, cb, m8, r8, ks, cj, k16]
    return t.permute(1, 4, 0, 5, 2, 3, 6).contiguous().view(torch.uint8).reshape(-1)


def a_digits(buf, rows, Kd):
    """A-type planes (block rows 128) -> (7, rows padded to 128, Kd) int8 digit tensor (inverse of encode_a_planes)."""
    npad = (rows + 127) // 128 * 128
    nks = Kd // 32
    t = buf[:npad * Kd * 7].view(torch.int8).view(npad // 128, 7, nks, 2, 16, 8, 16)  # [rb, p, ks, cj, m8, r8, k16]
    return t.permute(1, 0, 4, 5, 2, 3, 6).reshape(7, npad, Kd)


def b_digits(buf, rows, Kd):
    """B-type planes (block rows 64) -> (7, rows padded to 64, Kd) int8 digit tensor (inverse of encode_b_planes)."""
    rpad = (rows + 63) // 64 * 64
    nks = Kd // 32
    t = buf[:rpad * Kd * 7].view(torch.int8).view(rpad // 64, nks, 7, 2, 8, 8, 16)   # [cb, ks, p, cj, m8, r8, k16]
    return t.permute(2, 0, 4, 5, 1, 3, 6).reshape(7, rpad, Kd)


def digits_value(D):
    """(7, R, K) digits -> the integers y = sum_p a_p 256^(6-p) (int64)."""
    y = D[0].to(torch.int64)
    for p in range(1, NS):
        y = y * 256 + D[p].to(torch.int64)
    return y


# ---- exact arithmetic ------------------------------------------------------------------------------------------------
def pow2(k):
    """2^k (int64 tensor, normal range) as an exactly built double tensor."""
    return ((k.to(torch.int64) + 1023) << 52).view(torch.float64)


def scale_or_nan(e, shift):
    """o8_scale_or_nan: 2^(e + shift), NaN for a poisoned exponent."""
    e = e.to(torch.int64)
    bad = e == POISON
    out = pow2(torch.where(bad, torch.zeros_like(e), e + shift))
    return torch.where(bad, torch.full_like(out, float("nan")), out)


def exponent_of_scale(s):
    """o8_exponent_of_scale of a positive Python float."""
    import math
    if not (s > 0.0) or not (s < 1.7e308):
        return POISON
    return max(math.frexp(s * 1.0000000001)[1], EMIN)


def digit_products(DA, DB):
    """G (7, m, n) float64 (exact integers): G_t = sum_{p+q=t} A_p B_q^T over the contraction, DA (7, m, K), DB (7, n, K)."""
    A = DA.to(torch.float64)
    B = DB.to(torch.float64)
    G = torch.empty(NS, A.shape[1], B.shape[1], dtype=torch.float64, device=A.device)
    for t in range(NS):
        # one GEMM per t over the concatenated contraction: every partial sum stays below 7 K 2^14 < 2^53
        G[t] = torch.cat([A[p] for p in range(t + 1)], 1) @ torch.cat([B[t - p] for p in range(t + 1)], 1).T
    return G


def recombine(G):
    """o8_recombine of exact G_t (any float / int tensor holding integers with |G_t| < 2^31 * n_sums): double per entry."""
    g = G.to(torch.int64)
    hi = ((g[0] * 256 + g[1]) * 256 + g[2]) * 256 + g[3]
    lo = (g[4] * 256 + g[5]) * 256 + g[6]
    return hi.double() + lo.double() * 2.0 ** -24


def gemm_reference(DA, ea, DB, eb, row_block=4096):
    """T = A B^T as o8_rowquad_kernel stores it: recombine(G) * 2^(e_i - 36) * 2^(f_j), in that order.  DA (7, n, K) with
    per-row exponents ea (n,), DB (7, N, K) with per-row exponents eb (N,).  Row blocks bound the memory."""
    n = DA.shape[1]
    sc = scale_or_nan(eb, 0)[None, :]
    out = torch.empty(n, DB.shape[1], dtype=torch.float64, device=DA.device)
    for i0 in range(0, n, row_block):
        i1 = min(n, i0 + row_block)
        v = recombine(digit_products(DA[:, i0:i1], DB))
        out[i0:i1] = v * scale_or_nan(ea[i0:i1], -36)[:, None] * sc
    return out


def gamma(k):
    u = 2.0 ** -53
    return k * u / (1 - k * u)


# ---- the SYRK's work split (O8SegIter and o8_syrk_shape of csrc/oz8.cu, ported line by line) --------------------------
def cdiv(a, b):
    return (a + b - 1) // b


def syrk_tiles(M):
    n_rb, n_cb = M // 128, M // 64
    return n_rb * n_cb - n_rb * (n_rb - 1)


def tile_rc(tl, M):
    n_cb = M // 64
    rb = 0
    while tl >= n_cb - 2 * rb:
        tl -= n_cb - 2 * rb
        rb += 1
    return rb, 2 * rb + tl


def cta_segments(n_tiles, nks, spc, cta, n_cta):
    """The segments (tile, k0, k1) CTA `cta` produces, in order (O8SegIter.next)."""
    n_chunks = cdiv(nks, spc)
    n_items = n_tiles * n_chunks
    full = n_items // n_cta
    out = []
    for wave in range(full):
        item = wave * n_cta + cta
        chunk = item // n_tiles
        k0 = chunk * spc
        out.append((item - chunk * n_tiles, k0, min(k0 + spc, nks)))
    totalB = (n_items - full * n_cta) * spc
    LB = cdiv(totalB, n_cta)
    posB = cta * LB
    endB = min(posB + LB, totalB)
    while posB < endB:
        j = posB // spc
        item = full * n_cta + j
        chunk = item // n_tiles
        kk = posB - j * spc
        seg_end = min((j + 1) * spc, endB)
        k0 = chunk * spc + kk
        k1 = min(k0 + (seg_end - posB), nks)
        posB = seg_end
        if k1 > k0:
            out.append((item - chunk * n_tiles, k0, k1))
    return out


def syrk_shape(nks, n_tiles, M):
    """(n_cta, spc, slots) as o8_syrk_shape chooses them."""
    bytes_per_stage = NUM_SMS / n_tiles * 32 * float(M) * NS
    max_spc = int(110e6 / bytes_per_stage)
    max_spc = max(min(max_spc, MAX_SEG), 32)
    spc = cdiv(nks, cdiv(nks, max_spc))
    items = n_tiles * cdiv(nks, spc)
    n_cta = min(items, NUM_SMS)
    worst = max([1] + [len(cta_segments(n_tiles, nks, spc, c, n_cta)) for c in range(n_cta)])
    return n_cta, spc, worst


def syrk_plan(n, M):
    """Work split of npgp_o8_syrk_digits(n, M): dict with the shape and, per tile, its segments (k0, k1, cta, index) in the
    order the finishing kernel adds them (chunk by chunk, then CTA by CTA: ascending k0)."""
    nks = cdiv(cdiv(n, 128) * 128, 32)
    n_tiles = syrk_tiles(M)
    n_cta, spc, slots = syrk_shape(nks, n_tiles, M)
    per_tile = [[] for _ in range(n_tiles)]
    for c in range(n_cta):
        for idx, (t, k0, k1) in enumerate(cta_segments(n_tiles, nks, spc, c, n_cta)):
            per_tile[t].append((k0, k1, c, idx))
    for segs in per_tile:
        segs.sort()
    n_items = n_tiles * cdiv(nks, spc)
    return dict(nks=nks, n_tiles=n_tiles, n_cta=n_cta, spc=spc, slots=slots, n_items=n_items,
                full=n_items // n_cta, segments=per_tile)


def syrk_reference(D, e, plan, M, alpha=1.0, w0=1.0, skip=None):
    """Out of npgp_o8_syrk_digits from the (7, npad, M) digits D of X and the matrix-wide exponent e: every segment's exact
    partial tile recombined and scaled as the SYRK epilogue does, the partials added in the finishing kernel's order, the
    skip rows' exact correction subtracted, then scaled by alpha * w0.  Returns the full symmetric M x M matrix."""
    dev = D.device
    ee = torch.tensor(e, device=dev)
    rs, sc = scale_or_nan(ee, -36), scale_or_nan(ee, 0)
    Dp = D.permute(1, 0, 2).to(torch.float64)  # (npad, 7, M): a segment's rows are contiguous
    out = torch.empty(M, M, dtype=torch.float64, device=dev)
    corr = None
    if skip is not None and len(skip) > 0:
        Ds = D[:, torch.as_tensor(skip, device=dev).long()]
        corr = recombine(digit_products(Ds.transpose(1, 2), Ds.transpose(1, 2)))  # (M, M), exact over the list
    scale = alpha * w0
    for t, segs in enumerate(plan["segments"]):
        rb, cb = tile_rc(t, M)
        r0, c0 = rb * 128, cb * 64
        acc = torch.zeros(128, 64, dtype=torch.float64, device=dev)
        for k0, k1, _, _ in segs:
            rows = slice(32 * k0, 32 * k1)
            # all 49 digit products of the segment in one GEMM (entries <= 16384 * 2^14: exact), then G_t
            A = Dp[rows, :, r0:r0 + 128].reshape(-1, NS * 128)
            B = Dp[rows, :, c0:c0 + 64].reshape(-1, NS * 64)
            P = (A.T @ B).view(NS, 128, NS, 64)
            G = torch.stack([sum(P[p, :, u - p] for p in range(u + 1)) for u in range(NS)])
            acc = acc + recombine(G) * rs * sc
        if corr is not None:
            acc = acc - corr[r0:r0 + 128, c0:c0 + 64] * rs * sc
        acc = acc * scale
        out[r0:r0 + 128, c0:c0 + 64] = acc
    iu = torch.triu_indices(M, M, device=dev)
    sym = out.clone()
    sym[iu[1], iu[0]] = out[iu[0], iu[1]]
    return sym
