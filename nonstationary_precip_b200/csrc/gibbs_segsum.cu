// Pair sums of the Gibbs kernels over segments of one point set, and segmented weighted column sums of a kernel chunk: the
// two row-side reductions behind the posterior of regional totals (npgp_svgp_region_moments in csrc/svgp_step.cu).
//
// Pair sums.  Rows are sorted by region, region r = rows [seg[r], seg[r+1]).  Each region is cut into tiles of kSegTile
// rows, tiles numbered g = 0 .. S-1 in row order.  A work item is a pair of tiles (g, h), g <= h: the rows of tile g
// against the columns of tile h, pairs i < j only (so a tile against itself evaluates its upper triangle, and a pair of
// rows of two regions r < r' is evaluated once).  One CTA of 128 threads holds 2 columns per thread in registers and walks
// the rows staged 32 at a time in shared memory, as the forward tile kernels do; the per-pair arithmetic is theirs
// (pairmath.cuh), so kappa_ij is bitwise the entry npgp_gibbs_*_fwd(x, x) computes unscaled.  Per thread
// acc_c = sum_i w_i kappa_ij, then w_j acc_c, then a fixed-tree block sum: one FP64 partial per item.  Items are taken from
// a device counter by resident CTAs, so a long region spreads over the whole GPU.  Items of one region: 2 * partial,
// + sum_i w_i^2 on the tile's own item (the same-row pairs, which are not evaluated: kappa(x, x) = 1).
// The item table is the scan of the tile counts (one small kernel reads seg and validates it: no host read, capturable);
// a finishing kernel adds each entry's items in a fixed order (one warp per entry): bitwise reproducible.
#include <cstddef>

#include "common.cuh"
#include "pairmath.cuh"
#include "segsum.cuh"
#include "../../include/npgp.h"

namespace npgp {

constexpr int kSegTile = 256;   // rows of a tile (row and column tiles are the same tiling)
constexpr int kSegNT = 128;     // threads of a pair CTA, 2 columns each
constexpr int kColSlice = 256;  // rows of a slice of the segmented column sums

struct SegHeader {
  int bad;                  // seg is not non-decreasing from 0 to n: every output is NaN (segsum_bad_flag)
  int pad;
  long ntiles, nitems;
  unsigned long long next;  // item counter of the pair kernel
};
static_assert(offsetof(SegHeader, bad) == 0, "segsum_bad_flag reads the first int of the workspace");

struct SegLayout {
  SegHeader* hd;
  long* tile_start;  // R + 1: first tile of region r
  long* item_start;  // R + 1 (variances only): first item of region r
  double* part;      // one partial per item
  long bytes;
};

static inline long align256(long b) { return (b + 255) & ~255L; }

// Largest tile count, largest item count: sum_r ceil(n_r / T) <= ceil(n / T) + R - 1 tiles (and <= n); items of the
// variances sum_r t_r (t_r + 1) / 2 <= f(ceil(n / T)) + R - 1 by convexity, of the full matrix S (S + 1) / 2.
static SegLayout seg_layout(long n, int R, int full, void* work) {
  const long t0 = (n + kSegTile - 1) / kSegTile;
  long smax = t0 + R - 1;
  if (smax > n) smax = n;
  long items = smax * (smax + 1) / 2;
  if (!full) {
    const long b = t0 * (t0 + 1) / 2 + R - 1;
    if (b < items) items = b;
  }
  char* base = static_cast<char*>(work);
  SegLayout L;
  long off = 0;
  L.hd = reinterpret_cast<SegHeader*>(base);
  off += align256(sizeof(SegHeader));
  L.tile_start = reinterpret_cast<long*>(base + off);
  off += align256(8L * (R + 1));
  L.item_start = reinterpret_cast<long*>(base + off);
  off += align256(8L * (R + 1));
  L.part = reinterpret_cast<double*>(base + off);
  off += align256(8L * (items > 0 ? items : 1));
  L.bytes = off;
  return L;
}

// largest r in [0, R) with a[r] <= v (a non-decreasing; a[0] <= v assumed); bounded for any a
__device__ __forceinline__ int upper_region(const long* __restrict__ a, int R, long v) {
  int lo = 0, hi = R - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (a[mid] <= v) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// t = b (b + 1) / 2 + a, 0 <= a <= b
__device__ __forceinline__ void tri_split(long t, long& a, long& b) {
  b = (long)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (b * (b + 1) / 2 > t) --b;
  while ((b + 1) * (b + 2) / 2 <= t) ++b;
  a = t - b * (b + 1) / 2;
}

__device__ __forceinline__ long ntiles_of(long rows) { return (rows + kSegTile - 1) / kSegTile; }

// One CTA: validates seg and scans the tile (and, for the variances, item) counts of the regions.
__global__ void __launch_bounds__(1024) segsum_scan_kernel(long n, int R, const long* __restrict__ seg, int full, SegLayout L) {
  __shared__ long s_t[1024], s_i[1024];
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  if (tid == 0) s_bad = (seg[0] != 0 || seg[R] != n);
  __syncthreads();
  const int per = (R + 1023) / 1024;
  const int r0 = min(R, tid * per), r1 = min(R, r0 + per);
  long ct = 0, ci = 0;
  for (int r = r0; r < r1; ++r) {
    const long len = seg[r + 1] - seg[r];
    if (len < 0) s_bad = 1;
    const long t = ntiles_of(len > 0 ? len : 0);
    ct += t;
    ci += t * (t + 1) / 2;
  }
  s_t[tid] = ct;
  s_i[tid] = ci;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // inclusive scan of the per-thread totals
    const long vt = tid >= o ? s_t[tid - o] : 0, vi = tid >= o ? s_i[tid - o] : 0;
    __syncthreads();
    s_t[tid] += vt;
    s_i[tid] += vi;
    __syncthreads();
  }
  long at = tid ? s_t[tid - 1] : 0, ai = tid ? s_i[tid - 1] : 0;
  for (int r = r0; r < r1; ++r) {
    L.tile_start[r] = at;
    if (!full) L.item_start[r] = ai;
    const long len = seg[r + 1] - seg[r];
    const long t = ntiles_of(len > 0 ? len : 0);
    at += t;
    ai += t * (t + 1) / 2;
  }
  if (tid == 1023) {
    const long S = s_t[1023];
    L.tile_start[R] = S;
    if (!full) L.item_start[R] = s_i[1023];
    L.hd->bad = s_bad;
    L.hd->ntiles = s_bad ? 0 : S;
    L.hd->nitems = s_bad ? 0 : (full ? S * (S + 1) / 2 : s_i[1023]);
    L.hd->next = 0ull;
  }
}

// tile g -> region and rows [i0, i1)
__device__ __forceinline__ int tile_rows(const SegLayout& L, const long* __restrict__ seg, int R, long g, long& i0, long& i1) {
  const int r = upper_region(L.tile_start, R, g);
  i0 = seg[r] + (g - L.tile_start[r]) * kSegTile;
  i1 = min(i0 + kSegTile, seg[r + 1]);
  return r;
}

// item k -> tiles (g, h), g <= h
__device__ __forceinline__ void item_tiles(const SegLayout& L, int R, int full, long k, long& g, long& h) {
  if (full) {
    tri_split(k, g, h);
  } else {
    const int r = upper_region(L.item_start, R, k);
    long a, b;
    tri_split(k - L.item_start[r], a, b);
    g = L.tile_start[r] + a;
    h = L.tile_start[r] + b;
  }
}

// ---- point policies: the forward tile kernels' per-point constants and pair evaluation
template <int D>
struct DiagPoint {
  static constexpr int NF = D;
  double x[D], a[D], c;
  __device__ __forceinline__ void load(long n, long i, const double* __restrict__ X, const double* __restrict__ F) {
    double prod = 1.0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
      x[k] = X[i * D + k];
      const double lv = F[(long)k * n + i];
      a[k] = lv * lv;
      prod *= 1.4142135623730951 * lv;  // 2^(D/2) prod l
    }
    c = sqrt(prod);
  }
  __device__ __forceinline__ void dummy() {
#pragma unroll
    for (int k = 0; k < D; ++k) x[k] = 0.0, a[k] = 1.0;
    c = 1.0;
  }
  __device__ __forceinline__ double eval(const DiagPoint& col, double, const double* etab) const {
    return gibbs_diag_eval<D>(x, a, c, col.x, col.a, col.c, etab);
  }
};

template <int d>
struct FullPoint {
  static constexpr int P = sym_size(d);
  double x[d], S[P], q;  // row point: q = det(S)^(1/4); column point: q = full_col_factor (2^(d/2) folded in)
  template <bool COL>
  __device__ __forceinline__ void load_t(long i, const double* __restrict__ X, const double* __restrict__ F) {
#pragma unroll
    for (int k = 0; k < d; ++k) x[k] = X[i * d + k];
#pragma unroll
    for (int p = 0; p < P; ++p) S[p] = F[i * P + p];
    q = COL ? full_col_factor<d>(sym_det<d>(S)) : sqrt(sqrt(sym_det<d>(S)));
  }
  __device__ __forceinline__ void dummy() {
#pragma unroll
    for (int k = 0; k < d; ++k) x[k] = 0.0;
#pragma unroll
    for (int p = 0; p < P; ++p) S[p] = 0.0;
#pragma unroll
    for (int k = 0; k < d; ++k) S[sym_idx(d, k, k)] = 1.0;
    q = 1.0;
  }
  __device__ __forceinline__ double eval(const FullPoint& col, double jit2, const double* etab) const {
    return gibbs_full_eval<d>(x, S, q, col.x, col.S, col.q, jit2, etab);
  }
};

template <class Pt>
__device__ __forceinline__ void load_point(Pt& p, long n, long i, const double* X, const double* F, bool col);
template <int D>
__device__ __forceinline__ void load_point(DiagPoint<D>& p, long n, long i, const double* X, const double* F, bool) {
  p.load(n, i, X, F);
}
template <int d>
__device__ __forceinline__ void load_point(FullPoint<d>& p, long, long i, const double* X, const double* F, bool col) {
  if (col) p.template load_t<true>(i, X, F);
  else p.template load_t<false>(i, X, F);
}

struct PairArgs {
  long n;
  int R, full, part, nparts;
  const double* x;
  const double* F;  // ell (D, n) or Sigma (n, P)
  const double* w;
  const long* seg;
  double jit2;
  SegLayout L;
};

template <class Pt, bool TRI>
__device__ __forceinline__ void item_rows(const Pt (&rows)[kTI], const double* sw, int nr, long ib, const Pt (&col)[2],
                                          const long* jg, double jit2, const double* etab, double (&acc)[2]) {
#pragma unroll 2
  for (int r = 0; r < nr; ++r) {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      double k = rows[r].eval(col[c], jit2, etab);
      if (TRI) k = (jg[c] > ib + r) ? k : 0.0;
      acc[c] = fma(sw[r], k, acc[c]);
    }
  }
}

template <class Pt>
__global__ void __launch_bounds__(kSegNT) segsum_pairs_kernel(PairArgs a) {
  __shared__ Pt rows[kTI];
  __shared__ double sw[kTI], sexp[256], red[32];
  __shared__ long s_k;
  load_exp_table(sexp);
  const SegHeader* hd = a.L.hd;
  const long nitems = hd->nitems;  // 0 for a bad seg
  const long k0 = nitems * a.part / a.nparts, k1 = nitems * (a.part + 1) / a.nparts;
  const int tid = threadIdx.x, warp = tid >> 5;
  for (;;) {
    __syncthreads();  // everyone has read s_k of the previous item
    if (tid == 0) s_k = k0 + (long)atomicAdd(&a.L.hd->next, 1ull);
    __syncthreads();
    const long k = s_k;
    if (k >= k1) break;
    long g, h, i0, i1, j0, j1;
    item_tiles(a.L, a.R, a.full, k, g, h);
    const int rg = tile_rows(a.L, a.seg, a.R, g, i0, i1);
    const int rh = tile_rows(a.L, a.seg, a.R, h, j0, j1);
    Pt col[2];
    long jg[2];
    double wj[2], acc[2] = {0.0, 0.0};
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      jg[c] = j0 + 2 * tid + c;
      const bool valid = jg[c] < j1;
      if (valid) load_point(col[c], a.n, jg[c], a.x, a.F, true);
      else col[c].dummy();
      wj[c] = valid ? (a.w ? a.w[jg[c]] : 1.0) : 0.0;
    }
    // a tile against itself: a row needs the columns right of it only, so a warp stops at its last column
    const long jw = min(j0 + 64 * warp + 63, j1 - 1);
    double w2 = 0.0;
    for (long ib = i0; ib < i1; ib += kTI) {
      __syncthreads();
      const int nr = (int)min((long)kTI, i1 - ib);
      if (tid < nr) {
        load_point(rows[tid], a.n, ib + tid, a.x, a.F, false);
        const double wi = a.w ? a.w[ib + tid] : 1.0;
        sw[tid] = wi;
        w2 = fma(wi, wi, w2);
      }
      __syncthreads();
      if (g == h) {
        const int rhi = (int)max(0L, min((long)nr, jw - ib));
        item_rows<Pt, true>(rows, sw, rhi, ib, col, jg, a.jit2, sexp, acc);
      } else {
        item_rows<Pt, false>(rows, sw, nr, 0, col, jg, a.jit2, sexp, acc);
      }
    }
    const double t = block_sum(fma(wj[0], acc[0], wj[1] * acc[1]), red);
    const double tw = (g == h) ? block_sum(w2, red) : 0.0;
    if (tid == 0) a.L.part[k] = (rg == rh) ? fma(2.0, t, tw) : t;
  }
}

// One warp per output entry (r, r'), r <= r' (variances: r' = r): adds the entry's items of this part in a fixed order
// (lane-strided over the entry's tile pairs, then a butterfly), scales by *scale and writes Gdiag / G (mirrored).
__global__ void __launch_bounds__(256) segsum_finish_kernel(int R, int full, int part, int nparts, const double* __restrict__ scale,
                                                             SegLayout L, double* __restrict__ Gdiag, double* __restrict__ G,
                                                             long ldg) {
  const long e = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const long nent = full ? (long)R * (R + 1) / 2 : R;
  if (e >= nent) return;
  long r, rp;
  if (full) tri_split(e, r, rp);  // e = rp (rp + 1) / 2 + r, r <= rp
  else r = rp = e;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  double v;
  if (L.hd->bad) {
    v = nan;
  } else {
    const long nitems = L.hd->nitems;
    const long k0 = nitems * part / nparts, k1 = nitems * (part + 1) / nparts;
    const long tr = L.tile_start[r], nt = L.tile_start[r + 1] - tr;
    const long trp = L.tile_start[rp], ntp = L.tile_start[rp + 1] - trp;
    const long cnt = (r == rp) ? nt * (nt + 1) / 2 : nt * ntp;
    double s = 0.0;
    for (long t = lane; t < cnt; t += 32) {
      long ta, tb;
      if (r == rp) tri_split(t, ta, tb);
      else ta = t / ntp, tb = t % ntp;
      const long g = tr + ta, h = trp + tb;
      const long k = full ? h * (h + 1) / 2 + g : L.item_start[r] + tb * (tb + 1) / 2 + ta;
      if (k >= k0 && k < k1) s += L.part[k];
    }
    s = warp_sum(s);
    v = scale ? *scale * s : s;
  }
  if (lane) return;
  if (r == rp) Gdiag[r] = v;
  if (full) {
    G[r * ldg + rp] = v;
    G[rp * ldg + r] = v;
  }
}

// ---- segmented weighted column sums of one chunk of K (rows row0 .. row0 + n - 1 of the sorted set)
// piece of region r in the chunk: [max(seg[r], c0), min(seg[r+1], c1))
// Pass 1, thread (slice s, column j): walks the slice's rows in order.  A piece that lies in the slice is added to out
// directly (its only contributor in this launch); the part of a piece that began in an earlier slice goes to head[s], the
// part of one that begins here and continues goes to tail[s].
__global__ void __launch_bounds__(128) segcol_pass1_kernel(int n, int M, const double* __restrict__ K, long ldk,
                                                           const double* __restrict__ w, long row0, int R,
                                                           const long* __restrict__ seg, double* __restrict__ out, long ldo,
                                                           double* __restrict__ head, double* __restrict__ tail) {
  const int j = blockIdx.x * 128 + threadIdx.x, s = blockIdx.y;
  if (j >= M) return;
  const long c0 = row0, c1 = row0 + n;
  const long lo = row0 + (long)s * kColSlice, hi = min(lo + kColSlice, c1);
  int r = upper_region(seg, R, lo);
  long nb = seg[r + 1], start = lo;
  double acc = 0.0;
  auto flush = [&](long end) {
    if (end <= start) return;
    const long plo = max(seg[r], c0), phi = min(seg[r + 1], c1);
    if (plo < lo) head[(long)s * M + j] = acc;
    else if (phi > hi) tail[(long)s * M + j] = acc;
    else out[(long)r * ldo + j] += acc;
  };
  for (long gi = lo; gi < hi; ++gi) {
    if (gi >= nb && r < R - 1) {
      flush(gi);
      while (r < R - 1 && seg[r + 1] <= gi) ++r;
      nb = seg[r + 1];
      start = gi;
      acc = 0.0;
    }
    const long i = gi - row0;
    acc = fma(w ? w[i] : 1.0, K[i * ldk + j], acc);
  }
  flush(hi);
}

// Pass 2, thread (slice s, column j): the owner of the piece that begins in slice s and continues adds its tail and the
// heads of the following slices in order.
__global__ void __launch_bounds__(128) segcol_pass2_kernel(int n, int M, long row0, int R, const long* __restrict__ seg,
                                                           double* __restrict__ out, long ldo, const double* __restrict__ head,
                                                           const double* __restrict__ tail) {
  const int j = blockIdx.x * 128 + threadIdx.x, s = blockIdx.y;
  if (j >= M) return;
  const long c0 = row0, c1 = row0 + n;
  const long lo = row0 + (long)s * kColSlice, hi = min(lo + kColSlice, c1);
  const int r = upper_region(seg, R, hi - 1);
  const long plo = max(seg[r], c0), phi = min(seg[r + 1], c1);
  if (!(plo >= lo && phi > hi)) return;
  double acc = tail[(long)s * M + j];
  for (long t = s + 1; row0 + t * kColSlice < phi; ++t) acc += head[t * M + j];
  out[(long)r * ldo + j] += acc;
}

template <class Pt>
static int launch_pairs(const PairArgs& a, cudaStream_t st) {
  static int per_sm = 0;
  if (!per_sm) {
    NPGP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, segsum_pairs_kernel<Pt>, kSegNT, 0));
    if (per_sm < 1) per_sm = 1;
  }
  segsum_pairs_kernel<Pt><<<kNumSMs * per_sm, kSegNT, 0, st>>>(a);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

}  // namespace npgp

using namespace npgp;

extern "C" long npgp_segsum_workspace_bytes(long n, int R, int full) {
  if (n < 0 || n >= (1L << 31) || R < 1) return -1;
  return seg_layout(n, R, full, nullptr).bytes;
}

static int segsum_run(int variant, int D, long n, const double* x, const double* F, double jitter, const double* w, int R,
                      const long* seg, int full, int part, int nparts, const double* scale, double* Gdiag, double* G, long ldg,
                      void* work, long work_bytes, cudaStream_t st) {
  if (R < 1 || n < 0 || n >= (1L << 31) || nparts < 1 || part < 0 || part >= nparts) return NPGP_EINVAL;
  if (variant == 0 ? (D < 1 || D > 6) : (D != 2 && D != 3)) return NPGP_EINVAL;
  if (!seg || !Gdiag || !work || (full && (!G || ldg < R)) || (n > 0 && (!x || !F))) return NPGP_EINVAL;
  if (reinterpret_cast<uintptr_t>(work) & 255) return NPGP_EUNSUPPORTED;
  const SegLayout L = seg_layout(n, R, full, work);
  if (work_bytes < L.bytes) return NPGP_EWORKSPACE;
  segsum_scan_kernel<<<1, 1024, 0, st>>>(n, R, seg, full, L);
  NPGP_LAUNCH_CHECK();
  PairArgs a{n, R, full, part, nparts, x, F, w, seg, 2.0 * jitter, L};
  if (n > 0) {
    int rc = NPGP_OK;
    if (variant == 1) rc = D == 2 ? launch_pairs<FullPoint<2>>(a, st) : launch_pairs<FullPoint<3>>(a, st);
    else switch (D) {
        case 1: rc = launch_pairs<DiagPoint<1>>(a, st); break;
        case 2: rc = launch_pairs<DiagPoint<2>>(a, st); break;
        case 3: rc = launch_pairs<DiagPoint<3>>(a, st); break;
        case 4: rc = launch_pairs<DiagPoint<4>>(a, st); break;
        case 5: rc = launch_pairs<DiagPoint<5>>(a, st); break;
        default: rc = launch_pairs<DiagPoint<6>>(a, st); break;
      }
    if (rc) return rc;
  }
  const long nent = full ? (long)R * (R + 1) / 2 : R;
  segsum_finish_kernel<<<(unsigned)((nent + 7) / 8), 256, 0, st>>>(R, full, part, nparts, scale, L, Gdiag, G, ldg);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

extern "C" int npgp_gibbs_diag_segsum(int D, long n, const double* x, const double* ell, const double* w, int R, const long* seg,
                                      int full, int part, int nparts, const double* scale, double* Gdiag, double* G, long ldg,
                                      void* work, long work_bytes, cudaStream_t stream) {
  return segsum_run(0, D, n, x, ell, 0.0, w, R, seg, full, part, nparts, scale, Gdiag, G, ldg, work, work_bytes, stream);
}

extern "C" int npgp_gibbs_full_segsum(int d, long n, const double* x, const double* S, double jitter, const double* w, int R,
                                      const long* seg, int full, int part, int nparts, const double* scale, double* Gdiag,
                                      double* G, long ldg, void* work, long work_bytes, cudaStream_t stream) {
  return segsum_run(1, d, n, x, S, jitter, w, R, seg, full, part, nparts, scale, Gdiag, G, ldg, work, work_bytes, stream);
}

extern "C" long npgp_segment_colwsum_workspace_bytes(int n, int M) {
  if (n < 0 || M < 1) return -1;
  return 2L * ((n + kColSlice - 1) / kColSlice) * M * 8;
}

extern "C" int npgp_segment_colwsum(int n, int M, const double* K, long ldk, const double* w, long row0, int R, const long* seg,
                                    double* out, long ldo, void* work, long work_bytes, cudaStream_t stream) {
  if (n < 0 || M < 1 || R < 1 || row0 < 0 || ldk < M || ldo < M) return NPGP_EINVAL;
  if (n == 0) return NPGP_OK;
  if (!K || !seg || !out || !work) return NPGP_EINVAL;
  if (reinterpret_cast<uintptr_t>(work) & 7) return NPGP_EUNSUPPORTED;
  if (work_bytes < npgp_segment_colwsum_workspace_bytes(n, M)) return NPGP_EWORKSPACE;
  const int ns = ceil_div(n, kColSlice);
  double* head = static_cast<double*>(work);
  double* tail = head + (long)ns * M;
  dim3 grid(ceil_div(M, 128), ns);
  segcol_pass1_kernel<<<grid, 128, 0, stream>>>(n, M, K, ldk, w, row0, R, seg, out, ldo, head, tail);
  NPGP_LAUNCH_CHECK();
  segcol_pass2_kernel<<<grid, 128, 0, stream>>>(n, M, row0, R, seg, out, ldo, head, tail);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}
