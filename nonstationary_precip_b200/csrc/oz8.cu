// Exact FP64 contractions on the int8 tensor cores (tcgen05.mma kind::i8, accumulators in TMEM), byte-digit edition:
//     row-quadratic:  T = K C,  q_i = sum_j T_ij K_ij,  optional du = K^T g         (npgp_rowquad_i8*, npgp_o8_rowquad_digits)
//     SYRK:           Out = alpha w0 K^T K                                          (npgp_syrk_i8*,    npgp_o8_syrk_digits)
// replacing the reference's dense products k_ux1.matmul(inv_root) / A^T (S - I) A (models/gibbs_kernels.py:222-232 and the
// whitened VariationalStrategy driven by models/dgps.py:25-35).  B200 has no FP64 tcgen05 kind and DMMA peaks at 37 TFLOP/s.
//
// Arithmetic (oz8.cuh): each operand entry is the integer y = rint(x 2^(54-e)) with a power-of-two scale per row (or per
// matrix), written as 7 signed base-256 digits.  Then
//     T_ij = 2^(e_i + f_j - 12) sum_{t=0..6} 2^(-8t) G_t,     G_t = sum_{p+q=t} (a_p c_q^T)_ij   exact in int32,
// 28 digit products (round 1: 8 seven-bit digits, 36 products); the dropped terms t >= 7 are below 2^-52 of
// (row max)(column max) per contraction entry, the size of the FP64 rounding bound itself.  The seven G_t live in seven
// TMEM accumulators of 128 lanes x 64 columns.
//
// Data flow.  Digit planes arrive in the row layout of oz8.cuh -- written by the slicing kernels below for arbitrary
// operands, or directly by the Gibbs tile kernels (gibbs_digits.cu) for K(X,Z), which then never exists in FP64.  Warp
// roles per CTA (one persistent CTA per SM): warp 0 producer (cp.async.bulk / TMA tensor copies global -> shared, mbarrier
// completion), warp 1 MMA issuer (one elected lane, 28 MMAs per 32-byte k-step, A-operand collector reuse across the B
// digits, tcgen05.commit frees the stage), epilogue warps (4 in the SYRK, 8 in the row-quadratic kernel, which releases TMEM
// as soon as the accumulators sit in registers: tcgen05.ld, integer recombination, power-of-two scaling,
// fused row dot / column sums against the K tile rebuilt from the digits while the MMAs run).
// The SYRK contracts over the ROWS of K.  With a matrix-wide scale it reads the same row-layout planes MN-major
// (instruction descriptor a_major = b_major = 1; verified by tools/probes/umma_i8_probe2.cu), each operand tile fetched by
// one 5-D TMA box; with per-column scales (general operands) it reads transposed planes written by o8_slice_t_kernel.
// Row chunks of <= 16384 rows keep int32 exact; every (tile, chunk) segment stores its FP64 partial tile and a finishing kernel
// adds a tile's segments in a fixed order (no FP64 atomics: results are bitwise reproducible).  Work decomposition: O8SegIter.
// Descriptor encodings: cute/arch/mma_sm100_desc.hpp of the vendored CUTLASS.
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)
#include <cstring>
#include <cstdint>

#include "common.cuh"
#include "oz8.cuh"

namespace npgp {

constexpr int O8_THREADS = 192;             // SYRK: producer, MMA issuer, 4 epilogue warps
constexpr int O8_RQ_THREADS = 320;          // row-quadratic kernel: producer, MMA issuer, 8 epilogue warps
constexpr int O8_RQ_STAGES = 3;
constexpr int O8_SY_STAGES = 4;
constexpr int O8_KLD = O8_BN + 2;            // leading dimension (doubles) of the staged K tile
constexpr int O8_MAX_SEG = 512;              // <= 16384 contraction rows per int32 accumulation of the SYRK (bound: 18724)
constexpr int O8_RQ_SMEM = O8_RQ_STAGES * (O8_A_STAGE + O8_B_STAGE) + O8_BM * O8_KLD * 8 + 1024;
constexpr int O8_SY_SMEM = O8_SY_STAGES * (O8_A_STAGE + O8_B_STAGE) + 1024;

// ---------------------------------------------------------------------------------------------------------------------
// slicing kernels for arbitrary FP64 operands
// ---------------------------------------------------------------------------------------------------------------------
// Row-wise: operand rows = rows of X (R x Kd), contraction along the columns.  CTA = 8 consecutive rows x 64 chunks of 16
// columns (512 threads; longer rows loop).  Rows >= R (up to Rpad) are written as zeros.
template <int BR>
__global__ void __launch_bounds__(512, 2) o8_slice_rows_kernel(int R, int Rpad, int Kd, const double* __restrict__ X, long ldx,
                                                               int8_t* __restrict__ out, int* __restrict__ expo) {
  __shared__ unsigned long long smax[16][8];
  __shared__ int sexp[8];
  const int t = threadIdx.x, rr = t & 7, ch = t >> 3, warp = t >> 5;
  const int r = blockIdx.x * 8 + rr;
  const int nks = Kd / O8_KS, nch = Kd / 16;
  double v[16];
  unsigned long long mx = 0;
  for (int c = ch; c < nch; c += 64) {
    if (r < R) {
      const double2* src = reinterpret_cast<const double2*>(X + (long)r * ldx + c * 16);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const double2 d = src[j];
        if (c == ch) { v[2 * j] = d.x; v[2 * j + 1] = d.y; }
        const unsigned long long bx = (unsigned long long)__double_as_longlong(fabs(d.x));
        const unsigned long long by = (unsigned long long)__double_as_longlong(fabs(d.y));
        mx = max(mx, max(bx, by));
      }
    } else if (c == ch) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = 0.0;
    }
  }
  mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
  mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
  if ((t & 31) < 8) smax[warp][rr] = mx;
  __syncthreads();
  if (t < 8) {
    unsigned long long m = 0;
#pragma unroll
    for (int w = 0; w < 16; ++w) m = max(m, smax[w][t]);
    const int e = o8_exponent_of_max(m);
    sexp[t] = e;
    if (blockIdx.x * 8 + t < Rpad) expo[blockIdx.x * 8 + t] = e;
  }
  __syncthreads();
  if (r >= Rpad) return;
  const int e = sexp[rr];
  const double sc = (e == O8_POISON) ? 0.0 : o8_pow2(O8_FRAC - e);
  const long blk = (long)(r / BR) * nks;
  const int rin = ((r % BR) / 8) * 128 + (r % 8) * 16;
  for (int c = ch; c < nch; c += 64) {
    if (c != ch && r < R) {
      const double2* src = reinterpret_cast<const double2*>(X + (long)r * ldx + c * 16);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const double2 d = src[j];
        v[2 * j] = d.x;
        v[2 * j + 1] = d.y;
      }
    }
    long long y[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) y[j] = (e == O8_POISON) ? 0ll : o8_quantise(v[j], sc);
    if (BR == O8_BM)  // A-type layout: digit-major inside the row block
      o8_store_digits(y, out + o8_a_offset(r, c * 16, nks), (long)nks * O8_A_PLANE);
    else              // B-type layout: stage-contiguous
      o8_store_digits(y, out + ((blk + c / 2) * O8_NS * 2 + (c & 1)) * (long)(BR * 16) + rin, 2L * (BR * 16));
  }
}

// Column maxima of |X| (R x Kd) as bit patterns (non-negative doubles order like integers; inf / nan sort last); cmax zeroed
// by the caller.  Optionally the same pass accumulates the weighted column sums wsum[j] += sum_i w_i X_ij.
__global__ void __launch_bounds__(256) o8_colmax_kernel(int R, int Kd, const double* __restrict__ X, long ldx, int rows_per_cta,
                                                        unsigned long long* __restrict__ cmax, const double* __restrict__ w,
                                                        double* __restrict__ wsum) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= Kd) return;
  const int i0 = blockIdx.y * rows_per_cta, i1 = min(R, i0 + rows_per_cta);
  unsigned long long m = 0;
  double acc = 0.0;
  for (int i = i0; i < i1; ++i) {
    const double v = X[(long)i * ldx + j];
    m = max(m, (unsigned long long)__double_as_longlong(fabs(v)));
    if (w) acc = fma(w[i], v, acc);
  }
  if (w) atomicAdd(&wsum[j], acc);
  atomicMax(&cmax[j], m);
}

__global__ void o8_exp_from_max_kernel(int n, const unsigned long long* __restrict__ cmax, int* __restrict__ expo) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) expo[j] = o8_exponent_of_max(cmax[j]);
}

// Transposed slicing for the general SYRK: operand rows = columns j of X (R x Kd), contraction along the rows i, per-column
// scales.  CTA = one k-stage (32 rows i) x 128 columns j.  Layout as o8_slice_rows_kernel<128> with (row, k) = (j, i).
__global__ void __launch_bounds__(256) o8_slice_t_kernel(int R, int Kd, const double* __restrict__ X, long ldx,
                                                         const int* __restrict__ expo, int8_t* __restrict__ out) {
  __shared__ double tile[32][129];
  const int ks = blockIdx.x, jb = blockIdx.y, nks = gridDim.x;
  for (int e = threadIdx.x; e < 32 * 128; e += 256) {
    const int i = e >> 7, j = e & 127;
    const int gi = ks * 32 + i, gj = jb * 128 + j;
    tile[i][j] = (gi < R && gj < Kd) ? X[(long)gi * ldx + gj] : 0.0;
  }
  __syncthreads();
  const int j = threadIdx.x & 127, half = threadIdx.x >> 7;
  const int gj = jb * 128 + j;
  const int e = (gj < Kd) ? expo[gj] : 0;
  const double sc = (e == O8_POISON) ? 0.0 : o8_pow2(O8_FRAC - e);
  long long y[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) y[k] = (e == O8_POISON) ? 0ll : o8_quantise(tile[half * 16 + k][j], sc);
  o8_store_digits(y, out + o8_a_offset((long)jb * O8_BM + j, ks * O8_KS + half * 16, nks), (long)nks * O8_A_PLANE);
}

// ---------------------------------------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t o8_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void o8_mbar_init(uint64_t* b, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(o8_smem(b)), "r"(count));
}
__device__ __forceinline__ void o8_mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
        : "=r"(done)
        : "r"(o8_smem(b)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void o8_mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(o8_smem(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void o8_mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(o8_smem(b)) : "memory");
}
__device__ __forceinline__ void o8_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* b) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(o8_smem(dst)),
               "l"(src), "r"(bytes), "r"(o8_smem(b))
               : "memory");
}
// one 5-D TMA box (tile mode) global -> shared, completion on the mbarrier
__device__ __forceinline__ void o8_tma_5d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, int c4, uint64_t* b) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(
          o8_smem(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(o8_smem(b))
      : "memory");
}
__device__ __forceinline__ void o8_commit(uint64_t* b) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(o8_smem(b)) : "memory");
}
// one elected lane of a fully active warp: a tcgen05 instruction under this predicate is issued once, without the
// elect-and-retry loop the compiler wraps around the same instruction in a `lane == 0` branch
__device__ __forceinline__ bool o8_elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint64_t o8_desc(uint32_t lo, uint32_t hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}
__device__ __forceinline__ void o8_tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}

#define O8_DEFINE_MMA(NAME, COLL)                                                                                        \
  __device__ __forceinline__ void NAME(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {             \
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"                                                       \
                 "tcgen05.mma.cta_group::1.kind::i8" COLL " [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d),                       \
                 "l"(da), "l"(db), "r"(idesc), "r"(acc)                                                                  \
                 : "memory");                                                                                            \
  }
O8_DEFINE_MMA(o8_mma_plain, "")
O8_DEFINE_MMA(o8_mma_fill, ".collector::a::fill")
O8_DEFINE_MMA(o8_mma_use, ".collector::a::use")
O8_DEFINE_MMA(o8_mma_last, ".collector::a::lastuse")

// The 28 digit products of one k-step: A digit p (descriptor a_lo + p * a_plane16) against B digits q = 0 .. 6 - p, into
// accumulator p + q.  The A operand of a fixed p is reused across its B digits (collector hints).
template <bool COLL>
__device__ __forceinline__ void o8_issue_kstep(uint32_t tmem, uint32_t a_lo, uint32_t a_hi, uint32_t a_plane16, uint32_t b_lo,
                                               uint32_t b_hi, uint32_t b_plane16, uint32_t idesc_base, uint32_t first) {
#pragma unroll
  for (int p = 0; p < O8_NS; ++p) {
    const uint64_t da = o8_desc(a_lo + p * a_plane16, a_hi);
#pragma unroll
    for (int qq = 0; qq < O8_NS - p; ++qq) {
      const uint64_t db = o8_desc(b_lo + qq * b_plane16, b_hi);
      const uint32_t idesc = idesc_base;  // every digit is signed: S8 x S8
      const uint32_t d = tmem + (uint32_t)((p + qq) * O8_BN);
      const uint32_t acc = p > 0 ? 1u : first;
      if (!COLL || p == O8_NS - 1) o8_mma_plain(d, da, db, idesc, acc);
      else if (qq == 0) o8_mma_fill(d, da, db, idesc, acc);
      else if (qq == O8_NS - 1 - p) o8_mma_last(d, da, db, idesc, acc);
      else o8_mma_use(d, da, db, idesc, acc);
    }
  }
}

// sum_t 2^(-8t) G_t = 2^-24 (hi + 2^-24 lo) with hi, lo exact 64-bit integers
__device__ __forceinline__ double o8_recombine(const uint32_t (&g)[O8_NS][8], int j) {
  long long hi = (int)g[0][j], lo = (int)g[4][j];
#pragma unroll
  for (int t = 1; t < 4; ++t) hi = hi * 256 + (int)g[t][j];
#pragma unroll
  for (int t = 5; t < O8_NS; ++t) lo = lo * 256 + (int)g[t][j];
  return fma((double)lo, 5.9604644775390625e-08 /* 2^-24 */, (double)hi);
}

__device__ __forceinline__ double o8_scale_or_nan(int e, int shift) {
  return (e == O8_POISON) ? __longlong_as_double(0x7FF8000000000000ll) : o8_pow2(e + shift);
}

// first k-step of column block cb of a lower-triangular B operand: blocks at or past the split column start there
__device__ __forceinline__ int o8_tri_klo(int cb, int ms_ks) { return (ms_ks > 0 && 2 * cb >= ms_ks) ? ms_ks : 0; }
// column block of tile `tile` (row block rb): row-block-major, snake order in the TRI mode
template <bool TRI>
__device__ __forceinline__ int o8_rq_cb(int tile, int rb, int n_cb) {
  if constexpr (TRI) return (rb & 1) ? n_cb - 1 - tile % n_cb : tile % n_cb;
  else return tile % n_cb;
}

// ---------------------------------------------------------------------------------------------------------------------
// T (n x N) = K C,  q += rowdot(T, K),  du_part[rb] = column sums of g_i K_ij over the rows of row block rb.
// Persistent: grid = #SMs, tiles (rb, cb) in row-block-major order so that CTAs working at the same time share A through L2.
//   As / ea: A digit planes (row layout, BR = 128) and per-row exponents; ea == NULL: one exponent for the matrix, derived
//            from the positive device scalar *a_scale (the Gibbs kernels' outputscale; entries lie in [0, scale]).
//   Bs / eb: digit planes of the symmetric C (BR = 64) and its per-row (= per-column) exponents.
//   Kmat:    optional FP64 K for the row dot / column sums; NULL: K is rebuilt from the A digits.
//   q:       q_stride == 0: q[row] += (atomics);  q_stride > 0: q[cb * q_stride + row] = partial (deterministic)
//   WT:      false: T is not stored (T unused, q required); the row dot is formed from the same products in the same order
// The row dot and the column sums need N == Kd (they pair T with K); with q and du_part NULL the output width N (B rows) and
// the contraction length Kd are independent: T = A B^T of npgp_o8_gemm_digits.
//   TRI:     B is lower triangular (npgp_o8_trinorm_digits): q[cb * q_stride + row] = sum_{j in cb} T_ij^2 (T, K never
//            formed), column block cb contracts over k-steps [klo(cb), 2 (cb + 1)) only, klo = ms_ks for blocks at or past
//            the split column (ms_ks k-steps; 0: no split), else 0.  The tiles of a row block run in snake order (cb
//            descending on odd row blocks) so that the persistent CTAs, which take every gridDim.x-th tile, get even work.
// ---------------------------------------------------------------------------------------------------------------------
template <bool COLL, bool WT, bool TRI = false>
__global__ void __launch_bounds__(O8_RQ_THREADS, 1)
o8_rowquad_kernel(int n, int N, int Kd, const int8_t* __restrict__ As, const int* __restrict__ ea,
                  const double* __restrict__ a_scale, const int8_t* __restrict__ Bs, const int* __restrict__ eb,
                  const double* __restrict__ Kmat, long ldk, double* __restrict__ T, long ldt, double* __restrict__ q,
                  long q_stride, const double* __restrict__ gvec, double* __restrict__ du_part, long long* __restrict__ dbg,
                  int ms_ks) {
  extern __shared__ __align__(1024) uint8_t o8_sm[];
  uint8_t* sA = o8_sm;
  uint8_t* sB = o8_sm + O8_RQ_STAGES * O8_A_STAGE;
  double* sK = reinterpret_cast<double*>(o8_sm + O8_RQ_STAGES * (O8_A_STAGE + O8_B_STAGE));  // 128 x O8_KLD tile of K
  __shared__ double scol[O8_BN], sg[O8_BM], sq[O8_BM];
  __shared__ __align__(8) uint64_t full[O8_RQ_STAGES], empty[O8_RQ_STAGES], acc_full, acc_empty;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nks = Kd / O8_KS, n_rb = (n + O8_BM - 1) / O8_BM, n_cb = N / O8_BN;
  const int n_tiles = n_rb * n_cb;

  if (tid == 0) {
    for (int s = 0; s < O8_RQ_STAGES; ++s) {
      o8_mbar_init(&full[s], 1);
      o8_mbar_init(&empty[s], 1);
    }
    o8_mbar_init(&acc_full, 1);
    o8_mbar_init(&acc_empty, 8);  // one arrival per epilogue warp
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(o8_smem(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_s;

  if (warp == 0) {
    // ===== producer: lanes 0..6 copy the seven digit planes of the A block's k-step (4 KB each), lane 7 the B stage =====
    int stage = 0;
    uint32_t phase = 0;
    long long w_empty = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int rb = tile / n_cb, cb = o8_rq_cb<TRI>(tile, rb, n_cb);
      const int8_t* a = As + ((long)rb * O8_NS + lane) * nks * O8_A_PLANE;  // lane = digit
      const int8_t* b = Bs + (long)cb * nks * O8_B_STAGE;
      const int k_lo = TRI ? o8_tri_klo(cb, ms_ks) : 0, k_hi = TRI ? min(nks, 2 * (cb + 1)) : nks;
      for (int ks = k_lo; ks < k_hi; ++ks) {
        const long long c0 = dbg ? clock64() : 0;
        o8_mbar_wait(&empty[stage], phase ^ 1);
        if (dbg) w_empty += clock64() - c0;
        if (lane == 0) o8_mbar_expect_tx(&full[stage], O8_A_STAGE + O8_B_STAGE);
        __syncwarp();
        if (lane < O8_NS)
          o8_bulk_g2s(sA + stage * O8_A_STAGE + lane * O8_A_PLANE, a + (long)ks * O8_A_PLANE, O8_A_PLANE, &full[stage]);
        else if (lane == O8_NS)
          o8_bulk_g2s(sB + stage * O8_B_STAGE, b + (long)ks * O8_B_STAGE, O8_B_STAGE, &full[stage]);
        if (++stage == O8_RQ_STAGES) { stage = 0; phase ^= 1; }
      }
    }
    if (dbg && blockIdx.x == 0 && lane == 0) dbg[0] = w_empty;
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp runs the loop (warp-uniform control flow), one elected lane issues =====
    const bool leader = o8_elect_one();
    // c_format S32 (2) @4, a/b format signed 8 bit (1) @7/@10, both K-major, N>>3 @17, M>>4 @24
    const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(O8_BN >> 3) << 17) | ((uint32_t)(O8_BM >> 4) << 24);
    constexpr uint32_t kHi = (128u >> 4) | (1u << 14);  // stride byte offset 128 (next 8 rows), descriptor version 1
    int stage = 0;
    uint32_t phase = 0, acc_phase = 0;
    long long w_acc = 0, w_full = 0, t_all = dbg ? clock64() : 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      long long c0 = dbg ? clock64() : 0;
      o8_mbar_wait(&acc_empty, acc_phase ^ 1);  // epilogue has drained the accumulators of the previous tile
      if (dbg) w_acc += clock64() - c0;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int k_lo = TRI ? o8_tri_klo(o8_rq_cb<TRI>(tile, tile / n_cb, n_cb), ms_ks) : 0;
      const int k_hi = TRI ? min(nks, 2 * (o8_rq_cb<TRI>(tile, tile / n_cb, n_cb) + 1)) : nks;
      for (int ks = k_lo; ks < k_hi; ++ks) {
        c0 = dbg ? clock64() : 0;
        o8_mbar_wait(&full[stage], phase);
        if (dbg) w_full += clock64() - c0;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (leader) {
          // leading byte offset = distance of the two 16-byte halves of the k-step (BR * 16)
          const uint32_t a_lo = ((o8_smem(sA + stage * O8_A_STAGE) >> 4) & 0x3FFFu) | ((uint32_t)(O8_BM * 16 >> 4) << 16);
          const uint32_t b_lo = ((o8_smem(sB + stage * O8_B_STAGE) >> 4) & 0x3FFFu) | ((uint32_t)(O8_BN * 16 >> 4) << 16);
          o8_issue_kstep<COLL>(tmem, a_lo, kHi, 2 * O8_BM * 16 >> 4, b_lo, kHi, 2 * O8_BN * 16 >> 4, idesc, ks > k_lo ? 1u : 0u);
          o8_commit(&empty[stage]);  // frees the stage when these MMAs have read it
        }
        __syncwarp();
        if (++stage == O8_RQ_STAGES) { stage = 0; phase ^= 1; }
      }
      if (leader) o8_commit(&acc_full);
      __syncwarp();
      acc_phase ^= 1;
    }
    if (dbg && blockIdx.x == 0 && leader) {
      dbg[1] = w_acc;
      dbg[2] = w_full;
      dbg[3] = clock64() - t_all;
    }
  } else {
    // ===== epilogue: warps 2..9.  TMEM lane quadrant = warp % 4 (hardware rule), column half = (warp - 2) / 4: a thread owns
    // 32 columns of one row.  Phase 1 (the only part the MMA issuer waits for): TMEM -> registers, recombined to one double per
    // entry, then the accumulators are released; phase 2 (scaling, T stores, row dot) runs under the next tile's MMAs. =====
    const int quad = warp & 3, half = (warp - 2) >> 2, et = tid - 64;  // et: 0..255
    const int rloc = quad * 32 + lane;                                 // this thread's row inside the tile (= its TMEM lane)
    constexpr int HC = O8_BN / 2;                                      // columns per thread
    const bool need_k = !TRI && ((q != nullptr) || (du_part != nullptr));
    const int e_all = ea ? 0 : o8_exponent_of_scale(*a_scale);
    uint32_t acc_phase = 0;
    long long w_accfull = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int rb = tile / n_cb, cb = o8_rq_cb<TRI>(tile, rb, n_cb);
      const int row = rb * O8_BM + rloc;
      const int er = ea ? ((row < n_rb * O8_BM) ? ea[row] : 0) : e_all;
      // while the MMAs of this tile run: the K tile (row dot, column sums) and the column scales
      if (need_k) {
        if (Kmat) {
          for (int rr = et >> 5; rr < O8_BM; rr += 8) {  // one row (512 contiguous bytes) per warp instruction
            const int gr = rb * O8_BM + rr;
            double2 d = make_double2(0.0, 0.0);
            if (gr < n) d = *reinterpret_cast<const double2*>(Kmat + (long)gr * ldk + cb * O8_BN + 2 * lane);
            *reinterpret_cast<double2*>(sK + rr * O8_KLD + 2 * lane) = d;
          }
        } else {
          // rebuild the thread's 32 columns from the digit planes (= one k-step of the A block: two 16-byte halves)
          const double asc = (er == O8_POISON) ? __longlong_as_double(0x7FF8000000000000ll) : o8_pow2(er - O8_FRAC);
          const int8_t* ab = As + o8_a_offset((long)rb * O8_BM + rloc, cb * O8_BN + half * HC, nks);
#pragma unroll
          for (int h = 0; h < 2; ++h) {  // 16-column half of the k-step
            uint4 dg[O8_NS];
#pragma unroll
            for (int p = 0; p < O8_NS; ++p)
              dg[p] = *reinterpret_cast<const uint4*>(ab + (long)p * nks * O8_A_PLANE + h * (O8_BM * 16));
            double* dst = sK + rloc * O8_KLD + half * HC + h * 16;
#pragma unroll
            for (int g4 = 0; g4 < 4; ++g4) {
              uint32_t w[O8_NS];
#pragma unroll
              for (int p = 0; p < O8_NS; ++p) w[p] = g4 == 0 ? dg[p].x : g4 == 1 ? dg[p].y : g4 == 2 ? dg[p].z : dg[p].w;
#pragma unroll
              for (int c = 0; c < 4; c += 2)
                *reinterpret_cast<double2*>(dst + g4 * 4 + c) =
                    make_double2(o8_digits_to_double(w, c) * asc, o8_digits_to_double(w, c + 1) * asc);
            }
          }
        }
      }
      if (et < O8_BN) scol[et] = o8_scale_or_nan(eb[cb * O8_BN + et], 0);
      if (du_part && half == 0) sg[rloc] = (row < n) ? gvec[row] : 0.0;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (du_part && et < O8_BN) {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll 8
        for (int r = 0; r < O8_BM; r += 2) {
          a0 = fma(sg[r], sK[r * O8_KLD + et], a0);
          a1 = fma(sg[r + 1], sK[(r + 1) * O8_KLD + et], a1);
        }
        du_part[(long)rb * N + cb * O8_BN + et] = a0 + a1;
      }
      const long long c0 = dbg ? clock64() : 0;
      o8_mbar_wait(&acc_full, acc_phase);
      if (dbg) w_accfull += clock64() - c0;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // ---- phase 1: 7 x 32 accumulator columns of this row -> 32 doubles (exact integers, unscaled)
      double val[HC];
#pragma unroll
      for (int c0i = 0; c0i < HC; c0i += 8) {
        uint32_t g[O8_NS][8];
#pragma unroll
        for (int t = 0; t < O8_NS; ++t)
          o8_tmem_ld8(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(t * O8_BN + half * HC + c0i), g[t]);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 8; ++j) val[c0i + j] = o8_recombine(g, j);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) o8_mbar_arrive(&acc_empty);  // the next tile's MMAs may overwrite TMEM from here on
      acc_phase ^= 1;
      // ---- phase 2
      const double rs = o8_scale_or_nan(er, -36);  // 2^(e_i - 12 - 24)
      const double* krow = sK + rloc * O8_KLD + half * HC;
      const double* sc = scol + half * HC;
      double qsum = 0.0;
      if (row < n) {
        double* tp = WT ? T + (long)row * ldt + cb * O8_BN + half * HC : nullptr;
#pragma unroll
        for (int j = 0; j < HC; j += 2) {
          const double o0 = val[j] * rs * sc[j], o1 = val[j + 1] * rs * sc[j + 1];
          if (WT) *reinterpret_cast<double2*>(tp + j) = make_double2(o0, o1);
          if (TRI) {
            qsum = fma(o0, o0, qsum);
            qsum = fma(o1, o1, qsum);
          } else if (q) {
            const double2 kk = *reinterpret_cast<const double2*>(krow + j);
            qsum = fma(o0, kk.x, qsum);
            qsum = fma(o1, kk.y, qsum);
          }
        }
      }
      if (q && q_stride == 0 && row < n) atomicAdd(&q[row], qsum);
      if (q && q_stride > 0 && half == 1) sq[rloc] = qsum;
      asm volatile("bar.sync 1, 256;" ::: "memory");  // everyone is done with sK / scol / sg before the next tile overwrites them
      // (sq is rewritten only after the next tile's first barrier, which these readers pass first)
      if (q && q_stride > 0 && half == 0 && row < n) q[(long)cb * q_stride + row] = qsum + sq[rloc];
    }
    if (dbg && blockIdx.x == 0 && warp == 2 && lane == 0) dbg[4] = w_accfull;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// ---------------------------------------------------------------------------------------------------------------------
// Work decomposition of the SYRK.  Items = (row chunk, tile), chunk-major, a chunk being <= O8_MAX_SEG k-stages (int32
// exactness) -- CTAs that run at the same time work on the same rows of X, which therefore come from L2 (a first version
// that gave every CTA one contiguous range of the (tile, stage) space was DRAM bound: 6 GB of traffic instead of 0.56).
// Full waves of items go one item per CTA; the items of the last, partial wave ("stream-K" remainder) are cut into equal
// contiguous stage ranges so that all CTAs finish together (72 upper tiles x 9 chunks on 148 SMs: 4.38 waves cost 4.38,
// not 5).  Every segment ends in one FP64 partial tile, stored in slot cta * slots_per_cta + index.  The same iterator runs
// in all warp roles, in the finishing kernel (which adds a tile's segments in chunk / stage order: bitwise reproducible)
// and on the host (sizing).
// ---------------------------------------------------------------------------------------------------------------------
struct O8SegIter {
  int n_tiles, nks, spc, n_cta, cta;
  int n_items, full;     // items, full waves
  int wave;              // phase A cursor
  long posB, endB;       // phase B: range of this CTA in the remainder's (item, stage) space, stride spc per item
  // spc_ < 0: measurement switch, whole items only (the last wave stays partial, as before the remainder split)
  __host__ __device__ O8SegIter(int n_tiles_, int nks_, int spc_, int cta_, int n_cta_, bool remainder_only = false)
      : n_tiles(n_tiles_), nks(nks_), spc(spc_ < 0 ? -spc_ : spc_), n_cta(n_cta_), cta(cta_) {
    const int n_chunks = (nks + spc - 1) / spc;
    n_items = n_tiles * n_chunks;
    full = spc_ < 0 ? (n_items + n_cta - 1) / n_cta : n_items / n_cta;
    wave = remainder_only ? full : 0;
    long totalB = (long)(n_items - full * n_cta) * spc;
    if (totalB < 0) totalB = 0;
    const long LB = (totalB + n_cta - 1) / n_cta;
    posB = (long)cta * LB;
    endB = posB + LB < totalB ? posB + LB : totalB;
  }
  __host__ __device__ long remainder_share() const {
    long totalB = (long)(n_items - full * n_cta) * spc;
    if (totalB < 0) totalB = 0;
    const long lb = (totalB + n_cta - 1) / n_cta;
    return lb > 0 ? lb : 1;
  }
  __host__ __device__ bool next(int& tile, int& k0, int& k1) {
    while (wave < full && wave * n_cta + cta >= n_items) ++wave;  // (only with the measurement switch)
    if (wave < full) {
      const int item = wave * n_cta + cta;
      ++wave;
      const int chunk = item / n_tiles;
      tile = item - chunk * n_tiles;
      k0 = chunk * spc;
      k1 = k0 + spc < nks ? k0 + spc : nks;
      return true;
    }
    while (posB < endB) {
      const int j = (int)(posB / spc);
      const int item = full * n_cta + j;
      const int chunk = item / n_tiles;
      tile = item - chunk * n_tiles;
      const int kk = (int)(posB - (long)j * spc);
      const long item_end = (long)(j + 1) * spc;
      const long seg_end = item_end < endB ? item_end : endB;
      k0 = chunk * spc + kk;
      k1 = k0 + (int)(seg_end - posB);
      if (k1 > nks) k1 = nks;  // a shorter last chunk
      posB = seg_end;
      if (k1 > k0) return true;
    }
    return false;
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// SYRK partials: part[chunk][M x M] (upper 128 x 64 tiles) = X^T X over the rows of one chunk.
//   MN = true : row-layout planes of X itself (R x M), one matrix-wide scale (*x_scale); operands MN-major.  A stage holds
//               32 rows i of X: the A tile (128 columns j) and the B tile (64 columns) are 5-D TMA boxes (tmA, tmB) over
//               [8-byte words of a 2048-byte plane | 16-byte half | column k-step | digit | row block] that land in shared
//               memory as [digit][16-column group][4 core matrices of 8 rows x 16 bytes].
//   MN = false: Xs = transposed planes (operand rows = columns of X, o8_slice_t_kernel), per-column exponents ex; K-major.
// Work item = (chunk, tile), chunk-major so that the CTAs running together read the same rows (L2 reuse).
// ---------------------------------------------------------------------------------------------------------------------
template <bool MN, bool COLL>
__global__ void __launch_bounds__(O8_THREADS, 1)
o8_syrk_kernel(int M, int nks_total, int spc, int slots_per_cta, const int8_t* __restrict__ Xs, const int* __restrict__ ex,
               const double* __restrict__ x_scale, const double* __restrict__ uniform_count, double uniform_target,
               double* __restrict__ part, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB) {
  if (uniform_count && *uniform_count != uniform_target) return;  // unequal weights: handled by the correction kernels
  extern __shared__ __align__(1024) uint8_t o8_sm[];
  uint8_t* sA = o8_sm;
  uint8_t* sB = o8_sm + O8_SY_STAGES * O8_A_STAGE;
  __shared__ __align__(8) uint64_t full[O8_SY_STAGES], empty[O8_SY_STAGES], acc_full, acc_empty;
  __shared__ uint32_t tmem_base_s;
  __shared__ double scol[O8_BN];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_rb = M / O8_BM, n_cb = M / O8_BN;
  const int n_tiles = n_rb * n_cb - n_rb * (n_rb - 1);  // sum_rb (n_cb - 2 rb): tiles with cb >= 2 rb
  auto tile_rc = [&](int tl, int& rb, int& cb) {
    rb = 0;
    while (tl >= n_cb - 2 * rb) {
      tl -= n_cb - 2 * rb;
      ++rb;
    }
    cb = 2 * rb + tl;
  };

  if (tid == 0) {
    for (int s = 0; s < O8_SY_STAGES; ++s) {
      o8_mbar_init(&full[s], 1);
      o8_mbar_init(&empty[s], 1);
    }
    o8_mbar_init(&acc_full, 1);
    o8_mbar_init(&acc_empty, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(o8_smem(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_s;

  if (warp == 0) {
    // ===== producer =====
    int stage = 0;
    uint32_t phase = 0;
    O8SegIter it(n_tiles, nks_total, spc, blockIdx.x, gridDim.x);
    int tl, rb, cb, k0, k1;
    while (it.next(tl, k0, k1)) {
      tile_rc(tl, rb, cb);
      for (int ks = k0; ks < k1; ++ks) {
        o8_mbar_wait(&empty[stage], phase ^ 1);
        if (lane == 0) o8_mbar_expect_tx(&full[stage], O8_A_STAGE + O8_B_STAGE);
        __syncwarp();
        uint8_t* dA = sA + stage * O8_A_STAGE;
        uint8_t* dB = sB + stage * O8_B_STAGE;
        if (MN) {
          // rows ks*32 .. +31 of X = row block ks / 4, core-matrix rows (ks % 4) * 4 .. +3 = 8-byte words (ks % 4) * 64 .. +63
          // of every plane; box = (64 words, 2 halves, 4 | 2 column k-steps, 7 digits, 1 row block)
          if (lane == 0) o8_tma_5d(dA, &tmA, (ks & 3) * 64, 0, 4 * rb, 0, ks >> 2, &full[stage]);
          else if (lane == 1) o8_tma_5d(dB, &tmB, (ks & 3) * 64, 0, 2 * cb, 0, ks >> 2, &full[stage]);
        } else {
          // A: the seven digit planes of (row block rb, k-step ks), 4 KB each; B: 64 of the 128 rows of (block cb / 2): per
          // digit and 16-byte half one piece of 64 rows x 16 bytes
          if (lane < O8_NS)
            o8_bulk_g2s(dA + lane * O8_A_PLANE, Xs + (((long)rb * O8_NS + lane) * nks_total + ks) * O8_A_PLANE, O8_A_PLANE,
                        &full[stage]);
          else if (lane < 3 * O8_NS) {
            const int pp = lane - O8_NS, pd = pp >> 1, half = pp & 1;
            o8_bulk_g2s(dB + pp * (O8_BN * 16),
                        Xs + (((long)(cb >> 1) * O8_NS + pd) * nks_total + ks) * O8_A_PLANE + half * (O8_BM * 16) +
                            (cb & 1) * (O8_BN * 16),
                        O8_BN * 16, &full[stage]);
          }
        }
        if (++stage == O8_SY_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    const bool leader = o8_elect_one();
    uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(O8_BN >> 3) << 17) | ((uint32_t)(O8_BM >> 4) << 24);
    if (MN) idesc |= (1u << 15) | (1u << 16);
    // K-major: LBO = distance of the two 16-byte k halves, SBO = 128 (next 8 rows)
    // MN-major: LBO = 128 (next 8 contraction rows), SBO = 512 (next 16 operand rows)
    constexpr uint32_t kHi = ((MN ? 512u : 128u) >> 4) | (1u << 14);
    constexpr uint32_t lboA = MN ? 128u : (uint32_t)(O8_BM * 16), lboB = MN ? 128u : (uint32_t)(O8_BN * 16);
    int stage = 0;
    uint32_t phase = 0, acc_phase = 0;
    O8SegIter it(n_tiles, nks_total, spc, blockIdx.x, gridDim.x);
    int tl, k0, k1;
    while (it.next(tl, k0, k1)) {
      o8_mbar_wait(&acc_empty, acc_phase ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      for (int ks = k0; ks < k1; ++ks) {
        o8_mbar_wait(&full[stage], phase);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (leader) {
          const uint32_t a_lo = ((o8_smem(sA + stage * O8_A_STAGE) >> 4) & 0x3FFFu) | ((lboA >> 4) << 16);
          const uint32_t b_lo = ((o8_smem(sB + stage * O8_B_STAGE) >> 4) & 0x3FFFu) | ((lboB >> 4) << 16);
          o8_issue_kstep<COLL>(tmem, a_lo, kHi, 4096 >> 4, b_lo, kHi, 2048 >> 4, idesc, ks > k0 ? 1u : 0u);
          o8_commit(&empty[stage]);
        }
        __syncwarp();
        if (++stage == O8_SY_STAGES) { stage = 0; phase ^= 1; }
      }
      if (leader) o8_commit(&acc_full);
      __syncwarp();
      acc_phase ^= 1;
    }
  } else {
    const int quad = warp & 3, et = tid - 64;
    uint32_t acc_phase = 0;
    const int e_all = MN ? o8_exponent_of_scale(*x_scale) : 0;
    O8SegIter it(n_tiles, nks_total, spc, blockIdx.x, gridDim.x);
    int tl, rb, cb, k0, k1, seg = 0;
    while (it.next(tl, k0, k1)) {
      tile_rc(tl, rb, cb);
      const int rloc = quad * 32 + lane;
      const int row = rb * O8_BM + rloc;
      if (et < O8_BN) scol[et] = o8_scale_or_nan(MN ? e_all : ex[cb * O8_BN + et], 0);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      o8_mbar_wait(&acc_full, acc_phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const double rs = o8_scale_or_nan(MN ? e_all : ex[row], -36);
      double* prow = part + ((long)blockIdx.x * slots_per_cta + seg) * (O8_BM * O8_BN) + rloc * O8_BN;  // slot: 128 x 64 tile
      ++seg;
      for (int c0i = 0; c0i < O8_BN; c0i += 8) {
        uint32_t g[O8_NS][8];
#pragma unroll
        for (int t = 0; t < O8_NS; ++t)
          o8_tmem_ld8(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(t * O8_BN + c0i), g[t]);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 8; j += 2)
          *reinterpret_cast<double2*>(prow + c0i + j) =
              make_double2(o8_recombine(g, j) * rs * scol[c0i + j], o8_recombine(g, j + 1) * rs * scol[c0i + j + 1]);
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) o8_mbar_arrive(&acc_empty);
      acc_phase ^= 1;
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// one entry of a row-layout digit matrix (A-type planes) as a double, without the power-of-two scale
__device__ __forceinline__ double o8_entry(const int8_t* __restrict__ digits, int nks, int r, int k) {
  const int8_t* b = digits + o8_a_offset(r, k & ~15, nks) + (k & 15);
  long long y = 0;
#pragma unroll
  for (int p = 0; p < O8_NS; ++p) y = y * 256 + (long long)b[(long)p * nks * O8_A_PLANE];  // seven signed digits
  return (double)y;
}

// Out (symmetric) (+)= alpha * w0 * (sum of the tile's segment partials - sum_{i in skip} x_i x_i^T).  One CTA per upper
// 128 x 64 tile; the segments of the tile are found by re-running the CTAs' segment iterators (a handful of integer steps)
// and added in CTA / index order (bitwise reproducible).  skip (optional): rows whose weight is 0 instead of w0 (rows of the
// SVGP step whose predictive variance was clamped: their gradient is zero), rebuilt from the digit planes; normally empty.
__global__ void __launch_bounds__(256) o8_syrk_finish_kernel(int M, int nks_total, int spc, int n_cta, int slots_per_cta,
                                                             const double* __restrict__ part, double alpha,
                                                             const double* __restrict__ w0, const double* __restrict__ uniform_count,
                                                             double uniform_target, int accumulate, double* __restrict__ Out,
                                                             long ldo, const int* __restrict__ skip_count,
                                                             const int* __restrict__ skip_rows, const int8_t* __restrict__ digits,
                                                             const double* __restrict__ x_scale) {
  if (uniform_count && *uniform_count != uniform_target) return;
  const int n_rb = M / O8_BM, n_cb = M / O8_BN;
  const int n_tiles = n_rb * n_cb - n_rb * (n_rb - 1);
  const int tile = blockIdx.x;
  int rb = 0, tl = tile;
  while (tl >= n_cb - 2 * rb) {
    tl -= n_cb - 2 * rb;
    ++rb;
  }
  const int cb = 2 * rb + tl;
  constexpr int NSPLIT = 4;                           // CTAs per tile (blockIdx.y): 32 rows each
  constexpr int EPT = O8_BM * O8_BN / 256 / NSPLIT;   // elements per thread: e = e0 + threadIdx.x + 256 i (coalesced)
  const int e0 = blockIdx.y * (O8_BM * O8_BN / NSPLIT);
  double acc[EPT];
#pragma unroll
  for (int i = 0; i < EPT; ++i) acc[i] = 0.0;
  {
    const O8SegIter probe(n_tiles, nks_total, spc, 0, n_cta);
    const int aspc = probe.spc;  // (spc < 0 carries the measurement switch)
    const int n_chunks = (nks_total + aspc - 1) / aspc;
    const long LB = probe.remainder_share();
    for (int chunk = 0; chunk < n_chunks; ++chunk) {
      const int item = chunk * n_tiles + tile;
      if (item < probe.full * n_cta) {  // a full-wave item: one segment, owned by CTA item % n_cta as its (item / n_cta)-th
        const double* src = part + ((long)(item % n_cta) * slots_per_cta + item / n_cta) * (O8_BM * O8_BN) + e0 + threadIdx.x;
#pragma unroll
        for (int i = 0; i < EPT; ++i) acc[i] += src[256 * i];
        continue;
      }
      // an item of the remainder: its stages are spread over the CTAs c_first .. c_last
      const int j = item - probe.full * n_cta;
      const int c_first = (int)(((long)j * aspc) / LB), c_last = (int)((((long)j + 1) * aspc - 1) / LB);
      for (int c = c_first; c <= c_last && c < n_cta; ++c) {
        O8SegIter it(n_tiles, nks_total, spc, c, n_cta, true);
        int t2, k0, k1, idx = probe.full;
        while (it.next(t2, k0, k1)) {
          if (t2 == tile && k0 / aspc == chunk) {
            const double* src = part + ((long)c * slots_per_cta + idx) * (O8_BM * O8_BN) + e0 + threadIdx.x;
#pragma unroll
            for (int i = 0; i < EPT; ++i) acc[i] += src[256 * i];
          }
          ++idx;
        }
      }
    }
  }
  const int n_skip = skip_count ? *skip_count : 0;
  const double scale = alpha * (w0 ? w0[0] : 1.0);
#pragma unroll
  for (int i = 0; i < EPT; ++i) {
    const int e = e0 + threadIdx.x + 256 * i;
    const int r = rb * O8_BM + e / O8_BN, c = cb * O8_BN + e % O8_BN;
    if (c < r) continue;
    double s = acc[i];
    if (n_skip > 0) {
      const int ex = o8_exponent_of_scale(*x_scale);
      const double sc2 = o8_pow2(2 * (ex - O8_FRAC));
      double corr = 0.0;
      for (int t = 0; t < n_skip; ++t) {
        const int ii = skip_rows[t];
        corr = fma(o8_entry(digits, M / O8_KS, ii, r), o8_entry(digits, M / O8_KS, ii, c), corr);
      }
      s -= corr * sc2;
    }
    s *= scale;
    if (accumulate) {
      Out[(long)r * ldo + c] += s;
      if (c != r) Out[(long)c * ldo + r] += s;
    } else {
      Out[(long)r * ldo + c] = s;
      Out[(long)c * ldo + r] = s;
    }
  }
}

// out[j] = sum_b part[b * N + j] in a fixed order (column sums of the row-quadratic kernel's per-row-block partials).
// CTA = 32 columns x 8 row groups: thread (g, c) adds rows g, g + 8, ... (four independent chains), the eight groups are
// combined in index order through shared memory -- bitwise reproducible, and 32x more CTAs than one thread per column.
__global__ void __launch_bounds__(256) o8_sum_partials_kernel(int nb, int N, const double* __restrict__ part,
                                                              double* __restrict__ out) {
  __shared__ double sm[8][33];
  const int c = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + c;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  if (j < N) {
    int b = g;
    for (; b + 24 < nb; b += 32) {
      a0 += part[(long)b * N + j];
      a1 += part[(long)(b + 8) * N + j];
      a2 += part[(long)(b + 16) * N + j];
      a3 += part[(long)(b + 24) * N + j];
    }
    for (; b < nb; b += 8) a0 += part[(long)b * N + j];
  }
  sm[g][c] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (g == 0 && j < N) {
    double t = sm[0][c];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += sm[k][c];
    out[j] = t;
  }
}

static int g_o8_syrk_whole_items = 0;  // measurement switch (npgp_o8_set_syrk_split(0)): no split of the last partial wave

// Launch shape of the SYRK: CTAs, stages per row chunk and the largest number of segments any CTA produces (host run of the
// device iterator).  The chunk length is the largest that (i) keeps int32 exact (O8_MAX_SEG) and (ii) lets the rows a wave
// of CTAs works on (kNumSMs / n_tiles chunks) stay resident in L2 (~110 MB of the 126 MB): every extra chunk costs one
// more epilogue per CTA, too long a chunk turns the kernel DRAM bound.
static int o8_syrk_shape(int nks, int n_tiles, int M, int* n_cta_out, int* spc_out) {
  const double bytes_per_stage = (double)kNumSMs / n_tiles * O8_KS * (double)M * O8_NS;  // of the chunks in flight
  int max_spc = (int)(110e6 / bytes_per_stage);
  if (max_spc > O8_MAX_SEG) max_spc = O8_MAX_SEG;
  if (max_spc < 32) max_spc = 32;
  const int best_chunks = ceil_div(nks, max_spc);
  const int spc = ceil_div(nks, best_chunks);
  const long items = (long)n_tiles * ceil_div(nks, spc);
  const int n_cta = (int)(items < kNumSMs ? items : kNumSMs);
  int worst = 1;
  for (int c = 0; c < n_cta; ++c) {
    O8SegIter it(n_tiles, nks, g_o8_syrk_whole_items ? -spc : spc, c, n_cta);
    int t, k0, k1, cnt = 0;
    while (it.next(t, k0, k1)) ++cnt;
    if (cnt > worst) worst = cnt;
  }
  *n_cta_out = n_cta;
  *spc_out = g_o8_syrk_whole_items ? -spc : spc;
  return worst;
}

static inline int o8_syrk_tiles(int M) {
  const int n_rb = M / O8_BM, n_cb = M / O8_BN;
  return n_rb * n_cb - n_rb * (n_rb - 1);
}

}  // namespace npgp

using namespace npgp;

static long long* g_o8_dbg = nullptr;  // debugging aid only (npgp_rowquad_i8_debug); NULL in production
static int g_o8_collector = 1;         // measurement switch (npgp_o8_set_collector)

// debugging aid: device buffer of 8 counters filled by CTA 0 (cycles the producer / MMA issuer / epilogue spend waiting)
extern "C" void npgp_rowquad_i8_debug(long long* dev_counters) { g_o8_dbg = dev_counters; }
// measurement switch: 1 (default) = A-operand collector reuse hints on the digit products, 0 = plain MMAs
extern "C" int npgp_o8_set_collector(int on) {
  g_o8_collector = on ? 1 : 0;
  return NPGP_OK;
}

// measurement switch: 1 (default) = the items of the last partial wave of the SYRK are split evenly over the CTAs, 0 = whole items
extern "C" int npgp_o8_set_syrk_split(int on) {
  g_o8_syrk_whole_items = on ? 0 : 1;
  return NPGP_OK;
}

extern "C" long npgp_o8_digits_bytes(int rows, int Kd, int block_rows) {
  if (rows < 0 || Kd < 0 || (block_rows != O8_BM && block_rows != O8_BN)) return -1;
  return o8_digits_bytes(rows, Kd, block_rows);
}

// Digit planes (row layout, block_rows = 128 for an A operand / 64 for the symmetric B operand) and per-row exponents of an
// arbitrary FP64 matrix X (R x Kd); expo has ceil(R / block_rows) * block_rows entries.  Kd % 32 == 0.
extern "C" int npgp_o8_slice_rows(int R, int Kd, const double* X, long ldx, int block_rows, void* digits, int* expo,
                                  cudaStream_t stream) {
  if (R < 0 || Kd < 0 || (block_rows != O8_BM && block_rows != O8_BN)) return NPGP_EINVAL;
  if (R == 0 || Kd == 0) return NPGP_OK;
  if (!X || !digits || !expo) return NPGP_EINVAL;
  if (Kd % O8_KS || (ldx & 1) || (reinterpret_cast<uintptr_t>(X) & 15)) return NPGP_EUNSUPPORTED;
  const long rpad = ((long)R + block_rows - 1) / block_rows * block_rows;
  if (block_rows == O8_BM)
    o8_slice_rows_kernel<O8_BM><<<(unsigned)(rpad / 8), 512, 0, stream>>>(R, (int)rpad, Kd, X, ldx, (int8_t*)digits, expo);
  else
    o8_slice_rows_kernel<O8_BN><<<(unsigned)(rpad / 8), 512, 0, stream>>>(R, (int)rpad, Kd, X, ldx, (int8_t*)digits, expo);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

// T = K C, q, column sums from ready-made digit planes.
//   a_digits / a_expo: A operand (n x M); a_expo NULL -> one matrix-wide exponent from the positive device scalar *a_scale
//   c_digits / c_expo: symmetric C (M x M, block_rows 64)
//   Kmat (optional): FP64 K for the row dot; NULL -> rebuilt from the digits
//   T (optional when q is given): NULL -> only the row dot is formed (bitwise the q of a run with T), no T stores
//   q (optional): q_stride == 0 -> q[i] += (atomics; zeroed by the caller); q_stride >= n -> q[cb * q_stride + i] = partial of
//                 column block cb (M / 64 blocks, plain stores: deterministic)
//   gvec / du_part (optional, both or none): du_part[rb * M + j] = sum over the rows of row block rb of gvec_i K_ij
template <bool COLL, bool WT, bool TRI = false>
static int o8_rowquad_launch(int n, int N, int Kd, const void* a_digits, const int* a_expo, const double* a_scale,
                             const void* c_digits, const int* c_expo, const double* Kmat, long ldk, double* T, long ldt,
                             double* q, long q_stride, const double* gvec, double* du_part, cudaStream_t stream,
                             int ms_ks = 0) {
  const long npad = ((long)n + O8_BM - 1) / O8_BM * O8_BM;
  const long tiles = npad / O8_BM * (N / O8_BN);
  const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
  NPGP_CUDA(cudaFuncSetAttribute(o8_rowquad_kernel<COLL, WT, TRI>, cudaFuncAttributeMaxDynamicSharedMemorySize, O8_RQ_SMEM));
  o8_rowquad_kernel<COLL, WT, TRI><<<grid, O8_RQ_THREADS, O8_RQ_SMEM, stream>>>(
      n, N, Kd, (const int8_t*)a_digits, a_expo, a_scale, (const int8_t*)c_digits, c_expo, Kmat, ldk, T, ldt, q, q_stride, gvec,
      du_part, g_o8_dbg, ms_ks);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

extern "C" int npgp_o8_rowquad_digits(int n, int M, const void* a_digits, const int* a_expo, const double* a_scale,
                                      const void* c_digits, const int* c_expo, const double* Kmat, long ldk, double* T,
                                      long ldt, double* q, long q_stride, const double* gvec, double* du_part,
                                      cudaStream_t stream) {
  if (n < 0 || M < 0) return NPGP_EINVAL;
  if (n == 0 || M == 0) return NPGP_OK;
  if (!a_digits || (!a_expo && !a_scale) || !c_digits || !c_expo || (!T && !q)) return NPGP_EINVAL;
  if ((gvec == nullptr) != (du_part == nullptr)) return NPGP_EINVAL;
  if (M % O8_BN || M > O8_MAX_KD || (T && ((ldt & 1) || (reinterpret_cast<uintptr_t>(T) & 15))) ||
      (Kmat && ((ldk & 1) || (reinterpret_cast<uintptr_t>(Kmat) & 15))) || (q_stride != 0 && q_stride < n))
    return NPGP_EUNSUPPORTED;
#define NPGP_RQ(COLL, WT) \
  o8_rowquad_launch<COLL, WT>(n, M, M, a_digits, a_expo, a_scale, c_digits, c_expo, Kmat, ldk, T, ldt, q, q_stride, gvec, \
                              du_part, stream)
  int rc;
  if (T) rc = g_o8_collector ? NPGP_RQ(true, true) : NPGP_RQ(false, true);
  else rc = g_o8_collector ? NPGP_RQ(true, false) : NPGP_RQ(false, false);
#undef NPGP_RQ
  return rc;
}

// T (n x N) = A B^T from planes: A (n x Kd, block_rows 128; a_expo NULL -> matrix-wide exponent from *a_scale), B (N x Kd,
// block_rows 64, per-row exponents b_expo = per-column scales of T).  The row-quadratic kernel with T stored and neither the
// row dot nor the column sums: its output width N and contraction length Kd are independent.
extern "C" int npgp_o8_gemm_digits(int n, int N, int Kd, const void* a_digits, const int* a_expo, const double* a_scale,
                                   const void* b_digits, const int* b_expo, double* T, long ldt, cudaStream_t stream) {
  if (n < 0 || N < 0 || Kd < 0) return NPGP_EINVAL;
  if (n == 0 || N == 0) return NPGP_OK;
  if (!a_digits || (!a_expo && !a_scale) || !b_digits || !b_expo || !T) return NPGP_EINVAL;
  if (N % O8_BN || Kd == 0 || Kd % O8_KS || Kd > O8_MAX_KD || ldt < N || (ldt & 1) || (reinterpret_cast<uintptr_t>(T) & 15))
    return NPGP_EUNSUPPORTED;
  if (g_o8_collector)
    return o8_rowquad_launch<true, true>(n, N, Kd, a_digits, a_expo, a_scale, b_digits, b_expo, nullptr, 0, T, ldt, nullptr,
                                         0, nullptr, nullptr, stream);
  return o8_rowquad_launch<false, true>(n, N, Kd, a_digits, a_expo, a_scale, b_digits, b_expo, nullptr, 0, T, ldt, nullptr, 0,
                                        nullptr, nullptr, stream);
}

// q[cb * q_stride + i] = sum_{j in column block cb} (A B^T)_ij^2 from planes, B (N x Kd, block_rows 64, per-row exponents)
// lower triangular: block cb contracts over k < 64 (cb + 1) only, and from k = Ms on when 64 cb >= Ms (Ms > 0: B is
// block diagonal with its split at column Ms < Kd).  The skipped k-steps of B are never read.  T is never stored.
extern "C" int npgp_o8_trinorm_digits(int n, int N, int Kd, int Ms, const void* a_digits, const int* a_expo,
                                      const double* a_scale, const void* b_digits, const int* b_expo, double* q, long q_stride,
                                      cudaStream_t stream) {
  if (n < 0 || N < 0 || Kd <= 0 || !a_digits || (!a_expo && !a_scale) || !b_digits || !b_expo || !q) return NPGP_EINVAL;
  if (N % O8_BN || Kd % O8_KS || Kd > O8_MAX_KD || Ms < 0 || Ms % O8_BN || (Ms > 0 && Ms >= Kd) || q_stride < n)
    return NPGP_EINVAL;
  if (n == 0 || N == 0) return NPGP_OK;
  if (g_o8_collector)
    return o8_rowquad_launch<true, false, true>(n, N, Kd, a_digits, a_expo, a_scale, b_digits, b_expo, nullptr, 0, nullptr,
                                                0, q, q_stride, nullptr, nullptr, stream, Ms / O8_KS);
  return o8_rowquad_launch<false, false, true>(n, N, Kd, a_digits, a_expo, a_scale, b_digits, b_expo, nullptr, 0, nullptr, 0,
                                               q, q_stride, nullptr, nullptr, stream, Ms / O8_KS);
}

// out[j] = sum_b part[b * N + j], b in index order (e.g. du from the du_part of npgp_o8_rowquad_digits, nb = ceil(n / 128))
extern "C" int npgp_o8_sum_partials(int nb, int N, const double* part, double* out, cudaStream_t stream) {
  if (nb < 0 || N < 0) return NPGP_EINVAL;
  if (N == 0) return NPGP_OK;
  if (!part || !out) return NPGP_EINVAL;
  o8_sum_partials_kernel<<<ceil_div(N, 32), 256, 0, stream>>>(nb, N, part, out);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

// ---- general-operand wrappers (contract of round 1's npgp_rowquad_i8 family) -----------------------------------------
// workspace: A digits (ceil(n/128)*128 x M x 7 bytes) + C digits (M x M x 7) + exponents (int per padded row / column)
extern "C" long npgp_rowquad_i8_workspace_bytes(int n, int M) {
  const long npad = ((long)n + O8_BM - 1) / O8_BM * O8_BM;
  return npad * M * O8_NS + (long)M * M * O8_NS + (npad + M) * (long)sizeof(int) + 1024;
}

static int rowquad_i8_impl(int n, int M, const double* K, long ldk, const double* C, long ldc, double* T, long ldt, double* q,
                           void* work, long work_bytes, cudaStream_t stream, bool slice, bool gemm) {
  if (n < 0 || M < 0) return NPGP_EINVAL;
  if (n == 0 || M == 0) return NPGP_OK;
  if (!K || !work || (slice && !C) || (gemm && !T)) return NPGP_EINVAL;
  if (M % O8_BN || M > O8_MAX_KD) return NPGP_EUNSUPPORTED;
  if (work_bytes < npgp_rowquad_i8_workspace_bytes(n, M)) return NPGP_EWORKSPACE;
  const long npad = ((long)n + O8_BM - 1) / O8_BM * O8_BM;
  int8_t* As = static_cast<int8_t*>(work);
  int8_t* Bs = As + npad * M * O8_NS;
  int* ea = reinterpret_cast<int*>(Bs + (long)M * M * O8_NS);
  int* eb = ea + npad;
  if (slice) {
    int rc = npgp_o8_slice_rows(n, M, K, ldk, O8_BM, As, ea, stream);
    if (rc) return rc;
    rc = npgp_o8_slice_rows(M, M, C, ldc, O8_BN, Bs, eb, stream);
    if (rc) return rc;
  }
  if (!gemm) return NPGP_OK;
  return npgp_o8_rowquad_digits(n, M, As, ea, nullptr, Bs, eb, K, ldk, T, ldt, q, 0, nullptr, nullptr, stream);
}

// T (n x M) = K (n x M) @ C (M x M, symmetric);  q[i] += sum_j T_ij K_ij (q zeroed by the caller; NULL to skip).
// M must be a multiple of 64 (and <= 16384).  Replaces npgp_rowquad on the integer tensor-core path.
extern "C" int npgp_rowquad_i8(int n, int M, const double* K, long ldk, const double* C, long ldc, double* T, long ldt,
                               double* q, void* work, long work_bytes, cudaStream_t stream) {
  return rowquad_i8_impl(n, M, K, ldk, C, ldc, T, ldt, q, work, work_bytes, stream, true, true);
}
// The slicing passes alone (K and C into `work`); follow with npgp_rowquad_i8_gemm_only.
extern "C" int npgp_rowquad_i8_slice_only(int n, int M, const double* K, long ldk, const double* C, long ldc, void* work,
                                          long work_bytes, cudaStream_t stream) {
  return rowquad_i8_impl(n, M, K, ldk, C, ldc, nullptr, 0, nullptr, work, work_bytes, stream, true, false);
}
// The tensor-core kernel alone, on the digit planes a previous call with the same shapes left in `work`.
extern "C" int npgp_rowquad_i8_gemm_only(int n, int M, const double* K, long ldk, double* T, long ldt, double* q, void* work,
                                         long work_bytes, cudaStream_t stream) {
  return rowquad_i8_impl(n, M, K, ldk, nullptr, 0, T, ldt, q, work, work_bytes, stream, false, true);
}

// ---- SYRK ------------------------------------------------------------------------------------------------------------
// bytes of the partial-sum workspace of npgp_o8_syrk_digits for n contraction rows
extern "C" long npgp_o8_syrk_part_bytes(int n, int M) {
  if (n <= 0 || M <= 0 || M % O8_BM) return 0;
  int n_cta, spc;
  const int nks = ceil_div(((long)n + O8_BM - 1) / O8_BM * O8_BM, O8_KS);
  const int slots = o8_syrk_shape(nks, o8_syrk_tiles(M), M, &n_cta, &spc);
  return (long)n_cta * slots * (O8_BM * O8_BN) * (long)sizeof(double);
}

// 5-D tensor map over the A-type digit planes of X (n_rb row blocks x M columns) for the MN-major SYRK tiles, in units of
// 8-byte words: [256 words of a 2048-byte plane | 2 halves | M/32 column k-steps | 7 digits | n_rb row blocks];
// box = (64 words = 32 rows, 2, box_ksteps, 7, 1).  The encoder lives in the driver: fetched once per process.
typedef CUresult (*o8_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int o8_make_syrk_map(CUtensorMap* tm, const int8_t* digits, int M, int n_rb, int box_ksteps) {
  static o8_encode_fn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    NPGP_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !fn) return NPGP_EUNSUPPORTED;
    encode = reinterpret_cast<o8_encode_fn>(fn);
  }
  const cuuint64_t nks = (cuuint64_t)(M / O8_KS);
  const cuuint64_t dims[5] = {256, 2, nks, (cuuint64_t)O8_NS, (cuuint64_t)n_rb};
  const cuuint64_t strides[4] = {2048, (cuuint64_t)O8_A_PLANE, nks * O8_A_PLANE, (cuuint64_t)O8_NS * nks * O8_A_PLANE};  // bytes, dims 1..4
  const cuuint32_t box[5] = {64, 2, (cuuint32_t)box_ksteps, (cuuint32_t)O8_NS, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult r = encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, const_cast<int8_t*>(digits), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? NPGP_OK : NPGP_EUNSUPPORTED;
}

template <bool MN>
static int o8_syrk_launch(int M, int nks, const int8_t* Xs, const int* ex, const double* x_scale, double alpha,
                          const double* w0_dev, const double* uniform_count, double uniform_target, int accumulate,
                          double* Out, long ldo, double* part, const int* skip_count, const int* skip_rows,
                          cudaStream_t stream) {
  NPGP_CUDA(cudaFuncSetAttribute(o8_syrk_kernel<MN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, O8_SY_SMEM));
  NPGP_CUDA(cudaFuncSetAttribute(o8_syrk_kernel<MN, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, O8_SY_SMEM));
  CUtensorMap tmA, tmB;
  memset(&tmA, 0, sizeof(tmA));
  memset(&tmB, 0, sizeof(tmB));
  if (MN) {
    int rc = o8_make_syrk_map(&tmA, Xs, M, nks / 4, 4);
    if (rc) return rc;
    rc = o8_make_syrk_map(&tmB, Xs, M, nks / 4, 2);
    if (rc) return rc;
  }
  const int n_tiles = o8_syrk_tiles(M);
  int grid, spc;
  const int slots = o8_syrk_shape(nks, n_tiles, M, &grid, &spc);
  if (g_o8_collector)
    o8_syrk_kernel<MN, true><<<grid, O8_THREADS, O8_SY_SMEM, stream>>>(M, nks, spc, slots, Xs, ex, x_scale, uniform_count,
                                                                      uniform_target, part, tmA, tmB);
  else
    o8_syrk_kernel<MN, false><<<grid, O8_THREADS, O8_SY_SMEM, stream>>>(M, nks, spc, slots, Xs, ex, x_scale, uniform_count,
                                                                       uniform_target, part, tmA, tmB);
  NPGP_LAUNCH_CHECK();
  o8_syrk_finish_kernel<<<dim3(n_tiles, 4), 256, 0, stream>>>(M, nks, spc, grid, slots, part, alpha, w0_dev, uniform_count, uniform_target,
                                                     accumulate, Out, ldo, skip_count, skip_rows, MN ? Xs : nullptr, x_scale);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

// Out (M x M, symmetric) (+)= alpha * w0 * X^T X from the ROW-layout digit planes of X (n x M, rows padded to 128 with zero
// digits, one matrix-wide scale *x_scale): the planes the Gibbs tile kernels emit, read MN-major.  M % 128 == 0.
// skip_count / skip_rows (optional, device): *skip_count row indices whose contribution x_i x_i^T is removed again (rows with
// weight 0 instead of w0).  part: npgp_o8_syrk_part_bytes(n, M) bytes.
extern "C" int npgp_o8_syrk_digits(int n, int M, const void* x_digits, const double* x_scale, double alpha,
                                   const double* w0_dev, const int* skip_count, const int* skip_rows, int accumulate,
                                   double* Out, long ldo, void* part, long part_bytes, cudaStream_t stream) {
  if (n < 0 || M < 0 || ((skip_count != nullptr) != (skip_rows != nullptr))) return NPGP_EINVAL;
  if (M == 0) return NPGP_OK;
  if (!Out || !x_digits || !x_scale || !part) return NPGP_EINVAL;
  if (M % O8_BM) return NPGP_EUNSUPPORTED;
  if (n == 0) {
    if (!accumulate) NPGP_CUDA(cudaMemset2DAsync(Out, sizeof(double) * ldo, 0, sizeof(double) * M, M, stream));
    return NPGP_OK;
  }
  if (part_bytes < npgp_o8_syrk_part_bytes(n, M)) return NPGP_EWORKSPACE;
  const int nks = ceil_div(((long)n + O8_BM - 1) / O8_BM * O8_BM, O8_KS);
  return o8_syrk_launch<true>(M, nks, (const int8_t*)x_digits, nullptr, x_scale, alpha, w0_dev, nullptr, 0.0, accumulate,
                              Out, ldo, (double*)part, skip_count, skip_rows, stream);
}

// general operands: transposed planes (M x ceil(n/128)*128 x 7 bytes) + column maxima + exponents + chunk partials
extern "C" long npgp_syrk_i8_workspace_bytes(int n, int M) {
  const long npad = ((long)n + O8_BM - 1) / O8_BM * O8_BM;
  return npad * M * O8_NS + (long)M * (sizeof(unsigned long long) + sizeof(int)) + 1024 + npgp_o8_syrk_part_bytes(n, M);
}

static int syrk_i8_impl(int n, int M, double alpha, const double* K, long ldk, const double* w0_dev,
                        const double* uniform_count, double uniform_target, int accumulate, int phase, double* Out, long ldo,
                        void* work, long work_bytes, const double* colw, double* colwsum, cudaStream_t stream) {
  if (n < 0 || M < 0) return NPGP_EINVAL;
  if (M == 0) return NPGP_OK;
  if ((phase != 1 && !Out) || (n > 0 && !K) || !work || phase < 0 || phase > 2) return NPGP_EINVAL;
  if (M % O8_BM) return NPGP_EUNSUPPORTED;
  if (work_bytes < npgp_syrk_i8_workspace_bytes(n, M)) return NPGP_EWORKSPACE;
  const long npad = ((long)n + O8_BM - 1) / O8_BM * O8_BM;
  const int nks = (int)(npad / O8_KS);
  int8_t* Xs = static_cast<int8_t*>(work);
  unsigned long long* cmax = reinterpret_cast<unsigned long long*>(Xs + npad * M * O8_NS);
  int* ex = reinterpret_cast<int*>(cmax + M);
  double* part = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(ex + M) + 1023) & ~(uintptr_t)1023);
  if (colwsum) NPGP_CUDA(cudaMemsetAsync(colwsum, 0, sizeof(double) * M, stream));
  if (n == 0) {
    if (phase != 1 && !accumulate) NPGP_CUDA(cudaMemset2DAsync(Out, sizeof(double) * ldo, 0, sizeof(double) * M, M, stream));
    return NPGP_OK;
  }
  if (phase != 2) {
    NPGP_CUDA(cudaMemsetAsync(cmax, 0, sizeof(unsigned long long) * M, stream));
    const int rows_per_cta = 256;
    dim3 grid(ceil_div(M, 256), ceil_div(n, rows_per_cta));
    o8_colmax_kernel<<<grid, 256, 0, stream>>>(n, M, K, ldk, rows_per_cta, cmax, colw, colwsum);
    NPGP_LAUNCH_CHECK();
    o8_exp_from_max_kernel<<<ceil_div(M, 256), 256, 0, stream>>>(M, cmax, ex);
    NPGP_LAUNCH_CHECK();
    dim3 gs(nks, M / O8_BM);
    o8_slice_t_kernel<<<gs, 256, 0, stream>>>(n, M, K, ldk, ex, Xs);
    NPGP_LAUNCH_CHECK();
  }
  if (phase == 1) return NPGP_OK;
  return o8_syrk_launch<false>(M, nks, Xs, ex, nullptr, alpha, w0_dev, uniform_count, uniform_target, accumulate, Out, ldo,
                               part, nullptr, nullptr, stream);
}

// Out (M x M, symmetric) = alpha * w0 * K^T K with w0 = *w0_dev (NULL: 1), K (n x M) arbitrary FP64; M % 128 == 0.
// uniform_count / uniform_target (optional): device-side gate (see npgp_wsyrk_hint); accumulate != 0: add to Out.
// phase: 0 = slice K and run; 1 = slicing passes only; 2 = tensor-core kernel only, on the planes a phase-1 call left in work.
extern "C" int npgp_syrk_i8(int n, int M, double alpha, const double* K, long ldk, const double* w0_dev,
                            const double* uniform_count, double uniform_target, int accumulate, int phase, double* Out,
                            long ldo, void* work, long work_bytes, cudaStream_t stream) {
  return syrk_i8_impl(n, M, alpha, K, ldk, w0_dev, uniform_count, uniform_target, accumulate, phase, Out, ldo, work,
                      work_bytes, nullptr, nullptr, stream);
}

// The slicing passes of npgp_syrk_i8 (phase 1) with the weighted column sums wsum[j] = sum_i w_i K_ij (overwritten) fused
// into the column-maximum pass.
extern "C" int npgp_syrk_i8_prepare(int n, int M, const double* K, long ldk, const double* w, double* wsum, void* work,
                                    long work_bytes, cudaStream_t stream) {
  if ((w == nullptr) != (wsum == nullptr)) return NPGP_EINVAL;
  return syrk_i8_impl(n, M, 1.0, K, ldk, nullptr, nullptr, 0.0, 0, 1, nullptr, 0, work, work_bytes, w, wsum, stream);
}
