// FP64 tensor-core contractions (DMMA.8x8x4 through mma.sync.m8n8k4.f64 -- tcgen05 has no FP64 kind on sm_100a).
//
//   npgp_dgemm    C = alpha op(A) op(B) + beta C            (row-major, triangular-operand / triangular-output skipping)
//   npgp_rowquad  T = K C,  q_i = sum_j T_ij K_ij           (whitened-SVGP predictive variance term, fused row-dot)
//   npgp_wsyrk    Out = K^T diag(w) K                       (dL/dC of the SVGP ELBO, SGPR Phi = Kzx Kxz), split over rows
//
// These replace the cuBLAS/MAGMA calls GPyTorch issues for  A = L^-1 Kzx,  A^T (S - I) A  and  Kzx Kxz
// (reference models/gibbs_kernels.py:222-232 via LowRankRootLazyTensor; models/dgps.py:25-35 via VariationalStrategy).
//
// Tiling (templated, measured on B200, see profiles/): BK = 16, 3-stage cp.async pipeline, 32x32 warp tiles (32
// accumulator doubles per thread).  Default: 64x64 CTA tile, 4 warps per CTA, 3-4 CTAs resident per SM, so that one CTA's
// barrier / producer phase is covered by the others' DMMA streams (34.3 TF/s = 93 % of the DMMA peak at C2; the
// 128x64 / 8-warp / 2-CTA variant reaches 32.2, the 128x128 / 1-CTA variant 29.9; cuBLAS 35.2).  Shared-memory tiles are stored either K-contiguous [rows][16+4] or MN-contiguous
// [16][cols+4], whichever matches the operand's global layout; with a leading dimension = 4 (mod 16) doubles both
// fragment-load patterns are bank-conflict free for 64-bit accesses.  Chunk addresses are computed once per CTA; the
// per-stage producer work is a pointer bump (plus a byte count at ragged edges).
#include <cstdlib>
#include "common.cuh"

namespace npgp {


__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

struct GemmParams {
  int M, N, K;
  const double* A;
  long lda;
  const double* B;
  long ldb;
  double* C;
  long ldc;
  double alpha, beta;
  int tri_a, tri_b;  // structure of op(A) (M x K) / op(B) (K x N): 0 dense, 1 lower (col <= row), 2 upper (col >= row)
  int out_tri;       // 0 all tiles, 1 only tiles touching the lower triangle, 2 only the upper
  int splits;        // split-K factor (gridDim.z); > 1 => atomicAdd epilogue, C must be pre-scaled by the caller
  const double* w;   // optional weights along K (scales op(A)[m][k] by w[k])
  const double* w_uniform_count;  // optional device scalar: if *w_uniform_count == w_uniform_target every weight equals
  double w_uniform_target;        //   w[0], so the kernel skips the per-fragment multiplies and scales the epilogue
  int weighted_only;              // launch only the weighted instantiation (the equal-weights case is handled elsewhere)
  const double* dotK;  // optional: q[row] += sum_col acc[row][col] * dotK[row][col]
  long lddot;
  double* q;
};

// One operand tile of TR "rows" (the M or N extent) x BK, loaded with 16-byte cp.async.  A thread owns PASSES chunks
// that differ by a uniform stride, so the steady-state producer work per stage is PASSES cp.async + one pointer bump;
// only edge tiles and the ragged last k-step take the predicated path.
template <int TR, int BK, bool KCONTIG, int GEMM_THREADS>
struct TileLoader {
  static constexpr int LDS_K = BK + 4;                      // K-contiguous tile: [TR][BK+4], = 4 (mod 16)
  static constexpr int LDMN = TR + 4;                       // MN-contiguous tile: [BK][TR+4], = 4 (mod 16)
  static constexpr int TILE = KCONTIG ? TR * LDS_K : BK * LDMN;
  static constexpr int PASSES = TR * BK / 2 / GEMM_THREADS;  // 16-byte chunks per thread
  static constexpr int CPL = KCONTIG ? BK / 2 : TR / 2;      // chunks per tile line
  static constexpr int LPP = GEMM_THREADS / CPL;             // tile lines covered per pass
  static constexpr int SPASS = LPP * (KCONTIG ? LDS_K : LDMN);  // smem doubles between passes
  const double* g;    // this thread's chunk of pass 0, at the current stage
  const double* g0;   // operand base (always a valid address)
  long pass_stride;   // global elements between passes
  long stage_stride;  // global elements between stages
  int soff;           // smem offset (doubles) of pass 0
  int line, pos;      // tile line (row for K-contig, k for MN-contig) and position (k resp. column) of pass 0
  int r0, nrows;

  __device__ __forceinline__ void init(const double* __restrict__ G, long ld, int r0_, int nrows_, int kb) {
    line = threadIdx.x / CPL;
    pos = (threadIdx.x % CPL) * 2;
    r0 = r0_;
    nrows = nrows_;
    g0 = G;
    if (KCONTIG) {
      g = G + (long)(r0 + line) * ld + kb + pos;
      pass_stride = (long)LPP * ld;
      stage_stride = BK;
      soff = line * LDS_K + pos;
    } else {
      g = G + (long)(kb + line) * ld + r0 + pos;
      pass_stride = (long)LPP * ld;
      stage_stride = (long)BK * ld;
      soff = line * LDMN + pos;
    }
  }
  __device__ __forceinline__ void load_fast(double* s) {
#pragma unroll
    for (int it = 0; it < PASSES; ++it) cp_async16(s + soff + it * SPASS, g + it * pass_stride, 16);
    g += stage_stride;
  }
  // predicated variant: k0 = absolute k of this stage, kend = exclusive bound of valid k
  __device__ __forceinline__ void load_edge(double* s, int k0, int kend) {
#pragma unroll
    for (int it = 0; it < PASSES; ++it) {
      int bytes;
      if (KCONTIG) {
        const bool row_ok = (r0 + line + it * LPP) < nrows;
        bytes = row_ok ? max(0, min(2, kend - (k0 + pos))) * 8 : 0;
      } else {
        const bool k_ok = (k0 + line + it * LPP) < kend;
        bytes = k_ok ? max(0, min(2, nrows - (r0 + pos))) * 8 : 0;
      }
      cp_async16(s + soff + it * SPASS, bytes ? g + it * pass_stride : g0, bytes);
    }
    g += stage_stride;
  }
};

template <int BM, int BN, int WM, int WN, int BK, int STAGES, bool A_KCONTIG, bool B_KCONTIG, bool HAS_W, int MINB,
          int GEMM_THREADS>
__global__ void __launch_bounds__(GEMM_THREADS, MINB) dgemm_kernel(GemmParams p) {
  using LA = TileLoader<BM, BK, A_KCONTIG, GEMM_THREADS>;
  using LB = TileLoader<BN, BK, B_KCONTIG, GEMM_THREADS>;
  constexpr int STAGE_DOUBLES = LA::TILE + LB::TILE + BK;
  constexpr int MT = WM / 8, NT = WN / 8;
  constexpr int WARPS_N = BN / WN;
  static_assert((BM / WM) * WARPS_N == GEMM_THREADS / 32, "warp grid must cover the CTA tile");
  extern __shared__ __align__(16) double smem[];
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  if (p.out_tri == 1 && n0 > m0 + BM - 1) return;
  if (p.out_tri == 2 && n0 + BN - 1 < m0) return;

  // k-range of this tile: triangular operands, then split-K
  int kb = 0, ke = p.K;
  if (p.tri_a == 1) ke = min(ke, m0 + BM);   // op(A) lower: k <= m
  if (p.tri_a == 2) kb = max(kb, m0);        // op(A) upper: k >= m
  if (p.tri_b == 1) kb = max(kb, n0);        // op(B) lower: k >= n   (row index k, col index n)
  if (p.tri_b == 2) ke = min(ke, n0 + BN);   // op(B) upper: k <= n
  kb = (kb / BK) * BK;
  if (p.splits > 1) {
    const int span = ke - kb;
    int per = (span + p.splits - 1) / p.splits;
    per = ((per + BK - 1) / BK) * BK;
    const int b2 = kb + (int)blockIdx.z * per;
    ke = min(ke, b2 + per);
    kb = b2;
  }
  const int nk = (ke > kb) ? (ke - kb + BK - 1) / BK : 0;
  if (nk == 0 && p.splits > 1) return;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t4 = lane & 3;
  const int wm0 = (warp / WARPS_N) * WM, wn0 = (warp % WARPS_N) * WN;
  // Device-side weight hint: the launcher enqueues BOTH instantiations; the unweighted one runs when the flag says that
  // all weights are equal (w[0] folded into the epilogue), the weighted one otherwise; the other exits here.
  constexpr bool w_uniform = false;
  double alpha_eff = p.alpha;
  if (p.w_uniform_count) {
    const bool uni = (*p.w_uniform_count == p.w_uniform_target);
    if (HAS_W ? uni : !uni) return;
    if (!HAS_W) alpha_eff *= p.w[0];
  }

  double acc[MT][NT][2];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  LA la;
  LB lb;
  la.init(p.A, p.lda, m0, p.M, kb);
  lb.init(p.B, p.ldb, n0, p.N, kb);
  const bool full_mn = (m0 + BM <= p.M) && (n0 + BN <= p.N);
  const int nk_fast = full_mn ? (ke - kb) / BK : 0;  // stages that need no predicate at all

  // stages are issued strictly in order (0, 1, 2, ...), so the loaders just advance their pointers
  auto load_stage = [&](int idx) {
    double* sA = smem + (idx % STAGES) * STAGE_DOUBLES;
    double* sB = sA + LA::TILE;
    if (idx < nk_fast) {
      la.load_fast(sA);
      lb.load_fast(sB);
    } else {
      la.load_edge(sA, kb + idx * BK, ke);
      lb.load_edge(sB, kb + idx * BK, ke);
    }
    if (HAS_W && !w_uniform) {
      double* sW = sB + LB::TILE;
      const int k = kb + idx * BK + tid;
      if (tid < BK) sW[tid] = (k < ke) ? p.w[k] : 0.0;
    }
  };

#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    if (s < nk) load_stage(s);
    cp_async_commit();
  }
  for (int kt = 0; kt < nk; ++kt) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    {
      const int nxt = kt + STAGES - 1;
      if (nxt < nk) load_stage(nxt);
      cp_async_commit();
    }
    const double* sA = smem + (kt % STAGES) * STAGE_DOUBLES;
    const double* sB = sA + LA::TILE;
    const double* sW = sB + LB::TILE;
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
      double a[MT], b[NT];
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        const int m = wm0 + mt * 8 + g;
        a[mt] = A_KCONTIG ? sA[m * LA::LDS_K + kk + t4] : sA[(kk + t4) * LA::LDMN + m];
      }
      if (HAS_W && !w_uniform) {
        const double wk = sW[kk + t4];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) a[mt] *= wk;
      }
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const int n = wn0 + nt * 8 + g;
        b[nt] = B_KCONTIG ? sB[n * LB::LDS_K + kk + t4] : sB[(kk + t4) * LB::LDMN + n];
      }
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dmma(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
    }
  }
  cp_async_wait<0>();

  // epilogue
  const bool vec_c = (p.ldc % 2 == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    const int row = m0 + wm0 + mt * 8 + g;
    double rowdot = 0.0;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int col = n0 + wn0 + nt * 8 + 2 * t4;
      if (row < p.M && col < p.N) {
        const bool two = (col + 1 < p.N);
        double v0 = alpha_eff * acc[mt][nt][0], v1 = alpha_eff * acc[mt][nt][1];
        double* cp = p.C + (long)row * p.ldc + col;
        if (p.splits > 1) {
          atomicAdd(cp, v0);
          if (two) atomicAdd(cp + 1, v1);
        } else {
          if (p.beta != 0.0) {
            v0 = fma(p.beta, cp[0], v0);
            if (two) v1 = fma(p.beta, cp[1], v1);
          }
          if (two && vec_c) st_v2(cp, v0, v1);
          else {
            cp[0] = v0;
            if (two) cp[1] = v1;
          }
        }
        if (p.dotK) {
          const double* kp = p.dotK + (long)row * p.lddot + col;
          rowdot = fma(v0, kp[0], rowdot);
          if (two) rowdot = fma(v1, kp[1], rowdot);
        }
      }
    }
    if (p.dotK) {
      rowdot += __shfl_xor_sync(0xffffffffu, rowdot, 1);
      rowdot += __shfl_xor_sync(0xffffffffu, rowdot, 2);
      if (t4 == 0 && row < p.M) atomicAdd(&p.q[row], rowdot);
    }
  }
}

// tile configurations: 64x64 tiles of 4 warps; Cfg4 for tall problems (M N > 4096^2 or K > 8192), Cfg3 for the others
struct Cfg3 { static constexpr int BM = 64, BN = 64, WM = 32, WN = 32, BK = 16, ST = 3, MINB = 3, NT = 128; };     // 3 CTAs/SM
struct Cfg4 { static constexpr int BM = 64, BN = 64, WM = 32, WN = 32, BK = 16, ST = 3, MINB = 4, NT = 128; };     // 4 CTAs/SM

template <class Cfg, bool AK, bool BK_>
constexpr int gemm_smem_bytes() {
  return Cfg::ST * (TileLoader<Cfg::BM, Cfg::BK, AK, Cfg::NT>::TILE + TileLoader<Cfg::BN, Cfg::BK, BK_, Cfg::NT>::TILE +
                    Cfg::BK) * 8;
}

__global__ void scale_matrix_kernel(int M, int N, double* C, long ldc, double beta, int out_tri) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)M * N) return;
  const int r = (int)(idx / N), c = (int)(idx % N);
  (void)out_tri;
  double* p = C + (long)r * ldc + c;
  *p = (beta == 0.0) ? 0.0 : beta * *p;
}

// copy one triangle of a square matrix onto the other (make symmetric)
__global__ void symmetrize_kernel(int M, double* C, long ldc, int from_upper) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y * blockDim.y + threadIdx.y;
  if (r >= M || c >= M || c <= r) return;  // (r,c) strictly upper
  if (from_upper) C[(long)c * ldc + r] = C[(long)r * ldc + c];
  else C[(long)r * ldc + c] = C[(long)c * ldc + r];
}

template <class Cfg, bool AK, bool BK_>
static int launch_cfg(const GemmParams& p, cudaStream_t st) {
  constexpr int smem = gemm_smem_bytes<Cfg, AK, BK_>();
  constexpr int GEMM_THREADS = Cfg::NT;
  auto kern = dgemm_kernel<Cfg::BM, Cfg::BN, Cfg::WM, Cfg::WN, Cfg::BK, Cfg::ST, AK, BK_, false, Cfg::MINB, Cfg::NT>;
  auto kern_w = dgemm_kernel<Cfg::BM, Cfg::BN, Cfg::WM, Cfg::WN, Cfg::BK, Cfg::ST, AK, BK_, true, Cfg::MINB, Cfg::NT>;
  // per-device attribute, cheap call: set every time (a process may touch more than one GPU)
  NPGP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  NPGP_CUDA(cudaFuncSetAttribute(kern_w, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  dim3 grid(ceil_div(p.N, Cfg::BN), ceil_div(p.M, Cfg::BM), p.splits);
  if (p.w && p.w_uniform_count) {
    if (!p.weighted_only) {
      kern<<<grid, GEMM_THREADS, smem, st>>>(p);
      NPGP_LAUNCH_CHECK();
    }
    kern_w<<<grid, GEMM_THREADS, smem, st>>>(p);
  } else if (p.w) {
    kern_w<<<grid, GEMM_THREADS, smem, st>>>(p);
  } else {
    kern<<<grid, GEMM_THREADS, smem, st>>>(p);
  }
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

template <class Cfg>
static int launch_layout(bool a_kc, bool b_kc, const GemmParams& p, cudaStream_t st) {
  if (a_kc && b_kc) return launch_cfg<Cfg, true, true>(p, st);
  if (a_kc) return launch_cfg<Cfg, true, false>(p, st);
  if (b_kc) return launch_cfg<Cfg, false, true>(p, st);
  return launch_cfg<Cfg, false, false>(p, st);
}

static int launch_gemm(bool a_kc, bool b_kc, const GemmParams& p, cudaStream_t st) {
  if ((long)p.M * p.N > (4096L * 4096L) || p.K > 8192) return launch_layout<Cfg4>(a_kc, b_kc, p, st);
  return launch_layout<Cfg3>(a_kc, b_kc, p, st);
}

// Split-K sizing: tile shape, resident CTAs per SM and the least k (rows of the SYRK) per split.  kCtasPerSm is 4 although
// Cfg3 keeps 3 CTAs resident: the split count follows from it, and the split count decides which products accumulate with
// atomics, so another value would change results, not just speed.
constexpr int kTileBM = 64, kTileBN = 64, kCtasPerSm = 4, kMinSplitK = 256;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int dgemm_impl(int transA, int transB, int M, int N, int K, double alpha, const double* A, long lda, const double* B,
               long ldb, double beta, double* C, long ldc, int tri_a, int tri_b, int out_tri, cudaStream_t st) {
  if (M < 0 || N < 0 || K < 0) return NPGP_EINVAL;
  if (M == 0 || N == 0) return NPGP_OK;
  if (!C || (K > 0 && (!A || !B))) return NPGP_EINVAL;
  if ((lda & 1) || (ldb & 1) || !aligned16(A) || !aligned16(B)) return NPGP_EUNSUPPORTED;
  GemmParams p{};
  p.M = M; p.N = N; p.K = K; p.A = A; p.lda = lda; p.B = B; p.ldb = ldb; p.C = C; p.ldc = ldc;
  p.alpha = alpha; p.beta = beta; p.tri_a = tri_a; p.tri_b = tri_b; p.out_tri = out_tri; p.splits = 1;
  // small outputs with a long K: split K so that the 148 SMs have work.  At least 4 splits when the tiles alone do not
  // fill the resident-CTA slots: measured on the nine M = 1024 GEMMs of the SVGP O(M^3) chain (tools/bench_tri_gemm.py),
  // 2 splits (512 CTAs on 444 slots: 1.15 waves) cost 0.100 ms for the dense product against 0.075 ms with 4, and the
  // triangular ones gain 5-20 % because the k-range of each tile is split, which evens out their unequal lengths.
  const long tiles = (long)ceil_div(M, kTileBM) * ceil_div(N, kTileBN);
  if (tiles * 2 <= kNumSMs * kCtasPerSm && K >= 2 * kMinSplitK) {
    int s = (int)max(4L, kNumSMs * kCtasPerSm / tiles);
    s = min(s, K / kMinSplitK);
    s = min(s, 16);
    if (s > 1) p.splits = s;
  }
  if (p.splits > 1) {
    const long tot = (long)M * N;
    scale_matrix_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(M, N, C, ldc, beta, out_tri);
    NPGP_LAUNCH_CHECK();
  }
  return launch_gemm(transA == 0, transB != 0, p, st);
}

}  // namespace npgp

using namespace npgp;

extern "C" int npgp_dgemm(int transA, int transB, int M, int N, int K, double alpha, const double* A, long lda,
                          const double* B, long ldb, double beta, double* C, long ldc, int tri_a, int tri_b,
                          int out_tri, cudaStream_t stream) {
  return dgemm_impl(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, tri_a, tri_b, out_tri, stream);
}

// T (n x M) = K (n x M) @ C (M x M);  q[i] = sum_j T_ij K_ij   (q must be zeroed by the caller; pass q = NULL to skip)
extern "C" int npgp_rowquad(int n, int M, const double* K, long ldk, const double* C, long ldc, double* T, long ldt,
                            double* q, cudaStream_t stream) {
  if (n < 0 || M < 0) return NPGP_EINVAL;
  if (n == 0 || M == 0) return NPGP_OK;
  if (!K || !C || !T) return NPGP_EINVAL;
  if ((ldk & 1) || (ldc & 1) || !aligned16(K) || !aligned16(C)) return NPGP_EUNSUPPORTED;
  GemmParams p{};
  p.M = n; p.N = M; p.K = M; p.A = K; p.lda = ldk; p.B = C; p.ldb = ldc; p.C = T; p.ldc = ldt;
  p.alpha = 1.0; p.beta = 0.0; p.splits = 1;
  if (q) { p.dotK = K; p.lddot = ldk; p.q = q; }
  return launch_gemm(true, false, p, stream);
}

// Out (M x M, symmetric) = alpha * K^T diag(w) K, K is (n x M); w may be NULL.  Out is overwritten.
static int wsyrk_impl(int n, int M, double alpha, const double* K, long ldk, const double* w,
                      const double* w_uniform_count, double w_uniform_target, double* Out, long ldo, cudaStream_t stream,
                      int weighted_only = 0);

extern "C" int npgp_wsyrk(int n, int M, double alpha, const double* K, long ldk, const double* w, double* Out, long ldo,
                          cudaStream_t stream) {
  return wsyrk_impl(n, M, alpha, K, ldk, w, nullptr, 0.0, Out, ldo, stream);
}

// Same, with a device-side hint: when *uniform_count == uniform_target all weights are equal (to w[0]) and the kernel
// takes the unweighted inner loop.  (SVGP-Gibbs: w = g_v is constant unless a predictive variance was clamped;
// npgp_gauss_ell counts the unclamped rows.)
extern "C" int npgp_wsyrk_hint(int n, int M, double alpha, const double* K, long ldk, const double* w,
                               const double* uniform_count, double uniform_target, double* Out, long ldo,
                               cudaStream_t stream) {
  return wsyrk_impl(n, M, alpha, K, ldk, w, uniform_count, uniform_target, Out, ldo, stream);
}

static int wsyrk_impl(int n, int M, double alpha, const double* K, long ldk, const double* w,
                      const double* w_uniform_count, double w_uniform_target, double* Out, long ldo,
                      cudaStream_t stream, int weighted_only) {
  if (n < 0 || M < 0) return NPGP_EINVAL;
  if (M == 0) return NPGP_OK;
  if (!Out || (n > 0 && !K)) return NPGP_EINVAL;
  if ((ldk & 1) || !aligned16(K)) return NPGP_EUNSUPPORTED;
  GemmParams p{};
  p.M = M; p.N = M; p.K = n; p.A = K; p.lda = ldk; p.B = K; p.ldb = ldk; p.C = Out; p.ldc = ldo;
  p.alpha = alpha; p.beta = 0.0; p.out_tri = 2; p.w = w;
  p.w_uniform_count = w ? w_uniform_count : nullptr; p.w_uniform_target = w_uniform_target;
  p.weighted_only = weighted_only;
  const long tiles = ((long)ceil_div(M, kTileBM) * ceil_div(M, kTileBN) + ceil_div(M, kTileBM)) / 2;
  // split the row range so that tiles x splits fills whole waves of resident CTAs: the cost of a choice is
  // (number of waves) / splits; take the cheapest among 1..32 splits of at least 512 rows each
  const long slots = (long)kNumSMs * kCtasPerSm;
  const int smax = (int)max(1L, min(32L, (long)n / (2 * kMinSplitK)));
  int best_s = 1;
  double best_cost = 1e300;
  for (int sp = 1; sp <= smax; ++sp) {
    const double cost = (double)((tiles * sp + slots - 1) / slots) / sp;
    if (cost < best_cost * (1.0 - 1e-3)) {  // prefer fewer splits (less atomic traffic) on ties
      best_cost = cost;
      best_s = sp;
    }
  }
  p.splits = best_s;
  if (p.splits > 1 || weighted_only) {  // weighted_only: the kernel may exit without writing
    const long tot = (long)M * M;
    scale_matrix_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, stream>>>(M, M, Out, ldo, 0.0, 0);
    NPGP_LAUNCH_CHECK();
    if (weighted_only && p.splits == 1) p.beta = 1.0;
  }
  int rc = launch_gemm(false, false, p, stream);
  if (rc) return rc;
  dim3 blk(32, 8), grd(ceil_div(M, 32), ceil_div(M, 8));
  symmetrize_kernel<<<grd, blk, 0, stream>>>(M, Out, ldo, 1);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

// The unequal-weights half of npgp_wsyrk_hint: Out = alpha K^T diag(w) K if *uniform_count != uniform_target, else Out = 0
// (the equal-weights case is then added by npgp_syrk_i8 with accumulate = 1).
extern "C" int npgp_wsyrk_weighted_only(int n, int M, double alpha, const double* K, long ldk, const double* w,
                                        const double* uniform_count, double uniform_target, double* Out, long ldo,
                                        cudaStream_t stream) {
  if (!w || !uniform_count) return NPGP_EINVAL;
  return wsyrk_impl(n, M, alpha, K, ldk, w, uniform_count, uniform_target, Out, ldo, stream, 1);
}

extern "C" int npgp_symmetrize(int M, double* C, long ldc, int from_upper, cudaStream_t stream) {
  if (M <= 0 || !C) return M == 0 ? NPGP_OK : NPGP_EINVAL;
  dim3 blk(32, 8), grd(ceil_div(M, 32), ceil_div(M, 8));
  symmetrize_kernel<<<grd, blk, 0, stream>>>(M, C, ldc, from_upper);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

// X = op(L)^-1 B through the inverse factor P = L^-1 that npgp_potrf_inv_* return: one triangular-aware DMMA product,
// X = P B (trans = 0) or X = P^T B (trans = 1).  This is what the reference does with its Cholesky factor --
// inv_root = triangular_solve(eye, chol) followed by matmul (models/gibbs_kernels.py:205-208,222-225) -- and what GPyTorch's
// whitened strategy needs (L^-1 Kzx).  P (M x M, lower), B, X (M x k); ldb, ldx even, 16-byte aligned operands.
extern "C" int npgp_trsm(int trans, int M, int k, const double* P, long ldp, const double* B, long ldb, double* X, long ldx,
                         cudaStream_t stream) {
  if (M < 0 || k < 0 || (trans != 0 && trans != 1)) return NPGP_EINVAL;
  if (M == 0 || k == 0) return NPGP_OK;
  if (!P || !B || !X || ldp < M || ldb < k || ldx < k) return NPGP_EINVAL;
  return npgp_dgemm(trans, 0, M, k, M, 1.0, P, ldp, B, ldb, 0.0, X, ldx, trans ? 2 : 1, 0, 0, stream);
}
