// Matrix-free lengthscale-field interpolation:  out[b,i,c] = bias_b + sum_j os_b exp(-0.5 |(x_i - z_j)/lam_b|^2) V[b,j,c]
// and its backward (dV, dz).  The (n x m) RBF cross-covariances are generated in registers and never stored.
//
// Replaces the dense K^prior_xz @ alpha of LogNormalPriorProcess.conditional_sample
// (reference models/gibbs_kernels.py:85-93; NB = D independent ARD kernels, NV = 1) and the dense Kronecker product of
// SparseMultivariateGibbsKernel.expectation_conditional_matrix_variate_dist
// (reference models/sparse_multivariate_gibbs_kernel.py:67-80; NB = 1, NV = d right-hand sides).
#include "common.cuh"
#include "pairmath.cuh"

namespace npgp {

constexpr int kFT = 128;   // threads per CTA
constexpr int kFR = 32;    // rows (fwd) / columns (bwd) per CTA = lanes
constexpr int kFS = 4;     // slices of the reduced axis per CTA = warps

// Reduced-axis points staged per slice per round: 64 while the kernel's static shared memory (the staged points, the
// per-warp accumulators and the exp table) stays within 48 KB, which holds for every configuration up to d = 3; above
// that the largest multiple of 8 that fits (d = nb = 4: 64 forward, 56 backward; 5: 40 / 32; 6: 24 / 24).
template <int d, int NB, int NV, bool BWD>
constexpr int field_chunk() {
  constexpr long kLimit = 48 * 1024;
  constexpr long fixed = 8L * kFS * kFR * (NB * NV + (BWD ? d : 0)) + 8L * 256;
  constexpr long per_point = 8L * kFS * NB * (d + NV);
  constexpr long fit = (kLimit - fixed) / per_point / 8 * 8;
  return fit > 64 ? 64 : (int)fit;
}

// forward: lanes own rows, warps own column slices
template <int d, int NB, int NV>
__global__ void __launch_bounds__(kFT) rbf_matvec_fwd_kernel(int n, int m, const double* __restrict__ x,
                                                             const double* __restrict__ z,
                                                             const double* __restrict__ lam,
                                                             const double* __restrict__ os,
                                                             const double* __restrict__ V,
                                                             const double* __restrict__ bias, int apply_exp,
                                                             double* __restrict__ out) {
  constexpr int kChunk = field_chunk<d, NB, NV, false>();
  static_assert(kChunk >= 8, "field_chunk: configuration too large for static shared memory");
  __shared__ double sz[kFS][kChunk][NB][d];   // pre-scaled column coordinates z/lam_b
  __shared__ double sv[kFS][kChunk][NB][NV];  // os_b * V
  __shared__ double sacc[kFS][kFR][NB * NV];
  __shared__ double sexp[256];
  static_assert(sizeof(sz) + sizeof(sv) + sizeof(sacc) + sizeof(sexp) <= 48 * 1024, "static shared memory over 48 KB");
  load_exp_table(sexp);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * kFR + lane;
  double il[NB][d], xs[NB][d], acc[NB][NV];
#pragma unroll
  for (int b = 0; b < NB; ++b) {
#pragma unroll
    for (int a = 0; a < d; ++a) {
      il[b][a] = 1.0 / lam[b * d + a];
      xs[b][a] = (i < n ? x[(long)i * d + a] : 0.0) * il[b][a];
    }
#pragma unroll
    for (int c = 0; c < NV; ++c) acc[b][c] = 0.0;
  }
  // warp w handles columns [w*per, (w+1)*per)
  const int per = (m + kFS - 1) / kFS;
  const int jlo = warp * per, jhi = min(m, jlo + per);
  for (int j0 = jlo; j0 < jhi; j0 += kChunk) {
    const int nc = min(kChunk, jhi - j0);
    __syncwarp();
    for (int t = lane; t < nc; t += 32) {
      const int j = j0 + t;
#pragma unroll
      for (int b = 0; b < NB; ++b) {
#pragma unroll
        for (int a = 0; a < d; ++a) sz[warp][t][b][a] = z[(long)j * d + a] * il[b][a];
        const double o = os ? os[b] : 1.0;
#pragma unroll
        for (int c = 0; c < NV; ++c) sv[warp][t][b][c] = o * V[((long)b * m + j) * NV + c];
      }
    }
    __syncwarp();
    for (int t = 0; t < nc; ++t) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        double q = 0.0;
#pragma unroll
        for (int a = 0; a < d; ++a) {
          const double df = xs[b][a] - sz[warp][t][b][a];
          q = fma(df, df, q);
        }
        const double k = exp_neg(-0.5 * q, sexp);
#pragma unroll
        for (int c = 0; c < NV; ++c) acc[b][c] = fma(k, sv[warp][t][b][c], acc[b][c]);
      }
    }
  }
#pragma unroll
  for (int b = 0; b < NB; ++b)
#pragma unroll
    for (int c = 0; c < NV; ++c) sacc[warp][lane][b * NV + c] = acc[b][c];
  __syncthreads();
  for (int t = threadIdx.x; t < kFR * NB * NV; t += kFT) {
    const int r = t / (NB * NV), bc = t % (NB * NV);
    const int b = bc / NV, c = bc % NV;
    const int ii = blockIdx.x * kFR + r;
    if (ii >= n) continue;
    double v = bias ? bias[b] : 0.0;
#pragma unroll
    for (int w = 0; w < kFS; ++w) v += sacc[w][r][bc];
    out[((long)b * n + ii) * NV + c] = apply_exp ? exp(v) : v;
  }
}

// backward: lanes own columns (reduced axis = rows), warps own row slices inside the CTA's row range
template <int d, int NB, int NV>
__global__ void __launch_bounds__(kFT) rbf_matvec_bwd_kernel(int n, int m, const double* __restrict__ x,
                                                             const double* __restrict__ z,
                                                             const double* __restrict__ lam,
                                                             const double* __restrict__ os,
                                                             const double* __restrict__ V,
                                                             const double* __restrict__ dOut, int rows_per_cta,
                                                             double* __restrict__ dV, double* __restrict__ dz) {
  constexpr int kChunk = field_chunk<d, NB, NV, true>();
  static_assert(kChunk >= 8, "field_chunk: configuration too large for static shared memory");
  __shared__ double sxr[kFS][kChunk][NB][d];   // pre-scaled row coordinates x/lam_b
  __shared__ double sg[kFS][kChunk][NB][NV];   // os_b * dOut
  __shared__ double sacc[kFS][kFR][NB * NV + d];
  __shared__ double sexp[256];
  static_assert(sizeof(sxr) + sizeof(sg) + sizeof(sacc) + sizeof(sexp) <= 48 * 1024, "static shared memory over 48 KB");
  load_exp_table(sexp);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * kFR + lane;
  double il[NB][d], zs[NB][d], vj[NB][NV], aV[NB][NV], az[d];
#pragma unroll
  for (int b = 0; b < NB; ++b) {
#pragma unroll
    for (int a = 0; a < d; ++a) {
      il[b][a] = 1.0 / lam[b * d + a];
      zs[b][a] = (j < m ? z[(long)j * d + a] : 0.0) * il[b][a];
    }
#pragma unroll
    for (int c = 0; c < NV; ++c) {
      vj[b][c] = (j < m) ? V[((long)b * m + j) * NV + c] : 0.0;
      aV[b][c] = 0.0;
    }
  }
#pragma unroll
  for (int a = 0; a < d; ++a) az[a] = 0.0;
  const int rb = blockIdx.y * rows_per_cta, re = min(n, rb + rows_per_cta);
  const int per = (re - rb + kFS - 1) / kFS;
  const int ilo = rb + warp * per, ihi = min(re, ilo + per);
  for (int i0 = ilo; i0 < ihi; i0 += kChunk) {
    const int nc = min(kChunk, ihi - i0);
    __syncwarp();
    for (int t = lane; t < nc; t += 32) {
      const int i = i0 + t;
#pragma unroll
      for (int b = 0; b < NB; ++b) {
#pragma unroll
        for (int a = 0; a < d; ++a) sxr[warp][t][b][a] = x[(long)i * d + a] * il[b][a];
        const double o = os ? os[b] : 1.0;
#pragma unroll
        for (int c = 0; c < NV; ++c) sg[warp][t][b][c] = o * dOut[((long)b * n + i) * NV + c];
      }
    }
    __syncwarp();
    for (int t = 0; t < nc; ++t) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        double q = 0.0, df[d];
#pragma unroll
        for (int a = 0; a < d; ++a) {
          df[a] = sxr[warp][t][b][a] - zs[b][a];
          q = fma(df[a], df[a], q);
        }
        const double k = exp_neg(-0.5 * q, sexp);
        double gv = 0.0;
#pragma unroll
        for (int c = 0; c < NV; ++c) {
          const double kg = k * sg[warp][t][b][c];
          aV[b][c] += kg;
          gv = fma(kg, vj[b][c], gv);
        }
        // d k / d z_a = k (x_a - z_a) / lam_a^2 = k * df_a * il_a
#pragma unroll
        for (int a = 0; a < d; ++a) az[a] = fma(gv, df[a] * il[b][a], az[a]);
      }
    }
  }
#pragma unroll
  for (int b = 0; b < NB; ++b)
#pragma unroll
    for (int c = 0; c < NV; ++c) sacc[warp][lane][b * NV + c] = aV[b][c];
#pragma unroll
  for (int a = 0; a < d; ++a) sacc[warp][lane][NB * NV + a] = az[a];
  __syncthreads();
  constexpr int NC = NB * NV + d;
  for (int t = threadIdx.x; t < kFR * NC; t += kFT) {
    const int r = t / NC, comp = t % NC;
    const int jj = blockIdx.x * kFR + r;
    if (jj >= m) continue;
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < kFS; ++w) v += sacc[w][r][comp];
    if (comp < NB * NV) {
      const int b = comp / NV, c = comp % NV;
      // os was folded into sg, so this is os_b * sum_i k dOut
      atomicAdd(&dV[((long)b * m + jj) * NV + c], v);
    } else if (dz) {
      atomicAdd(&dz[(long)jj * d + (comp - NB * NV)], v);
    }
  }
}

template <int d, int NB, int NV>
static int launch_rbf_fwd(int n, int m, const double* x, const double* z, const double* lam, const double* os,
                          const double* V, const double* bias, int apply_exp, double* out, cudaStream_t st) {
  rbf_matvec_fwd_kernel<d, NB, NV><<<ceil_div(n, kFR), kFT, 0, st>>>(n, m, x, z, lam, os, V, bias, apply_exp, out);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

template <int d, int NB, int NV>
static int launch_rbf_bwd(int n, int m, const double* x, const double* z, const double* lam, const double* os,
                          const double* V, const double* dOut, double* dV, double* dz, cudaStream_t st) {
  const int col_blocks = ceil_div(m, kFR);
  long want = (long)kNumSMs * 8;
  long row_ctas = (want + col_blocks - 1) / col_blocks;
  long rpc = (n + row_ctas - 1) / row_ctas;
  constexpr int kChunk = field_chunk<d, NB, NV, true>();
  if (rpc < 4 * kChunk) rpc = 4 * kChunk;
  dim3 grid(col_blocks, ceil_div(n, rpc));
  rbf_matvec_bwd_kernel<d, NB, NV><<<grid, kFT, 0, st>>>(n, m, x, z, lam, os, V, dOut, (int)rpc, dV, dz);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

}  // namespace npgp

using namespace npgp;

#define NPGP_RBF_DISPATCH(FN, ...)                                        \
  if (d == 1 && nb == 1 && nv == 1) return FN<1, 1, 1>(__VA_ARGS__);      \
  if (d == 2 && nb == 2 && nv == 1) return FN<2, 2, 1>(__VA_ARGS__);      \
  if (d == 2 && nb == 1 && nv == 2) return FN<2, 1, 2>(__VA_ARGS__);      \
  if (d == 2 && nb == 1 && nv == 1) return FN<2, 1, 1>(__VA_ARGS__);      \
  if (d == 3 && nb == 3 && nv == 1) return FN<3, 3, 1>(__VA_ARGS__);      \
  if (d == 3 && nb == 1 && nv == 3) return FN<3, 1, 3>(__VA_ARGS__);      \
  if (d == 3 && nb == 1 && nv == 1) return FN<3, 1, 1>(__VA_ARGS__);      \
  if (d == 3 && nb == 2 && nv == 1) return FN<3, 2, 1>(__VA_ARGS__);      \
  if (d == 4 && nb == 4 && nv == 1) return FN<4, 4, 1>(__VA_ARGS__);      \
  if (d == 5 && nb == 5 && nv == 1) return FN<5, 5, 1>(__VA_ARGS__);      \
  if (d == 6 && nb == 6 && nv == 1) return FN<6, 6, 1>(__VA_ARGS__);      \
  return NPGP_EUNSUPPORTED;

extern "C" int npgp_rbf_matvec_fwd(int d, int nb, int nv, int n, int m, const double* x, const double* z,
                                   const double* lam, const double* os, const double* V, const double* bias,
                                   int apply_exp, double* out, cudaStream_t stream) {
  if (n < 0 || m < 0) return NPGP_EINVAL;
  if (n == 0) return NPGP_OK;
  if (!x || !lam || !out || (m > 0 && (!z || !V))) return NPGP_EINVAL;
  NPGP_RBF_DISPATCH(launch_rbf_fwd, n, m, x, z, lam, os, V, bias, apply_exp, out, stream);
}

extern "C" int npgp_rbf_matvec_bwd(int d, int nb, int nv, int n, int m, const double* x, const double* z,
                                   const double* lam, const double* os, const double* V, const double* dOut,
                                   double* dV, double* dz, cudaStream_t stream) {
  if (n < 0 || m < 0) return NPGP_EINVAL;
  if (n == 0 || m == 0) return NPGP_OK;
  if (!x || !z || !lam || !V || !dOut || !dV) return NPGP_EINVAL;
  NPGP_RBF_DISPATCH(launch_rbf_bwd, n, m, x, z, lam, os, V, dOut, dV, dz, stream);
}
