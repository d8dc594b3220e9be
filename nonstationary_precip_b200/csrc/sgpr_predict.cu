// Row-side kernels of the streamed SGPR posterior (sgpr.py, posterior().predictive() and .sample()): the finishing kernel that
// turns the per-column-block row norms of P k(x) and V k(x) into the predictive variances and test log-densities, the FP64
// per-column-block row norms that stand in for npgp_o8_trinorm_digits when the feature width is not a multiple of 128, and
// the finishing kernel of the posterior draws.
#include "common.cuh"
#include "sample.cuh"

namespace npgp {

constexpr double kSgprLog2Pi = 1.8378770664093453;

// q[cb * q_stride + i] = sum_{j in [64 cb, min(64 cb + 64, W))} G_ij^2: one warp per row, fixed shuffle tree.
__global__ void __launch_bounds__(256) sgpr_rownorm_parts_kernel(int n, int W, const double* __restrict__ G, long ldg,
                                                                 double* __restrict__ q, long q_stride) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const double* g = G + (long)row * ldg;
  for (int c0 = 0, cb = 0; c0 < W; c0 += 64, ++cb) {
    const double a = (c0 + lane < W) ? g[c0 + lane] : 0.0;
    const double b = (c0 + 32 + lane < W) ? g[c0 + 32 + lane] : 0.0;
    const double t = warp_sum(fma(a, a, b * b));
    if (lane == 0) q[(long)cb * q_stride + row] = t;
  }
}

// var_f of row i from its partials, each component's added in index order (scalars s, os_t read from device memory):
//   q_t = sum_{c < nb_t} qn[c, i],  q_s = sum_{nb_t <= c < nb_t + nb_s} qn[c, i],  q_v = sum_{c < nb_v} qv[c, i]
//   var_f = [nb_t > 0] max(os_t - q_t, 0) + s max(1 - q_s, 0) + q_v
// With nb_v = 0 it is the residual r of the posterior draws, the variance that is independent across rows.
__device__ __forceinline__ double sgpr_row_var(int i, const double* __restrict__ qn, long qn_stride, int nb_t, int nb_s,
                                               const double* __restrict__ qv, long qv_stride, int nb_v,
                                               const double* __restrict__ s, const double* __restrict__ os_t) {
  double qt = 0.0, qs = 0.0, q2 = 0.0;
  for (int c = 0; c < nb_t; ++c) qt += qn[(long)c * qn_stride + i];
  for (int c = nb_t; c < nb_t + nb_s; ++c) qs += qn[(long)c * qn_stride + i];
  for (int c = 0; c < nb_v; ++c) q2 += qv[(long)c * qv_stride + i];
  // max(., 0) as comparisons: a NaN row norm (a row with a missing coordinate) stays NaN
  const double rs = 1.0 - qs;
  double v = s[0] * (rs < 0.0 ? 0.0 : rs) + q2;
  if (nb_t > 0) {
    const double rt = os_t[0] - qt;
    v += (rt < 0.0 ? 0.0 : rt);
  }
  return v;
}

// Per row i of a chunk (scalars s, noise, os_t read from device memory):
//   q1_t = sum_{c < nb_t} qn[c, i],  q1_s = sum_{nb_t <= c < nb_t + nb_s} qn[c, i],  q2 = sum_{c < nb_v} qv[c, i]  (index order)
//   var_f = [nb_t > 0] max(os_t - q1_t, 0) + s max(1 - q1_s, 0) + q2,   var_y = var_f + noise
//   y: lpd = log N(y | mean, var_y);  sums += [sum (y - mean)^2, sum -lpd, n]: block partials in blk, added in index order by the
//   last block to finish (ticket), which leaves the ticket at 0 again.
__global__ void __launch_bounds__(256) sgpr_predict_finish_kernel(
    int n, const double* __restrict__ qn, long qn_stride, int nb_t, int nb_s, const double* __restrict__ qv, long qv_stride,
    int nb_v, const double* __restrict__ mean, const double* __restrict__ y, const double* __restrict__ s,
    const double* __restrict__ noise, const double* __restrict__ os_t, double* __restrict__ var_f, double* __restrict__ var_y,
    double* __restrict__ lpd, double* __restrict__ sums, double* __restrict__ blk, unsigned int* __restrict__ ticket) {
  __shared__ double red[32];
  __shared__ bool last;
  const int i = blockIdx.x * 256 + threadIdx.x;
  double r2 = 0.0, nl = 0.0;
  if (i < n) {
    const double v = sgpr_row_var(i, qn, qn_stride, nb_t, nb_s, qv, qv_stride, nb_v, s, os_t);
    const double vy = v + noise[0];
    var_f[i] = v;
    if (var_y) var_y[i] = vy;
    if (y) {
      const double r = y[i] - mean[i];
      const double l = -0.5 * (kSgprLog2Pi + log(vy) + r * r / vy);
      if (lpd) lpd[i] = l;
      r2 = r * r;
      nl = -l;
    }
  }
  if (!sums) return;  // the same for every thread
  double t = block_sum(r2, red);
  if (threadIdx.x == 0) blk[blockIdx.x] = t;
  t = block_sum(nl, red);
  if (threadIdx.x == 0) {
    blk[gridDim.x + blockIdx.x] = t;
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  for (int k = 0; k < 2; ++k) {
    double a = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += 256) a += __ldcg(blk + (long)k * gridDim.x + b);
    const double tk = block_sum(a, red);
    if (threadIdx.x == 0) sums[k] += tk;
  }
  if (threadIdx.x == 0) {
    sums[2] += (double)n;
    *ticket = 0u;
  }
}

// Posterior draws of one chunk of n rows, CTA = 32 rows x 8 thread rows (scalars s, noise, os_t read from device memory):
//   out[s ldo + i] = mean_i + (F[i ldf + s] + sqrt(r_i (+ noise)) xi_s(row0 + i)),   r_i = sgpr_row_var(i, .., nb_v = 0)
// F (n x ldf) = K W, stored by sample_store_rows (sample.cuh).
__global__ void __launch_bounds__(256) sgpr_sample_finish_kernel(int n, int S, const double* __restrict__ mean,
                                                                 const double* __restrict__ qn, long qn_stride, int nb_t,
                                                                 int nb_s, const double* __restrict__ F, long ldf,
                                                                 const double* __restrict__ s, const double* __restrict__ noise,
                                                                 const double* __restrict__ os_t, int add_noise,
                                                                 unsigned long long seed, long row0, double* __restrict__ out,
                                                                 long ldo) {
  __shared__ double tile[32][33];
  __shared__ double smean[32], ssd[32];
  const int tx = threadIdx.x, i = blockIdx.x * 32 + tx;
  if (threadIdx.y == 0) {
    double mu = 0.0, r = 0.0;
    if (i < n) {
      mu = mean[i];
      r = sgpr_row_var(i, qn, qn_stride, nb_t, nb_s, nullptr, 0, 0, s, os_t);
      if (add_noise) r += noise[0];
    }
    smean[tx] = mu;
    ssd[tx] = sqrt(r);
  }
  sample_store_rows(n, S, F, ldf, seed, row0, out, ldo, tile, smean, ssd);
}

}  // namespace npgp

using namespace npgp;

extern "C" int npgp_sgpr_rownorm_parts(int n, int W, const double* G, long ldg, double* q, long q_stride,
                                       cudaStream_t stream) {
  if (n < 0 || W < 0 || (n > 0 && W > 0 && (!G || !q || ldg < W || q_stride < n))) return NPGP_EINVAL;
  if (n == 0 || W == 0) return NPGP_OK;
  sgpr_rownorm_parts_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(n, W, G, ldg, q, q_stride);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

extern "C" long npgp_sgpr_predict_workspace_bytes(int n) {
  if (n < 0) return -1;
  return 256 + 2L * ceil_div(n > 0 ? n : 1, 256) * (long)sizeof(double);
}

extern "C" int npgp_sgpr_predict_finish(int n, const double* qn, long qn_stride, int nb_t, int nb_s, const double* qv,
                                        long qv_stride, int nb_v, const double* mean, const double* y, const double* s,
                                        const double* noise, const double* os_t, double* var_f, double* var_y, double* lpd,
                                        double* sums, void* work, long work_bytes, cudaStream_t stream) {
  if (n < 0 || nb_t < 0 || nb_s < 0 || nb_v < 0) return NPGP_EINVAL;
  if (n == 0) return NPGP_OK;
  if (!s || !noise || !var_f || (nb_t > 0 && !os_t) || ((lpd || sums) && (!y || !mean))) return NPGP_EINVAL;
  if ((nb_t + nb_s > 0 && (!qn || qn_stride < n)) || (nb_v > 0 && (!qv || qv_stride < n))) return NPGP_EINVAL;
  if (sums && (!work || work_bytes < npgp_sgpr_predict_workspace_bytes(n))) return NPGP_EINVAL;
  unsigned int* ticket = static_cast<unsigned int*>(work);
  double* blk = sums ? reinterpret_cast<double*>(static_cast<char*>(work) + 256) : nullptr;
  sgpr_predict_finish_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(n, qn, qn_stride, nb_t, nb_s, qv, qv_stride, nb_v, mean, y,
                                                                  s, noise, os_t, var_f, var_y, lpd, sums, blk, ticket);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

extern "C" int npgp_sgpr_sample_finish(int n, int S, const double* mean, const double* qn, long qn_stride, int nb_t, int nb_s,
                                       const double* F, long ldf, const double* s, const double* noise, const double* os_t,
                                       int add_noise, unsigned long long seed, long row0, double* out, long ldo,
                                       cudaStream_t stream) {
  if (n < 0 || S < 1 || S > 1024 || nb_t < 0 || nb_s < 0 || row0 < 0 || n > (1L << 48) - row0) return NPGP_EINVAL;
  if (n == 0) return NPGP_OK;
  if (!mean || !F || !s || !out || ldf < S || ldo < n || (nb_t > 0 && !os_t) || (add_noise && !noise)) return NPGP_EINVAL;
  if (nb_t + nb_s > 0 && (!qn || qn_stride < n)) return NPGP_EINVAL;
  sgpr_sample_finish_kernel<<<ceil_div(n, 32), dim3(32, 8), 0, stream>>>(n, S, mean, qn, qn_stride, nb_t, nb_s, F, ldf, s, noise,
                                                                         os_t, add_noise, seed, row0, out, ldo);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}
