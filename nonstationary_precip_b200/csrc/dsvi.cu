// Doubly-stochastic variational inference (DSVI) kernels for the deep GP (reference models/dgps.py:53-111 via GPyTorch's
// DeepGPLayer.__call__ and DeepApproximateMLL(VariationalELBO), SURVEY.md Appendix B.4/B.5):
//
//   npgp_dsvi_sample[_bwd]   h = mu + sqrt(var) * eps  -- the marginal (diagonal) reparameterised sample that replaces
//                            Normal(mean, sqrt(variance)).rsample(); eps ~ N(0,1) from Philox4x32-10 keyed by
//                            (seed, global element index), so the draw does not depend on how samples / rows are sharded
//                            over ranks; eps can also be supplied (parity tests) or returned.
//   npgp_gauss_ell_batched   per-sample expected log-likelihood sums over rows, sum_i E_q log N(y_i | f_si, s2), with
//                            warp-shuffle + block reductions, and the gradient seeds d/dmu, d/dvar.
#include "common.cuh"
#include "philox.cuh"

namespace npgp {

__global__ void dsvi_sample_kernel(long n, const double* __restrict__ mu, const double* __restrict__ var,
                                   const double* __restrict__ eps_in, unsigned long long seed,
                                   unsigned long long index_offset, double* __restrict__ h,
                                   double* __restrict__ eps_out) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double e = eps_in ? eps_in[i] : normal_from_index(seed, index_offset + (unsigned long long)i);
  h[i] = fma(sqrt(var[i]), e, mu[i]);
  if (eps_out) eps_out[i] = e;
}

__global__ void dsvi_sample_bwd_kernel(long n, const double* __restrict__ var, const double* __restrict__ eps,
                                       const double* __restrict__ dh, double* __restrict__ dmu,
                                       double* __restrict__ dvar) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  dmu[i] = dh[i];
  dvar[i] = 0.5 * dh[i] * eps[i] * rsqrt(var[i]);
}

// grid (ceil(n/256), S).  sums[s] += sum_i ell_si;  gmu, gvar (S,n) = wscale * d ell / d mu, d var
__global__ void __launch_bounds__(256) gauss_ell_batched_kernel(int n, const double* __restrict__ y,
                                                                const double* __restrict__ mu,
                                                                const double* __restrict__ var,
                                                                const double* __restrict__ noise_p, double wscale,
                                                                double* __restrict__ sums, double* __restrict__ sq,
                                                                double* __restrict__ gmu, double* __restrict__ gvar) {
  __shared__ double red[32];
  const int i = blockIdx.x * 256 + threadIdx.x, s = blockIdx.y;
  const double s2 = *noise_p;
  double e = 0.0, r2v = 0.0;
  if (i < n) {
    const long k = (long)s * n + i;
    const double r = y[i] - mu[k], v = var[k];
    r2v = r * r + v;
    e = -0.5 * (r2v / s2 + log(s2) + 1.8378770664093453);
    if (gmu) gmu[k] = wscale * r / s2;
    if (gvar) gvar[k] = -0.5 * wscale / s2;
  }
  double t = block_sum(e, red);
  if (threadIdx.x == 0) atomicAdd(&sums[s], t);
  if (sq) {
    t = block_sum(r2v, red);
    if (threadIdx.x == 0) atomicAdd(&sq[s], t);
  }
}

}  // namespace npgp

using namespace npgp;

extern "C" int npgp_dsvi_sample(long n, const double* mu, const double* var, const double* eps_in,
                                unsigned long long seed, unsigned long long index_offset, double* h, double* eps_out,
                                cudaStream_t stream) {
  if (n < 0) return NPGP_EINVAL;
  if (n == 0) return NPGP_OK;
  if (!mu || !var || !h) return NPGP_EINVAL;
  dsvi_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(n, mu, var, eps_in, seed, index_offset, h, eps_out);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

extern "C" int npgp_dsvi_sample_bwd(long n, const double* var, const double* eps, const double* dh, double* dmu,
                                    double* dvar, cudaStream_t stream) {
  if (n < 0) return NPGP_EINVAL;
  if (n == 0) return NPGP_OK;
  if (!var || !eps || !dh || !dmu || !dvar) return NPGP_EINVAL;
  dsvi_sample_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(n, var, eps, dh, dmu, dvar);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

extern "C" int npgp_gauss_ell_batched(int S, int n, const double* y, const double* mu, const double* var,
                                      const double* noise, double wscale, double* sums, double* sq, double* gmu,
                                      double* gvar, cudaStream_t stream) {
  if (S < 0 || n < 0) return NPGP_EINVAL;
  if (S == 0 || n == 0) return NPGP_OK;
  if (!y || !mu || !var || !noise || !sums) return NPGP_EINVAL;
  dim3 grid(ceil_div(n, 256), S);
  gauss_ell_batched_kernel<<<grid, 256, 0, stream>>>(n, y, mu, var, noise, wscale, sums, sq, gmu, gvar);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}
