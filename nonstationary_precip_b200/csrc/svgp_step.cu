// The whole SVGP-Gibbs ELBO step behind the C ABI: npgp_svgp_elbo_fwd / npgp_svgp_elbo_bwd / npgp_svgp_step.
//
// Composition (SURVEY.md Appendix B): InducingGibbsKernel's field handling (reference models/gibbs_kernels.py:210-223), the
// multivariate kernels (models/sparse_multivariate_gibbs_kernel.py:67-154), GPyTorch's whitened VariationalStrategy +
// VariationalELBO as driven by models/dgps.py:25-35 and experiments/deepgp_spatial_bench.py:61,84-87, Adam as in
// experiments/spatial_exp.py:193.  One call enqueues
//     field interpolation -> K(X_B,Z) as digit planes, Kzz -> Cholesky + inverse -> whitened predictive mean / variance ->
//     Gaussian E[log-lik] + KL (+ field prior) -> analytic backward -> [all-reduce of the flat gradient] -> guarded Adam
// on the caller's stream plus two plan-owned side streams (joined again before the call returns, so the whole step can be
// captured into a CUDA graph from the caller's stream).  All scratch memory is carved from ONE caller-supplied workspace;
// nothing is allocated per call, every buffer has a fixed address (no allocator hazards between streams).
//
// Gradient chain (E = S - I, S = Ls Ls^T, P = L^-1, L = chol(Kzz + jitter I), u = P^T m, C = P^T E P):
//     mu = K u,  v = s + jitter_xx + rowdot(K C, K)
//     G  = dELBO/dK = g_mu u^T + 2 diag(g_v) (K C)               (formed inside the Gibbs backward kernel)
//     du = K^T g_mu,  dC = K^T diag(g_v) K,  dm = P du,  dE = P dC P^T,  dLs = tril(2 dE Ls)
//     dKzz = sym( P^T Phi(-(2 E dE + m dm^T)) P )                (Cholesky + inverse backward folded)
// theta / grad layout (doubles): full : [Z (M,d) | H (M,d) | D (d,d) | m (M) | Ls (M,M) | raw_outputscale | raw_noise]
//                                diag : [Z (M,d) | log_ell_z (d,M)   | m (M) | Ls (M,M) | raw_outputscale | raw_noise]
// padded to an even count n_pad; grad has n_pad + 2 entries, grad[n_pad] = this rank's share of -ELBO (so ONE all-reduce
// of grad carries gradient and loss).
#include <cstring>
#include <new>

#include "common.cuh"
#include "philox.cuh"
#include "sample.cuh"
#include "svgp_glue.cuh"
#include "../../include/npgp.h"

namespace npgp {

constexpr double kLog2Pi = 1.8378770664093453;

__device__ __forceinline__ double softplus_t(double x) { return x > 20.0 ? x : log1p(exp(x)); }  // torch softplus, threshold 20
__device__ __forceinline__ double sigmoid_t(double x) { return 1.0 / (1.0 + exp(-x)); }

// scal = [s, noise, sigmoid(raw_os), sigmoid(raw_noise)]
__global__ void svgp_scalars_kernel(const double* __restrict__ raw_os, const double* __restrict__ raw_noise,
                                    double* __restrict__ scal) {
  if (threadIdx.x == 0) {
    scal[0] = softplus_t(*raw_os);
    scal[1] = 1e-4 + softplus_t(*raw_noise);
    scal[2] = sigmoid_t(*raw_os);
    scal[3] = sigmoid_t(*raw_noise);
  }
}

// dst (M x kp, zero padded) <- src (M x k, leading dimension lds) [- sub_b]
__global__ void svgp_pad_cols_kernel(int M, int k, int kp, const double* __restrict__ src, long lds, double* __restrict__ dst) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < M)
    for (int c = 0; c < kp; ++c) dst[(long)i * kp + c] = (c < k) ? src[(long)i * lds + c] : 0.0;
}

// out[i] = exp(in[i])
__global__ void svgp_exp_kernel(long n, const double* __restrict__ in, double* __restrict__ out) {
  const long i = (long)blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = exp(in[i]);
}

// out[i] = a[i] - *c
__global__ void svgp_sub_scalar_kernel(int n, const double* __restrict__ a, const double* __restrict__ c, double* __restrict__ out) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = a[i] - *c;
}

// out[i] = s * a[i]
__global__ void svgp_scale_vec_kernel(long n, double s, const double* __restrict__ a, double* __restrict__ out) {
  const long i = (long)blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = s * a[i];
}

// out[i] = a[i] * b[i]
__global__ void svgp_mul_vec_kernel(long n, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out) {
  const long i = (long)blockIdx.x * 256 + threadIdx.x;
  if (i < n) out[i] = a[i] * b[i];
}

// KL pieces, stage 1 (fixed order): part[0][b] = sum Ls_t^2 over block b's rows, part[1][b] = sum log(diag^2), part[2][b] = sum m^2
__global__ void __launch_bounds__(256) svgp_kl_part_kernel(int M, const double* __restrict__ Ls_t, const double* __restrict__ m,
                                                           double* __restrict__ part) {
  __shared__ double red[32];
  const int rows_per = (M + gridDim.x - 1) / gridDim.x;
  const int r0 = blockIdx.x * rows_per, r1 = min(M, r0 + rows_per);
  double a = 0.0, l = 0.0, mm = 0.0;
  for (int r = r0; r < r1; ++r) {
    for (int c = threadIdx.x; c <= r; c += 256) {
      const double v = Ls_t[(long)r * M + c];
      a = fma(v, v, a);
    }
    if (threadIdx.x == 0) {
      const double dg = Ls_t[(long)r * M + r];
      l += log(dg * dg);
      mm = fma(m[r], m[r], mm);
    }
  }
  double t = block_sum(a, red);
  if (threadIdx.x == 0) part[blockIdx.x] = t;
  t = block_sum(l, red);
  if (threadIdx.x == 0) part[gridDim.x + blockIdx.x] = t;
  t = block_sum(mm, red);
  if (threadIdx.x == 0) part[2 * gridDim.x + blockIdx.x] = t;
}

// g_m = -(dm - rep m / N);  g_Ls = -(tril(dLs) - rep (Ls_t - diag(1 / diag Ls_t)) / N)
__global__ void svgp_grad_m_ls_kernel(int M, const double* __restrict__ dLs, const double* __restrict__ Ls_t,
                                      const double* __restrict__ dm, const double* __restrict__ m, double rep_over_N,
                                      double* __restrict__ g_Ls, double* __restrict__ g_m) {
  const int c = blockIdx.x * 32 + threadIdx.x, r = blockIdx.y * 8 + threadIdx.y;
  if (r >= M || c >= M) return;
  const long o = (long)r * M + c;
  const double l = Ls_t[o];
  const double kl = (c == r) ? (l - 1.0 / l) : l;  // Ls_t is zero above the diagonal
  g_Ls[o] = -(((c <= r) ? dLs[o] : 0.0) - rep_over_N * kl);
  if (c == 0) g_m[r] = -(dm[r] - rep_over_N * m[r]);
}

// Gk[i][j] = alpha * sum_c a[i*lda + c] b[j*ldb + c], c < k  (+ beta_old * Gk)
__global__ void svgp_outer_kernel(int M, int k, double alpha, const double* __restrict__ a, long lda, const double* __restrict__ b,
                                  long ldb, double* __restrict__ G) {
  const int c = blockIdx.x * 32 + threadIdx.x, r = blockIdx.y * 8 + threadIdx.y;
  if (r >= M || c >= M) return;
  double s = 0.0;
  for (int t = 0; t < k; ++t) s = fma(a[(long)r * lda + t], b[(long)c * ldb + t], s);
  G[(long)r * M + c] = alpha * s;
}

struct AssembleArgs {
  int variant, M, d, nblk_kl, include_prior, B_local;
  long n_pad, n_params;
  double rep, N_total, B_global;
  const double* scal;     // s, noise, sig_os, sig_noise
  const double* acc4;     // sum ell, sum ((y-mu)^2+v), #unclamped, w0
  const double* kl_part;  // 3 x nblk_kl
  const double* ds_acc;   // d_scale of both Gibbs backward kernels
  const double* gZ;       // (M,d) accumulated dELBO/dZ
  // full
  const double* beta4;    // (M,kp) Kr^-1 dW
  int kp;
  const double* dHz;      // (M,d)
  const double* dD_acc;   // (d,d)
  // diag
  const double* g_logell;  // (d,M): beta_b - pw alpha_b
  const double* dfz_acc;   // (d,M)
  const double* ell_z;     // (d,M)
  const double* lp_part;   // (d,2): [-0.5 r_b . alpha_b, sum log Ldiag_b]
  double* grad;
  long off_Z, off_F, off_D, off_os, off_noise;
};

// final assembly of the small gradient blocks and the loss slot (one CTA; everything here is O(M d))
__global__ void __launch_bounds__(256) svgp_assemble_kernel(AssembleArgs a) {
  const int M = a.M, d = a.d;
  for (int i = threadIdx.x; i < M * d; i += 256) {
    a.grad[a.off_Z + i] = -a.gZ[i];
    if (a.variant == 1) {
      const int r = i / d, c = i % d;
      a.grad[a.off_F + i] = -(a.beta4[(long)r * a.kp + c] + a.dHz[i]);
    } else {
      a.grad[a.off_F + i] = -(a.g_logell[i] + a.dfz_acc[i] * a.ell_z[i]);
    }
  }
  if (a.variant == 1)
    for (int i = threadIdx.x; i < d * d; i += 256) a.grad[a.off_D + i] = -a.dD_acc[i];
  if (threadIdx.x == 0) {
    const double noise = a.scal[1];
    for (long i = a.n_params; i < a.n_pad; ++i) a.grad[i] = 0.0;  // padding slot
    // v = s + ...: d v / d s = 1 on every row -> + sum_i g_v,i = w0 * #unclamped
    const double ds = *a.ds_acc + a.acc4[3] * a.acc4[2];
    a.grad[a.off_os] = -(ds * a.scal[2]);
    const double dnoise = (0.5 / a.B_global) * (a.acc4[1] / (noise * noise) - (double)a.B_local / noise);
    a.grad[a.off_noise] = -(dnoise * a.scal[3]);
  }
}

// loss slot: grad[n_pad] = -(E[log-lik] / B_global + rep (-KL + log prior) / N), sums added in a fixed order
__global__ void svgp_loss_kernel(AssembleArgs a) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double sLs = 0.0, slog = 0.0, smm = 0.0;
  for (int b = 0; b < a.nblk_kl; ++b) {
    sLs += a.kl_part[b];
    slog += a.kl_part[a.nblk_kl + b];
    smm += a.kl_part[2 * a.nblk_kl + b];
  }
  const double kl = 0.5 * (sLs + smm - (double)a.M - slog);
  double lp = 0.0;
  if (a.variant == 0 && a.include_prior)
    for (int b = 0; b < a.d; ++b) lp += (a.lp_part[2 * b] - a.lp_part[2 * b + 1] - 0.5 * a.M * kLog2Pi) / a.M;
  const double ell = a.acc4[0] / a.B_global;
  const double elbo = ell + a.rep * (-kl + lp) / a.N_total;
  a.grad[a.n_pad] = -elbo;
  a.grad[a.n_pad + 1] = 0.0;
}

// diag variant prior pieces of dimension b: lp_part[2b] = -0.5 r . alpha, lp_part[2b+1] = sum_i log L_ii   (one CTA, fixed order)
__global__ void __launch_bounds__(256) svgp_lp_part_kernel(int M, const double* __restrict__ r, const double* __restrict__ alpha,
                                                           const double* __restrict__ L, double* __restrict__ out2) {
  __shared__ double red[32];
  double a = 0.0, l = 0.0;
  for (int i = threadIdx.x; i < M; i += 256) {
    a = fma(r[i], alpha[i], a);
    l += log(L[(long)i * M + i]);
  }
  double t = block_sum(a, red);
  if (threadIdx.x == 0) out2[0] = -0.5 * t;
  t = block_sum(l, red);
  if (threadIdx.x == 0) out2[1] = t;
}

// g_logell_b = beta - pw alpha;  rv = -beta + 0.5 pw alpha
__global__ void svgp_diag_prior_vec_kernel(int M, double pw, const double* __restrict__ beta, const double* __restrict__ alpha,
                                           double* __restrict__ g_logell, double* __restrict__ rv) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < M) {
    g_logell[i] = beta[i] - pw * alpha[i];
    rv[i] = -beta[i] + 0.5 * pw * alpha[i];
  }
}

// Posterior marginals of one chunk of n rows (scal = [s, noise, ...]).  mean_i = sum_s mu_part[s n + i] and q_i = sum_c
// q_part[c n + i], both added in index order as in the step; var_f = max(s + jitter_xx + q, min_var), var_y = var_f + noise.
// With y: lpd_i = log N(y_i | mean_i, var_y_i) and per-block partials blk[b] = sum (y - mean)^2, blk[nblk + b] = sum -lpd.
// var_y, lpd may be NULL.
__global__ void __launch_bounds__(256) svgp_predict_finish_kernel(int n, const double* __restrict__ mu_part, int nsplit,
                                                                  const double* __restrict__ q_part, int nq,
                                                                  const double* __restrict__ scal, double jitter_xx,
                                                                  double min_var, const double* __restrict__ y,
                                                                  double* __restrict__ mean, double* __restrict__ var_f,
                                                                  double* __restrict__ var_y, double* __restrict__ lpd,
                                                                  double* __restrict__ blk) {
  __shared__ double red[32];
  const int i = blockIdx.x * 256 + threadIdx.x;
  double r2 = 0.0, nl = 0.0;
  if (i < n) {
    double mu = 0.0, q = 0.0;
    for (int k = 0; k < nsplit; ++k) mu += mu_part[(long)k * n + i];
    for (int k = 0; k < nq; ++k) q += q_part[(long)k * n + i];
    double v = scal[0] + jitter_xx + q;
    if (v < min_var) v = min_var;
    const double vy = v + scal[1];
    mean[i] = mu;
    var_f[i] = v;
    if (var_y) var_y[i] = vy;
    if (y) {
      const double r = y[i] - mu;
      const double l = -0.5 * (kLog2Pi + log(vy) + r * r / vy);
      if (lpd) lpd[i] = l;
      r2 = r * r;
      nl = -l;
    }
  }
  if (!y) return;  // the same for every thread: no thread leaves a barrier of block_sum that others reach
  double t = block_sum(r2, red);
  if (threadIdx.x == 0) blk[blockIdx.x] = t;
  t = block_sum(nl, red);
  if (threadIdx.x == 0) blk[gridDim.x + blockIdx.x] = t;
}

// sums += [sum_b blk[b], sum_b blk[nblk + b], n]: one CTA, fixed assignment and tree (bitwise reproducible)
__global__ void __launch_bounds__(256) svgp_predict_sums_kernel(int nblk, int n, const double* __restrict__ blk,
                                                                double* __restrict__ sums) {
  __shared__ double red[32];
  for (int k = 0; k < 2; ++k) {
    double a = 0.0;
    for (int b = threadIdx.x; b < nblk; b += 256) a += blk[(long)k * nblk + b];
    const double t = block_sum(a, red);
    if (threadIdx.x == 0) sums[k] += t;
  }
  if (threadIdx.x == 0) sums[2] += (double)n;
}


// Et (Sp x W) = E^T of the samplers: Et[s][j] = E[j, s] = normal_from_index(seed, (s << 32) + j) for s < S, zero rows s >= S
__global__ void sample_normals_kernel(int W, int S, int Sp, unsigned long long seed, double* __restrict__ Et) {
  const long k = (long)blockIdx.x * 256 + threadIdx.x;
  if (k >= (long)Sp * W) return;
  const int s = (int)(k / W), j = (int)(k % W);
  Et[k] = s < S ? normal_from_index(seed, ((unsigned long long)s << 32) + (unsigned long long)j) : 0.0;
}

// Posterior draws of one chunk of n rows (scal = [s, noise, ...]), CTA = 32 rows x 8 thread rows:
//   out[s ldo + i] = mean_i + (F[i ldf + s] + sqrt(r_i) xi_s(row0 + i)),  r_i = max(s + jitter_xx - q_i, 0) (+ noise)
// mean_i and q_i are the partials added in index order (mean as in svgp_predict_finish_kernel); F (n x ldf) = K W is stored
// by sample_store_rows (sample.cuh).
__global__ void __launch_bounds__(256) svgp_sample_finish_kernel(int n, int S, const double* __restrict__ mu_part, int nsplit,
                                                                 const double* __restrict__ q_part, int nq,
                                                                 const double* __restrict__ scal, double jitter_xx, int noise,
                                                                 const double* __restrict__ F, int ldf, unsigned long long seed,
                                                                 long row0, double* __restrict__ out, long ldo) {
  __shared__ double tile[32][33];
  __shared__ double smean[32], ssd[32];
  const int tx = threadIdx.x, ty = threadIdx.y, i = blockIdx.x * 32 + tx;
  if (ty == 0) {
    double mu = 0.0, q = 0.0;
    if (i < n) {
      for (int k = 0; k < nsplit; ++k) mu += mu_part[(long)k * n + i];
      for (int k = 0; k < nq; ++k) q += q_part[(long)k * n + i];
    }
    double r = scal[0] + jitter_xx - q;
    if (r < 0.0) r = 0.0;  // (a NaN stays NaN)
    if (noise) r += scal[1];
    smean[tx] = mu;
    ssd[tx] = sqrt(r);
  }
  sample_store_rows(n, S, F, ldf, seed, row0, out, ldo, tile, smean, ssd);
}
}  // namespace npgp

using namespace npgp;

// ---------------------------------------------------------------------------------------------------------------------
// plan
// ---------------------------------------------------------------------------------------------------------------------
struct npgp_svgp_plan {
  npgp_svgp_config c;
  int P6, kp, nsplit, nb128, nblk_kl;
  long n_params, n_pad;
  long off_Z, off_F, off_D, off_m, off_Ls, off_os, off_noise;
  cudaStream_t side, side2;
  cudaEvent_t ev[12];
  bool fwd_done;
  // ---- workspace carve-up
  double *scal, *fz, *Ls_t, *E, *Kzz, *P, *u, *EP, *C;
  double *Kr, *Pr, *lam_b, *R4, *T4, *W4, *Wp, *Hx, *fx;   // full: Kr/Pr (1 set); diag: d sets (Kr = Kp_b, Pr = P_b)
  double *alpha, *rhs, *tmpv, *ell_x;                     // diag
  double *T, *mu_part, *q_part, *du_part, *syrk_part, *mu, *gmu0, *gmu, *gv, *gv2, *acc4, *gwork, *kl_part, *lp_part;
  double *du, *dC, *dm, *W2, *dE, *dLs, *X, *Y, *dK, *dKzz;
  double *zero_begin, *dfz_acc, *gZ, *dfx, *ds_acc, *dHx, *dD_acc, *dW, *dHz, *dummy_ell, *dalpha, *zero_end;
  double *beta4, *T4b, *R4b, *Gk, *dlog, *g_logell, *rv, *beta_v;
  int8_t *Ad, *Cd;
  int *cexp, *skip_count, *skip_rows, *info, *flags[8];  // flags[0]: Kzz, flags[1 + b]: prior-kernel factorisation b
  long flags_bytes, syrk_part_bytes, gwork_bytes;
  bool prepared;  // the Z-side factors of npgp_svgp_predict_prepare are in the workspace (cleared by fwd / step / jitter)
  // npgp_svgp_sample_prepare has filled sample_work for sample_S draws of sample_seed (cleared by fwd / step / jitter /
  // predict_prepare)
  bool sample_ready;
  int sample_S;
  unsigned long long sample_seed;
  void* sample_work;
};

namespace {

struct Carver {
  char* base;
  long off;
  template <typename T>
  T* take(long count) {
    off = (off + 255) & ~255L;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * (long)sizeof(T);
    return p;
  }
};

int svgp_layout(npgp_svgp_plan* p, void* workspace, long* bytes_out) {
  const npgp_svgp_config& c = p->c;
  const int M = c.M, d = c.d, B = c.B_local;
  if ((c.variant != 0 && c.variant != 1) || M <= 0 || B <= 0 || d < 1 || c.world_size < 1 || c.B_global < B) return NPGP_EINVAL;
  if (M % 128 || (c.variant == 1 && d != 2 && d != 3) || (c.variant == 0 && d > 6)) return NPGP_EUNSUPPORTED;
  p->P6 = (c.variant == 1) ? d * (d + 1) / 2 : d;  // per-point field entries
  p->kp = (d + 1) / 2 * 2 < 2 ? 2 : (d + 1) / 2 * 2;
  p->nsplit = npgp_gibbs_digits_splits(B, M);
  p->nb128 = (B + 127) / 128;
  p->nblk_kl = 64;
  long off = 0;
  p->off_Z = off, off += (long)M * d;
  p->off_F = off, off += (long)M * d;  // H (M,d) or log_ell_z (d,M)
  p->off_D = off, off += (c.variant == 1) ? (long)d * d : 0;
  p->off_m = off, off += M;
  p->off_Ls = off, off += (long)M * M;
  p->off_os = off, off += 1;
  p->off_noise = off, off += 1;
  p->n_params = off;
  p->n_pad = (off + 1) / 2 * 2;
  p->flags_bytes = npgp_potrf_flow_workspace_bytes(M);
  p->syrk_part_bytes = npgp_o8_syrk_part_bytes(B, M);
  p->gwork_bytes = npgp_gauss_ell_parts_workspace_bytes(B);
  const long MM = (long)M * M;
  const int nset = (c.variant == 1) ? 1 : d;  // prior-kernel factorisations kept for the backward
  Carver w{static_cast<char*>(workspace), 0};
  p->scal = w.take<double>(8);
  p->fz = w.take<double>((long)M * p->P6);
  p->Ls_t = w.take<double>(MM), p->E = w.take<double>(MM), p->Kzz = w.take<double>(MM), p->P = w.take<double>(MM);
  p->u = w.take<double>(M), p->EP = w.take<double>(MM), p->C = w.take<double>(MM);
  p->Kr = w.take<double>(MM * nset), p->Pr = w.take<double>(MM * nset);
  p->lam_b = w.take<double>((long)d * M * nset);
  p->R4 = w.take<double>((long)M * p->kp), p->T4 = w.take<double>((long)M * p->kp), p->W4 = w.take<double>((long)M * p->kp);
  p->Wp = w.take<double>((long)M * d);
  p->Hx = w.take<double>((long)B * d), p->fx = w.take<double>((long)B * p->P6);
  p->alpha = w.take<double>((long)d * M), p->rhs = w.take<double>((long)d * M), p->tmpv = w.take<double>(M);
  p->ell_x = w.take<double>((long)d * B);
  p->T = w.take<double>((long)B * M);
  p->mu_part = w.take<double>((long)p->nsplit * B), p->q_part = w.take<double>((long)(M / 64) * B);
  p->du_part = w.take<double>((long)p->nb128 * M);
  p->syrk_part = w.take<double>(p->syrk_part_bytes / 8 + 1);
  p->mu = w.take<double>(B), p->gmu0 = w.take<double>(B), p->gmu = w.take<double>(B), p->gv = w.take<double>(B);
  p->gv2 = w.take<double>(B), p->acc4 = w.take<double>(4), p->gwork = w.take<double>(p->gwork_bytes / 8 + 1);
  p->kl_part = w.take<double>(3 * p->nblk_kl), p->lp_part = w.take<double>(2 * 8);
  p->du = w.take<double>(M), p->dC = w.take<double>(MM), p->dm = w.take<double>(M), p->W2 = w.take<double>(MM);
  p->dE = w.take<double>(MM), p->dLs = w.take<double>(MM), p->X = w.take<double>(MM), p->Y = w.take<double>(MM);
  p->dK = w.take<double>(MM), p->dKzz = w.take<double>(MM);
  // accumulators (one memset per step): contiguous
  p->zero_begin = w.take<double>(0);
  p->dfz_acc = w.take<double>((long)M * p->P6), p->gZ = w.take<double>((long)M * d), p->dfx = w.take<double>((long)B * p->P6);
  p->ds_acc = w.take<double>(2), p->dHx = w.take<double>((long)B * d), p->dD_acc = w.take<double>((long)d * d);
  p->dW = w.take<double>((long)M * d), p->dHz = w.take<double>((long)M * d), p->dummy_ell = w.take<double>(2L * d * M);
  p->dalpha = w.take<double>((long)d * M);
  p->zero_end = w.take<double>(0);
  p->beta4 = w.take<double>((long)M * p->kp), p->T4b = w.take<double>((long)M * p->kp), p->R4b = w.take<double>((long)M * p->kp);
  p->Gk = w.take<double>(MM), p->dlog = w.take<double>((long)d * B);
  p->g_logell = w.take<double>((long)d * M), p->rv = w.take<double>(M), p->beta_v = w.take<double>(M);
  p->Ad = w.take<int8_t>(npgp_o8_digits_bytes(B, M, 128));
  p->Cd = w.take<int8_t>(npgp_o8_digits_bytes(M, M, 64));
  p->cexp = w.take<int>(M), p->skip_count = w.take<int>(4), p->skip_rows = w.take<int>(B), p->info = w.take<int>(8);
  for (int i = 0; i < 1 + nset; ++i) p->flags[i] = w.take<int>(p->flags_bytes / 4 + 1);
  *bytes_out = w.off + 256;
  return NPGP_OK;
}

// fork: `to` continues after everything enqueued on `from` so far
inline int fork_stream(cudaStream_t from, cudaStream_t to, cudaEvent_t ev) {
  NPGP_CUDA(cudaEventRecord(ev, from));
  NPGP_CUDA(cudaStreamWaitEvent(to, ev, 0));
  return NPGP_OK;
}

#define NPGP_TRY(call)        \
  do {                        \
    int rc__ = (call);        \
    if (rc__) return rc__;    \
  } while (0)

inline dim3 grid2(int M) { return dim3(ceil_div(M, 32), ceil_div(M, 8)); }
const dim3 kBlk2(32, 8);

template <int KP>
int tri_skinny(int M, const double* Pm, const double* R, double* tmp, double* out, cudaStream_t st) {
  svgp_tri_skinny_n_kernel<KP><<<ceil_div(M, 8), 256, 0, st>>>(M, Pm, R, tmp);
  NPGP_LAUNCH_CHECK();
  svgp_tri_skinny_t_kernel<KP><<<ceil_div(M, 8), 256, 0, st>>>(M, Pm, tmp, out);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

// out = P^T w (M): the transposed skinny product alone (u = P^T m)
int tri_t_vec(int M, const double* Pm, const double* w, double* out, cudaStream_t st) {
  svgp_tri_skinny_t_kernel<1><<<ceil_div(M, 8), 256, 0, st>>>(M, Pm, w, out);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

// K^-1 rhs for rhs (M): P^T (P rhs), K = L L^T, P = L^-1
int solve_vec(npgp_svgp_plan* p, const double* Pm, const double* rhs, double* tmp, double* out, cudaStream_t st) {
  return tri_skinny<1>(p->c.M, Pm, rhs, tmp, out, st);
}

// K^-1 rhs for rhs (M x k, leading dimension lds): padded to kp columns; result in out4 (M x kp)
int solve_cols(npgp_svgp_plan* p, const double* Pm, const double* rhs, long lds, int k, double* R4, double* T4, double* out4,
               cudaStream_t st) {
  const int M = p->c.M, kp = p->kp;
  svgp_pad_cols_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, k, kp, rhs, lds, R4);
  NPGP_LAUNCH_CHECK();
  if (kp == 2) return tri_skinny<2>(M, Pm, R4, T4, out4, st);
  if (kp == 4) return tri_skinny<4>(M, Pm, R4, T4, out4, st);
  NPGP_TRY(npgp_dgemm(0, 0, M, kp, M, 1.0, Pm, M, R4, kp, 0.0, T4, kp, 1, 0, 0, st));
  NPGP_TRY(npgp_dgemm(1, 0, M, kp, M, 1.0, Pm, M, T4, kp, 0.0, out4, kp, 2, 0, 0, st));
  return NPGP_OK;
}

int stamp(npgp_svgp_plan* p, int slot, cudaStream_t st) {
  if (!p->c.timeline) return NPGP_OK;
  return npgp_timestamp(p->c.timeline, slot, st);
}

}  // namespace

static const char* kSvgpSections[] = {"zz_fwd(potrf+M^3)", "field_fwd", "kxz_fwd", "rowquad", "gauss_ell", "wsyrk",
                                      "m3_bwd+kzz_bwd",    "kxz_bwd",   "field_bwd", "assemble", "allreduce", "adam"};
enum { SEC_ZZ = 0, SEC_FIELD, SEC_KXZ, SEC_RQ, SEC_ELL, SEC_SYRK, SEC_M3, SEC_KXZB, SEC_FIELDB, SEC_ASM, SEC_AR, SEC_ADAM, SEC_N };

extern "C" int npgp_svgp_num_sections(void) { return SEC_N; }
extern "C" const char* npgp_svgp_section_name(int i) { return (i >= 0 && i < SEC_N) ? kSvgpSections[i] : nullptr; }

extern "C" long npgp_svgp_theta_size(const npgp_svgp_config* cfg) {
  if (!cfg) return -1;
  npgp_svgp_plan tmp;
  tmp.c = *cfg;
  long bytes;
  if (svgp_layout(&tmp, nullptr, &bytes)) return -1;
  return tmp.n_pad;
}

extern "C" long npgp_svgp_workspace_bytes(const npgp_svgp_config* cfg) {
  if (!cfg) return -1;
  npgp_svgp_plan tmp;
  tmp.c = *cfg;
  long bytes;
  if (svgp_layout(&tmp, nullptr, &bytes)) return -1;
  return bytes;
}

extern "C" int npgp_svgp_plan_create(npgp_svgp_plan** out, const npgp_svgp_config* cfg, void* workspace, long workspace_bytes) {
  if (!out || !cfg || !workspace) return NPGP_EINVAL;
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return NPGP_EUNSUPPORTED;
  if (cfg->variant == 1 && (!cfg->row_os || !cfg->row_lam)) return NPGP_EINVAL;
  if (cfg->variant == 0 && (!cfg->prior_c || !cfg->prior_os || !cfg->prior_lam)) return NPGP_EINVAL;
  npgp_svgp_plan* p = new (std::nothrow) npgp_svgp_plan;
  if (!p) return NPGP_EINVAL;
  memset(p, 0, sizeof(*p));
  p->c = *cfg;
  long bytes;
  int rc = svgp_layout(p, workspace, &bytes);
  if (rc == NPGP_OK && workspace_bytes < bytes) rc = NPGP_EWORKSPACE;
  if (rc) {
    delete p;
    return rc;
  }
  cudaError_t e = cudaStreamCreateWithFlags(&p->side, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->side2, cudaStreamNonBlocking);
  for (int i = 0; i < 12 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&p->ev[i], cudaEventDisableTiming);
  if (e != cudaSuccess) {
    delete p;
    return (int)e;
  }
  *out = p;
  return NPGP_OK;
}

extern "C" int npgp_svgp_plan_destroy(npgp_svgp_plan* p) {
  if (!p) return NPGP_OK;
  for (int i = 0; i < 12; ++i)
    if (p->ev[i]) cudaEventDestroy(p->ev[i]);
  if (p->side) cudaStreamDestroy(p->side);
  if (p->side2) cudaStreamDestroy(p->side2);
  delete p;
  return NPGP_OK;
}

/* jitter added to Kzz on top of cfg.jitter_zz (psd_safe_cholesky ladder, driven by the host after a failed step) */
extern "C" int npgp_svgp_set_extra_jitter(npgp_svgp_plan* p, double extra) {
  if (!p || !(extra >= 0.0)) return NPGP_EINVAL;
  p->c.extra_jitter = extra;
  p->prepared = false;  // the prepared Cholesky used the old jitter
  p->sample_ready = false;
  return NPGP_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Z-side chain (independent of the rows), shared by the forward and npgp_svgp_predict_prepare: scalars, field at Z, the
// accumulator reset and the KL / prior sums of the loss; on the side streams Kzz -> Cholesky + inverse -> u = P^T m (event
// ev[10]) -> C = P^T (Ls Ls^T - I) P and its digit planes (event ev[3]); on `st` the prior-kernel factorisations and the
// interpolation weights of the field (alpha / W).  The side streams are NOT joined here: the forward waits for ev[10] and
// ev[3] at the points where it needs u and C.
// ---------------------------------------------------------------------------------------------------------------------
static int svgp_zside(npgp_svgp_plan* p, const double* theta, int* status, cudaStream_t st) {
  const npgp_svgp_config& c = p->c;
  const int M = c.M, d = c.d, full = c.variant == 1;
  const long MM = (long)M * M;
  const double* Z = theta + p->off_Z;
  const double* F = theta + p->off_F;   // H (M,d) or log_ell_z (d,M)
  const double* Dm = theta + p->off_D;  // full only
  const double* m = theta + p->off_m;
  const double* Ls = theta + p->off_Ls;
  const double* s = p->scal;
  cudaStream_t sd = p->side, sd2 = p->side2;

  svgp_scalars_kernel<<<1, 32, 0, st>>>(theta + p->off_os, theta + p->off_noise, p->scal);
  NPGP_LAUNCH_CHECK();
  NPGP_CUDA(cudaMemsetAsync(p->zero_begin, 0, (char*)p->zero_end - (char*)p->zero_begin, st));
  if (full) {
    NPGP_TRY(npgp_sigma_from_h_fwd(d, M, F, Dm, p->fz, st));
  } else {
    svgp_exp_kernel<<<ceil_div((long)d * M, 256), 256, 0, st>>>((long)d * M, F, p->fz);
    NPGP_LAUNCH_CHECK();
  }

  // ---- side stream: Kzz -> Cholesky + inverse -> u = P^T m, C = P^T (Ls Ls^T - I) P
  NPGP_TRY(fork_stream(st, sd, p->ev[0]));
  NPGP_TRY(stamp(p, 2 * SEC_ZZ, sd));
  svgp_tril_copy_kernel<<<grid2(M), kBlk2, 0, sd>>>(M, Ls, p->Ls_t);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(fork_stream(sd, sd2, p->ev[1]));
  {  // S - I does not depend on the factorisation: runs under the latency-bound Cholesky; so do the KL sums
    NPGP_TRY(npgp_dgemm(0, 1, M, M, M, 1.0, p->Ls_t, M, p->Ls_t, M, 0.0, p->E, M, 1, 2, 1, sd2));  // symmetric: lower tiles,
    NPGP_TRY(npgp_symmetrize(M, p->E, M, 0, sd2));                                                  // mirrored
    svgp_add_diag_kernel<<<ceil_div(M, 256), 256, 0, sd2>>>(M, p->E, M, -1.0);
    NPGP_LAUNCH_CHECK();
    svgp_kl_part_kernel<<<p->nblk_kl, 256, 0, sd2>>>(M, p->Ls_t, m, p->kl_part);
    NPGP_LAUNCH_CHECK();
    NPGP_CUDA(cudaEventRecord(p->ev[2], sd2));
  }
  if (full) NPGP_TRY(npgp_gibbs_full_fwd(d, M, M, Z, p->fz, Z, p->fz, c.kernel_jitter, s, p->Kzz, M, nullptr, nullptr, sd));
  else NPGP_TRY(npgp_gibbs_diag_fwd(d, M, M, Z, p->fz, Z, p->fz, s, p->Kzz, M, nullptr, nullptr, sd));
  svgp_add_diag_kernel<<<ceil_div(M, 256), 256, 0, sd>>>(M, p->Kzz, M, c.jitter_zz + c.extra_jitter);
  NPGP_LAUNCH_CHECK();
  NPGP_CUDA(cudaEventRecord(p->ev[8], sd));  // Kzz is built

  // ---- main stream: prior kernel(s) of the latent field at Z, then ALL factorisations of the step (Kzz and the prior
  // kernels) in one batched dataflow launch
  NPGP_TRY(stamp(p, 2 * SEC_FIELD, st));
  const int nset = full ? 1 : d;
  for (int b = 0; b < nset; ++b) {
    double* lamb = p->lam_b + (long)b * d * M;
    double* Kp = p->Kr + (long)b * MM;
    svgp_bcast_rows_kernel<<<ceil_div(M, 256), 256, 0, st>>>(d, M, full ? c.row_lam : c.prior_lam + (long)b * d, lamb);
    NPGP_LAUNCH_CHECK();
    NPGP_TRY(npgp_gibbs_diag_fwd(d, M, M, Z, lamb, Z, lamb, full ? c.row_os : c.prior_os + b, Kp, M, nullptr, nullptr, st));
    svgp_add_diag_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, Kp, M, full ? 1e-5 : 1e-4);
    NPGP_LAUNCH_CHECK();
  }
  NPGP_CUDA(cudaStreamWaitEvent(st, p->ev[8], 0));
  for (int first = 0; first < 1 + nset; first += 4) {  // matrix 0 = Kzz, 1 + b = prior kernel b; at most 4 per launch
    double* As[4];
    double* Ps[4];
    void* Ws[4];
    int* Is[4];
    int n = 0;
    for (int i = first; i < 1 + nset && n < 4; ++i, ++n) {
      As[n] = i == 0 ? p->Kzz : p->Kr + (long)(i - 1) * MM;
      Ps[n] = i == 0 ? p->P : p->Pr + (long)(i - 1) * MM;
      Ws[n] = p->flags[i];
      Is[n] = p->info + i;
    }
    NPGP_TRY(npgp_potrf_inv_flow_batch(n, M, As, M, Ps, M, Ws, p->flags_bytes, Is, st));
    if (status)
      for (int k = 0; k < n; ++k) NPGP_TRY(npgp_status_update(status, Is[k], nullptr, st));
    if (first == 0) NPGP_CUDA(cudaEventRecord(p->ev[9], st));  // L, P of Kzz are ready
  }

  // ---- side stream: u = P^T m, C = P^T (Ls Ls^T - I) P and its digit planes
  NPGP_CUDA(cudaStreamWaitEvent(sd, p->ev[9], 0));
  NPGP_TRY(tri_t_vec(M, p->P, m, p->u, sd));  // u = P^T m
  NPGP_CUDA(cudaEventRecord(p->ev[10], sd));   // all the K(X_B,Z) tile kernel needs from this chain; C is only needed by T = K C
  NPGP_CUDA(cudaStreamWaitEvent(sd, p->ev[2], 0));
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 1.0, p->E, M, p->P, M, 0.0, p->EP, M, 0, 1, 0, sd));
  // C = P^T (E P) is symmetric: only the tiles touching the lower triangle are computed, the rest is mirrored
  NPGP_TRY(npgp_dgemm(1, 0, M, M, M, 1.0, p->P, M, p->EP, M, 0.0, p->C, M, 2, 0, 1, sd));
  NPGP_TRY(npgp_symmetrize(M, p->C, M, 0, sd));
  NPGP_TRY(npgp_o8_slice_rows(M, M, p->C, M, 64, p->Cd, p->cexp, sd));
  NPGP_TRY(stamp(p, 2 * SEC_ZZ + 1, sd));
  NPGP_CUDA(cudaEventRecord(p->ev[3], sd));

  // ---- main stream: interpolation weights of the latent field
  if (full) {
    NPGP_TRY(solve_cols(p, p->Pr, F, d, d, p->R4, p->T4, p->W4, st));   // W = (K_row + 1e-5 I)^-1 H
    svgp_pad_cols_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, d, d, p->W4, p->kp, p->Wp);
    NPGP_LAUNCH_CHECK();
  } else {
    for (int b = 0; b < d; ++b) {
      const double* Pb = p->Pr + (long)b * MM;
      svgp_sub_scalar_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, F + (long)b * M, c.prior_c + b, p->rhs + (long)b * M);
      NPGP_LAUNCH_CHECK();
      NPGP_TRY(solve_vec(p, Pb, p->rhs + (long)b * M, p->tmpv, p->alpha + (long)b * M, st));
      if (c.include_prior) {
        svgp_lp_part_kernel<<<1, 256, 0, st>>>(M, p->rhs + (long)b * M, p->alpha + (long)b * M, p->Kr + (long)b * MM,
                                               p->lp_part + 2 * b);
        NPGP_LAUNCH_CHECK();
      }
    }
  }
  return NPGP_OK;
}

// The latent field at n rows x (matrix free): fx (n,P) = Sigma(x) (full) or ell_x (d,n) = ell(x) (diag).  Needs svgp_zside.
static int svgp_row_field(npgp_svgp_plan* p, int n, const double* x, const double* theta, cudaStream_t st) {
  const npgp_svgp_config& c = p->c;
  const int M = c.M, d = c.d;
  const double* Z = theta + p->off_Z;
  if (c.variant == 1) {
    NPGP_TRY(npgp_rbf_matvec_fwd(d, 1, d, n, M, x, Z, c.row_lam, c.row_os, p->Wp, nullptr, 0, p->Hx, st));
    return npgp_sigma_from_h_fwd(d, n, p->Hx, theta + p->off_D, p->fx, st);
  }
  return npgp_rbf_matvec_fwd(d, d, 1, n, M, x, Z, c.prior_lam, c.prior_os, p->alpha, c.prior_c, 1, p->ell_x, st);
}

// K(X,Z) of n rows as digit planes (p->Ad) with the per-split partials of K u (stride ku_stride).  Needs svgp_row_field and u.
static int svgp_kxz_digits(npgp_svgp_plan* p, int n, const double* x, const double* theta, double* ku_part, long ku_stride,
                           cudaStream_t st) {
  const npgp_svgp_config& c = p->c;
  const double* Z = theta + p->off_Z;
  if (c.variant == 1)
    return npgp_gibbs_full_fwd_digits(c.d, n, c.M, x, p->fx, Z, p->fz, c.kernel_jitter, p->scal, p->Ad, p->u, ku_part,
                                      ku_stride, st);
  return npgp_gibbs_diag_fwd_digits(c.d, n, c.M, x, p->ell_x, Z, p->fz, p->scal, p->Ad, p->u, ku_part, ku_stride, st);
}

// ---------------------------------------------------------------------------------------------------------------------
// forward: -ELBO share of this rank into grad[n_pad]; leaves everything the backward needs in the workspace
// ---------------------------------------------------------------------------------------------------------------------
static int svgp_forward(npgp_svgp_plan* p, const double* x, const double* y, const double* theta, double* grad, int* status,
                        cudaStream_t st) {
  const npgp_svgp_config& c = p->c;
  const int M = c.M, d = c.d, B = c.B_local;
  const double* s = p->scal;
  const double* noise = p->scal + 1;
  p->prepared = false;  // overwrites the Z-side factors, mu_part, q_part and the digit planes
  p->sample_ready = false;

  NPGP_TRY(svgp_zside(p, theta, status, st));
  NPGP_TRY(svgp_row_field(p, B, x, theta, st));
  NPGP_TRY(stamp(p, 2 * SEC_FIELD + 1, st));
  NPGP_CUDA(cudaStreamWaitEvent(st, p->ev[10], 0));

  // ---- data pass: K(X_B,Z) as digit planes (+ partial K u), T = K C with the row dot and K^T g_mu, E[log-lik]
  NPGP_TRY(stamp(p, 2 * SEC_KXZ, st));
  NPGP_TRY(svgp_kxz_digits(p, B, x, theta, p->mu_part, B, st));
  NPGP_TRY(npgp_mu_gmu_parts(B, y, p->mu_part, p->nsplit, B, noise, 1.0 / c.B_global, p->mu, p->gmu0, st));
  NPGP_TRY(stamp(p, 2 * SEC_KXZ + 1, st));
  NPGP_CUDA(cudaStreamWaitEvent(st, p->ev[3], 0));  // C and its digit planes (computed under the tile kernel above)
  NPGP_TRY(stamp(p, 2 * SEC_RQ, st));
  NPGP_TRY(npgp_o8_rowquad_digits(B, M, p->Ad, nullptr, s, p->Cd, p->cexp, nullptr, 0, p->T, M, p->q_part, B, p->gmu0,
                                  p->du_part, st));
  NPGP_TRY(stamp(p, 2 * SEC_RQ + 1, st));  // (the partial column sums du_part are added up in the backward, off this stream)
  NPGP_TRY(stamp(p, 2 * SEC_ELL, st));
  NPGP_CUDA(cudaMemsetAsync(p->skip_count, 0, sizeof(int), st));
  NPGP_TRY(npgp_gauss_ell_parts(B, y, p->mu, p->q_part, M / 64, B, s, c.jitter_xx, c.min_var, noise, 1.0 / c.B_global, nullptr,
                                p->gmu, p->gv, p->acc4, p->skip_count, p->skip_rows, p->gwork, p->gwork_bytes, st));
  svgp_scale_vec_kernel<<<ceil_div(B, 256), 256, 0, st>>>(B, 2.0, p->gv, p->gv2);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(stamp(p, 2 * SEC_ELL + 1, st));
  {
    AssembleArgs a;
    memset(&a, 0, sizeof(a));
    a.variant = c.variant, a.M = M, a.d = d, a.nblk_kl = p->nblk_kl, a.include_prior = c.include_prior, a.B_local = B;
    a.n_pad = p->n_pad, a.rep = 1.0 / c.world_size, a.N_total = (double)c.N_total, a.B_global = (double)c.B_global;
    a.acc4 = p->acc4, a.kl_part = p->kl_part, a.lp_part = p->lp_part, a.grad = grad;
    svgp_loss_kernel<<<1, 32, 0, st>>>(a);
    NPGP_LAUNCH_CHECK();
  }
  p->fwd_done = true;
  return NPGP_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// backward: fills grad[0 .. n_pad) and the loss slot
// ---------------------------------------------------------------------------------------------------------------------
static int svgp_backward(npgp_svgp_plan* p, const double* x, const double* theta, double* grad, void* comm, cudaStream_t st) {
  const npgp_svgp_config& c = p->c;
  const int M = c.M, d = c.d, B = c.B_local, full = c.variant == 1;
  const long MM = (long)M * M;
  const double* Z = theta + p->off_Z;
  const double* F = theta + p->off_F;
  const double* Dm = theta + p->off_D;
  const double* m = theta + p->off_m;
  const double* s = p->scal;
  const double rep = 1.0 / c.world_size;
  cudaStream_t sd = p->side, sd2 = p->side2;

  // ---- side stream: dC = K^T diag(g_v) K on the int8 tensor cores, then the latency-bound O(M^3) chain to dKzz
  NPGP_TRY(fork_stream(st, sd, p->ev[4]));
  NPGP_TRY(stamp(p, 2 * SEC_SYRK, sd));
  NPGP_TRY(npgp_o8_syrk_digits(B, M, p->Ad, s, 1.0, p->acc4 + 3, p->skip_count, p->skip_rows, 0, p->dC, M, p->syrk_part,
                               p->syrk_part_bytes, sd));
  NPGP_TRY(stamp(p, 2 * SEC_SYRK + 1, sd));
  NPGP_TRY(stamp(p, 2 * SEC_M3, sd));
  // dE = P dC P^T and E dE = (E P)(dC P^T): with W = dC P^T both follow from ONE product
  NPGP_TRY(npgp_dgemm(0, 1, M, M, M, 1.0, p->dC, M, p->P, M, 0.0, p->W2, M, 0, 2, 0, sd));
  NPGP_TRY(fork_stream(sd, sd2, p->ev[5]));
  {  // dL_s branch (and dm = P du, which the main chain needs only after its next product)
    NPGP_TRY(npgp_o8_sum_partials(p->nb128, M, p->du_part, p->du, sd2));  // du = K^T g_mu from the row-block partials
    NPGP_TRY(npgp_gemv_n(M, M, p->P, M, p->du, p->dm, sd2));
    NPGP_CUDA(cudaEventRecord(p->ev[11], sd2));
    // dE = P (dC P^T) is symmetric (lower tiles + mirror); only the lower triangle of dE Ls is used
    NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 1.0, p->P, M, p->W2, M, 0.0, p->dE, M, 1, 0, 1, sd2));
    NPGP_TRY(npgp_symmetrize(M, p->dE, M, 0, sd2));
    NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 2.0, p->dE, M, p->Ls_t, M, 0.0, p->dLs, M, 0, 1, 1, sd2));
    svgp_grad_m_ls_kernel<<<grid2(M), kBlk2, 0, sd2>>>(M, p->dLs, p->Ls_t, p->dm, m, rep / (double)c.N_total,
                                                      grad + p->off_Ls, grad + p->off_m);
    NPGP_LAUNCH_CHECK();
    // g_m and g_Ls (99 % of the flat gradient) are final here: their all-reduce runs under the rest of the O(M^3) chain
    if (comm) NPGP_TRY(npgp_allreduce_f64(comm, grad + p->off_m, (long)M + MM, sd2));
    NPGP_CUDA(cudaEventRecord(p->ev[6], sd2));
  }
  // Phi keeps the lower triangle only: the tiles strictly above the diagonal are not computed (half the flops of the
  // longest product of the chain)
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 2.0, p->EP, M, p->W2, M, 0.0, p->X, M, 0, 0, 1, sd));
  NPGP_CUDA(cudaStreamWaitEvent(sd, p->ev[11], 0));  // dm
  svgp_addr_phi_kernel<<<grid2(M), kBlk2, 0, sd>>>(M, p->X, m, p->dm);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(npgp_dgemm(1, 0, M, M, M, 1.0, p->P, M, p->X, M, 0.0, p->Y, M, 2, 1, 0, sd));
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 1.0, p->Y, M, p->P, M, 0.0, p->dK, M, 0, 1, 0, sd));
  svgp_sym_avg_kernel<<<dim3(ceil_div(M, 32), ceil_div(M, 32)), kBlk2, 0, sd>>>(M, p->dK, p->dKzz);
  NPGP_LAUNCH_CHECK();
  double* gZ = c.learn_z ? p->gZ : nullptr;
  if (full)
    NPGP_TRY(npgp_gibbs_full_bwd(d, M, M, Z, p->fz, Z, p->fz, c.kernel_jitter, s, p->dKzz, M, nullptr, nullptr, nullptr,
                                 p->dfz_acc, gZ, p->dfz_acc, gZ, p->ds_acc, sd));
  else
    NPGP_TRY(npgp_gibbs_diag_bwd(d, M, M, Z, p->fz, Z, p->fz, s, p->dKzz, M, nullptr, nullptr, nullptr, p->dfz_acc, gZ,
                                 p->dfz_acc, gZ, p->ds_acc, sd));
  NPGP_CUDA(cudaStreamWaitEvent(sd, p->ev[6], 0));
  NPGP_TRY(stamp(p, 2 * SEC_M3 + 1, sd));
  NPGP_CUDA(cudaEventRecord(p->ev[7], sd));

  // ---- main stream: backward of the data term through K(X_B,Z) (G formed inside the kernel), then the field interpolation
  NPGP_TRY(stamp(p, 2 * SEC_KXZB, st));
  if (full)
    NPGP_TRY(npgp_gibbs_full_bwd(d, B, M, x, p->fx, Z, p->fz, c.kernel_jitter, s, p->T, M, p->gv2, p->gmu, p->u, p->dfx,
                                 nullptr, p->dfz_acc, gZ, p->ds_acc, st));
  else
    NPGP_TRY(npgp_gibbs_diag_bwd(d, B, M, x, p->ell_x, Z, p->fz, s, p->T, M, p->gv2, p->gmu, p->u, p->dfx, nullptr,
                                 p->dfz_acc, gZ, p->ds_acc, st));
  NPGP_TRY(stamp(p, 2 * SEC_KXZB + 1, st));
  NPGP_TRY(stamp(p, 2 * SEC_FIELDB, st));
  if (full) {
    NPGP_TRY(npgp_sigma_from_h_bwd(d, B, p->Hx, Dm, p->dfx, p->dHx, p->dD_acc, st));
    NPGP_TRY(npgp_rbf_matvec_bwd(d, 1, d, B, M, x, Z, c.row_lam, c.row_os, p->Wp, p->dHx, p->dW, gZ, st));
    NPGP_TRY(solve_cols(p, p->Pr, p->dW, d, d, p->R4b, p->T4b, p->beta4, st));  // beta = Kr^-1 dW
    if (c.learn_z) {
      // dELBO/dKr = -beta W^T
      svgp_outer_kernel<<<grid2(M), kBlk2, 0, st>>>(M, d, -1.0, p->beta4, p->kp, p->W4, p->kp, p->Gk);
      NPGP_LAUNCH_CHECK();
      NPGP_TRY(npgp_gibbs_diag_bwd(d, M, M, Z, p->lam_b, Z, p->lam_b, c.row_os, p->Gk, M, nullptr, nullptr, nullptr,
                                   p->dummy_ell, gZ, p->dummy_ell + (long)d * M, gZ, nullptr, st));
    }
  } else {
    svgp_mul_vec_kernel<<<ceil_div((long)d * B, 256), 256, 0, st>>>((long)d * B, p->dfx, p->ell_x, p->dlog);
    NPGP_LAUNCH_CHECK();
    NPGP_TRY(npgp_rbf_matvec_bwd(d, d, 1, B, M, x, Z, c.prior_lam, c.prior_os, p->alpha, p->dlog, p->dalpha, gZ, st));
    const double pw = c.include_prior ? rep / ((double)c.N_total * M) : 0.0;
    for (int b = 0; b < d; ++b) {
      const double* Pb = p->Pr + (long)b * MM;
      const double* lamb = p->lam_b + (long)b * d * M;
      NPGP_TRY(solve_vec(p, Pb, p->dalpha + (long)b * M, p->tmpv, p->beta_v, st));
      svgp_diag_prior_vec_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, pw, p->beta_v, p->alpha + (long)b * M,
                                                                  p->g_logell + (long)b * M, p->rv);
      NPGP_LAUNCH_CHECK();
      if (c.learn_z) {
        // dELBO/dKp_b = -beta alpha^T (+ prior: pw (0.5 alpha alpha^T - 0.5 Kp^-1))
        const double* Gm = nullptr;
        if (c.include_prior) {
          NPGP_TRY(npgp_dgemm(1, 0, M, M, M, -0.5 * pw, Pb, M, Pb, M, 0.0, p->Gk, M, 2, 1, 0, st));
          Gm = p->Gk;
        }
        NPGP_TRY(npgp_gibbs_diag_bwd(d, M, M, Z, lamb, Z, lamb, c.prior_os + b, Gm, M, nullptr, p->rv, p->alpha + (long)b * M,
                                     p->dummy_ell, gZ, p->dummy_ell + (long)d * M, gZ, nullptr, st));
      }
    }
  }
  NPGP_TRY(stamp(p, 2 * SEC_FIELDB + 1, st));

  // ---- join the O(M^3) chain and assemble the small gradient blocks + the loss slot
  NPGP_CUDA(cudaStreamWaitEvent(st, p->ev[7], 0));
  NPGP_TRY(stamp(p, 2 * SEC_ASM, st));
  if (full) NPGP_TRY(npgp_sigma_from_h_bwd(d, M, F, Dm, p->dfz_acc, p->dHz, p->dD_acc, st));
  AssembleArgs a;
  memset(&a, 0, sizeof(a));
  a.variant = c.variant, a.M = M, a.d = d, a.nblk_kl = p->nblk_kl, a.include_prior = c.include_prior, a.B_local = B;
  a.n_pad = p->n_pad, a.n_params = p->n_params, a.rep = rep, a.N_total = (double)c.N_total, a.B_global = (double)c.B_global;
  a.scal = p->scal, a.acc4 = p->acc4, a.kl_part = p->kl_part, a.ds_acc = p->ds_acc, a.gZ = p->gZ;
  a.beta4 = p->beta4, a.kp = p->kp, a.dHz = p->dHz, a.dD_acc = p->dD_acc;
  a.g_logell = p->g_logell, a.dfz_acc = p->dfz_acc, a.ell_z = p->fz, a.lp_part = p->lp_part;
  a.grad = grad, a.off_Z = p->off_Z, a.off_F = p->off_F, a.off_D = p->off_D, a.off_os = p->off_os, a.off_noise = p->off_noise;
  svgp_assemble_kernel<<<1, 256, 0, st>>>(a);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(stamp(p, 2 * SEC_ASM + 1, st));
  return NPGP_OK;
}

static int svgp_check_args(npgp_svgp_plan* p, const double* x, const double* y, const double* theta, double* grad) {
  if (!p || !x || !y || !theta || !grad) return NPGP_EINVAL;
  if ((reinterpret_cast<uintptr_t>(theta) & 15) || (reinterpret_cast<uintptr_t>(grad) & 15)) return NPGP_EUNSUPPORTED;
  return NPGP_OK;
}

/* Forward pass: everything up to the expected log-likelihood; leaves K(X_B,Z) (digit planes), T = K C, the gradient seeds and
 * the Z-side factors in the plan's workspace for npgp_svgp_elbo_bwd.  status (optional, device, sticky): bit 0 is set when a
 * Cholesky failed. */
extern "C" int npgp_svgp_elbo_fwd(npgp_svgp_plan* p, const double* x, const double* y, const double* theta, double* grad,
                                  int* status, cudaStream_t stream) {
  NPGP_TRY(svgp_check_args(p, x, y, theta, grad));
  return svgp_forward(p, x, y, theta, grad, status, stream);
}

/* Backward pass of the forward that ran last on this plan (same x, theta): grad[0 .. n_pad) = d(-ELBO share)/d theta of this
 * rank's rows (replicated KL / prior terms weighted 1 / world_size), grad[n_pad] = this rank's share of -ELBO. */
extern "C" int npgp_svgp_elbo_bwd(npgp_svgp_plan* p, const double* x, const double* theta, double* grad, cudaStream_t stream) {
  if (!p || !x || !theta || !grad) return NPGP_EINVAL;
  if (!p->fwd_done) return NPGP_EINVAL;
  return svgp_backward(p, x, theta, grad, nullptr, stream);
}

/* One training step: forward, backward, optional all-reduce (comm: an npgp communicator, NULL for a single rank), sticky
 * status update on the (all-reduced) loss, guarded Adam on theta (mask: 0 entries are frozen; may be NULL). */
extern "C" int npgp_svgp_step(npgp_svgp_plan* p, const double* x, const double* y, double* theta, double* grad, double* adam_m,
                              double* adam_v, const double* mask, double* step_dev, int* status, double lr, double beta1,
                              double beta2, double eps, void* comm, cudaStream_t stream) {
  NPGP_TRY(svgp_check_args(p, x, y, theta, grad));
  if (!adam_m || !adam_v || !step_dev || !status) return NPGP_EINVAL;
  NPGP_TRY(svgp_forward(p, x, y, theta, grad, status, stream));
  NPGP_TRY(svgp_backward(p, x, theta, grad, comm, stream));
  if (comm) {  // what the early all-reduce (m, Ls) did not cover: [Z, field] in front of it, [scalars, padding, loss] behind
    NPGP_TRY(stamp(p, 2 * SEC_AR, stream));
    NPGP_TRY(npgp_allreduce_f64_pair(comm, grad, p->off_m, grad + p->off_os, p->n_pad + 2 - p->off_os, stream));
    NPGP_TRY(stamp(p, 2 * SEC_AR + 1, stream));
  }
  NPGP_TRY(stamp(p, 2 * SEC_ADAM, stream));
  NPGP_TRY(npgp_status_update(status, nullptr, grad + p->n_pad, stream));
  NPGP_TRY(npgp_adam_step_guarded(p->n_pad, theta, grad, adam_m, adam_v, mask, lr, beta1, beta2, eps, step_dev, 1.0, status,
                                  stream));
  NPGP_TRY(stamp(p, 2 * SEC_ADAM + 1, stream));
  return NPGP_OK;
}

/* Z-side factors of the posterior for theta (the forward's Z-side chain), side streams joined before the return. */
extern "C" int npgp_svgp_predict_prepare(npgp_svgp_plan* p, const double* theta, int* status, cudaStream_t stream) {
  if (!p || !theta) return NPGP_EINVAL;
  p->fwd_done = false;  // the forward's Z-side factors and partial sums are overwritten
  p->prepared = false;
  p->sample_ready = false;  // the sampler's G and W derive from the factors about to be replaced
  NPGP_TRY(svgp_zside(p, theta, status, stream));
  NPGP_CUDA(cudaStreamWaitEvent(stream, p->ev[3], 0));  // u, C, its digit planes (the side chain after both side streams)
  p->prepared = true;
  return NPGP_OK;
}

// Where the K u partials of an nc-row chunk of prediction or sampling go.  They take nsplit(nc) x nc doubles, and nsplit is not
// monotone in the row count: a short last chunk can need more than mu_part holds.  Then they go to the T buffer
// (B x M >= (M / 64) x nc), which neither prediction nor sampling uses.
static double* svgp_ku_parts(npgp_svgp_plan* p, int nc, int* nsplit) {
  *nsplit = npgp_gibbs_digits_splits(nc, p->c.M);
  return (long)*nsplit * nc <= (long)p->nsplit * p->c.B_local ? p->mu_part : p->T;
}

/* Posterior marginals at n rows, streamed through the workspace in chunks of B_local rows (one stream, no allocation). */
extern "C" int npgp_svgp_predict(npgp_svgp_plan* p, long n, const double* xs, const double* ys, const double* theta, double* mean,
                                 double* var_f, double* var_y, double* field, double* lpd, double* sums, cudaStream_t stream) {
  if (!p || n < 0 || !p->prepared) return NPGP_EINVAL;
  if (n == 0) return NPGP_OK;
  if (!xs || !theta || !mean || !var_f || ((lpd || sums) && !ys)) return NPGP_EINVAL;
  const npgp_svgp_config& c = p->c;
  const int M = c.M, d = c.d, B = c.B_local, nq = M / 64;
  p->fwd_done = false;  // mu_part, q_part, the digit planes and the row field are overwritten
  for (long lo = 0; lo < n; lo += B) {
    const int nc = (int)(n - lo < B ? n - lo : B);
    const double* x = xs + lo * d;
    const double* y = ys ? ys + lo : nullptr;
    NPGP_TRY(svgp_row_field(p, nc, x, theta, stream));
    if (field) {
      if (c.variant == 1)
        NPGP_CUDA(cudaMemcpyAsync(field + lo * p->P6, p->fx, sizeof(double) * nc * p->P6, cudaMemcpyDeviceToDevice, stream));
      else  // (d, nc) chunk -> columns [lo, lo + nc) of the caller's (d, n)
        NPGP_CUDA(cudaMemcpy2DAsync(field + lo, sizeof(double) * n, p->ell_x, sizeof(double) * nc, sizeof(double) * nc, d,
                                    cudaMemcpyDeviceToDevice, stream));
    }
    int nsplit;
    double* mu_part = svgp_ku_parts(p, nc, &nsplit);
    NPGP_TRY(svgp_kxz_digits(p, nc, x, theta, mu_part, nc, stream));
    NPGP_TRY(npgp_o8_rowquad_digits(nc, M, p->Ad, nullptr, p->scal, p->Cd, p->cexp, nullptr, 0, nullptr, M, p->q_part, nc,
                                    nullptr, nullptr, stream));
    const int nblk = ceil_div(nc, 256);  // <= the 3 ceil(B / 256) doubles of gwork
    svgp_predict_finish_kernel<<<nblk, 256, 0, stream>>>(nc, mu_part, nsplit, p->q_part, nq, p->scal, c.jitter_xx, c.min_var, y,
                                                         mean + lo, var_f + lo, var_y ? var_y + lo : nullptr,
                                                         lpd ? lpd + lo : nullptr, p->gwork);
    NPGP_LAUNCH_CHECK();
    if (sums) {
      svgp_predict_sums_kernel<<<1, 256, 0, stream>>>(nblk, nc, p->gwork, sums);
      NPGP_LAUNCH_CHECK();
    }
  }
  return NPGP_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// posterior sample fields (modified predictive process under q(u)): with the factors of the last predict_prepare,
//     f_s(x) = mean(x) + k(x)^T W_s + sqrt(r(x)) xi_s(x),  W = P^T Ls E,  r(x) = max(s + jitter_xx - k^T P^T P k, 0)
// Everything beyond the plan lives in the caller's `work`: G = P^T P and its planes, W^T (Sp = 64 ceil(S / 64) rows; E^T and
// Y = E^T Ls^T on the way) and its planes, and the B_local x Sp chunk of F = K W.
// ---------------------------------------------------------------------------------------------------------------------
/* E^T of S draws (Sp x W, zero rows s >= S), the one generator of both samplers' E (the SGPR one calls it from sgpr.py). */
extern "C" int npgp_sample_normals(int W, int S, int Sp, unsigned long long seed, double* Et, cudaStream_t st) {
  if (W < 0 || S < 0 || Sp < S) return NPGP_EINVAL;
  if ((long)Sp * W == 0) return NPGP_OK;
  if (!Et) return NPGP_EINVAL;
  sample_normals_kernel<<<(unsigned)ceil_div((long)Sp * W, 256), 256, 0, st>>>(W, S, Sp, seed, Et);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

struct SampleBufs {
  double *G, *Y, *Wt, *F;
  int8_t *Gd, *Wd;
  int *gexp, *wexp;
};

static inline int sample_pad(int S) { return (S + 63) / 64 * 64; }

static long sample_layout(const npgp_svgp_config& c, int S, void* work, SampleBufs* b) {
  const int M = c.M, Sp = sample_pad(S);
  Carver w{static_cast<char*>(work), 0};
  b->G = w.take<double>((long)M * M);
  b->Gd = w.take<int8_t>(npgp_o8_digits_bytes(M, M, 64)), b->gexp = w.take<int>(M);
  b->Y = w.take<double>((long)Sp * M), b->Wt = w.take<double>((long)Sp * M);
  b->Wd = w.take<int8_t>(npgp_o8_digits_bytes(Sp, M, 64)), b->wexp = w.take<int>(Sp);
  b->F = w.take<double>((long)c.B_local * Sp);
  return w.off + 256;
}

extern "C" long npgp_svgp_sample_workspace_bytes(const npgp_svgp_config* cfg, int S) {
  if (!cfg || S < 1 || S > 1024) return -1;
  npgp_svgp_plan tmp;
  tmp.c = *cfg;
  long bytes;
  if (svgp_layout(&tmp, nullptr, &bytes)) return -1;
  SampleBufs b;
  return sample_layout(*cfg, S, nullptr, &b);
}

/* The row-independent part of S draws: G = P^T P, W = P^T Ls E and their digit planes into work (one stream). */
extern "C" int npgp_svgp_sample_prepare(npgp_svgp_plan* p, const double* theta, int S, unsigned long long seed, void* work,
                                        long work_bytes, cudaStream_t st) {
  if (!p || !theta || !work || S < 1 || S > 1024 || !p->prepared) return NPGP_EINVAL;
  if (reinterpret_cast<uintptr_t>(work) & 255) return NPGP_EUNSUPPORTED;
  SampleBufs b;
  if (work_bytes < sample_layout(p->c, S, work, &b)) return NPGP_EWORKSPACE;
  const int M = p->c.M, Sp = sample_pad(S);
  p->fwd_done = false;
  p->sample_ready = false;
  // G = P^T P: op(A) = P^T upper, op(B) = P lower; the lower tiles, mirrored
  NPGP_TRY(npgp_dgemm(1, 0, M, M, M, 1.0, p->P, M, p->P, M, 0.0, b.G, M, 2, 1, 1, st));
  NPGP_TRY(npgp_symmetrize(M, b.G, M, 0, st));
  NPGP_TRY(npgp_o8_slice_rows(M, M, b.G, M, 64, b.Gd, b.gexp, st));
  // W^T = E^T Ls^T P: E^T into Wt, Y = E^T Ls^T (Ls_t lower), then Wt = Y P (P lower)
  NPGP_TRY(npgp_sample_normals(M, S, Sp, seed, b.Wt, st));
  NPGP_TRY(npgp_dgemm(0, 1, Sp, M, M, 1.0, b.Wt, M, p->Ls_t, M, 0.0, b.Y, M, 0, 2, 0, st));
  NPGP_TRY(npgp_dgemm(0, 0, Sp, M, M, 1.0, b.Y, M, p->P, M, 0.0, b.Wt, M, 0, 1, 0, st));
  NPGP_TRY(npgp_o8_slice_rows(Sp, M, b.Wt, M, 64, b.Wd, b.wexp, st));
  p->sample_S = S;
  p->sample_seed = seed;
  p->sample_work = work;
  p->sample_ready = true;
  return NPGP_OK;
}

/* S draws at n rows, streamed in chunks of B_local rows: out (S, n), leading dimension ldo. */
extern "C" int npgp_svgp_sample(npgp_svgp_plan* p, long n, const double* xs, long row_offset, const double* theta, int noise,
                                double* out, long ldo, void* work, long work_bytes, cudaStream_t st) {
  if (!p || n < 0 || row_offset < 0 || !p->sample_ready || work != p->sample_work) return NPGP_EINVAL;
  SampleBufs b;
  if (work_bytes < sample_layout(p->c, p->sample_S, work, &b)) return NPGP_EWORKSPACE;
  if (n == 0) return NPGP_OK;
  if (!xs || !theta || !out || ldo < n || n > (1L << 48) - row_offset) return NPGP_EINVAL;  // row index: 48 key bits
  const npgp_svgp_config& c = p->c;
  const int M = c.M, d = c.d, B = c.B_local, nq = M / 64, S = p->sample_S, Sp = sample_pad(S);
  p->fwd_done = false;  // mu_part, q_part, the digit planes and the row field are overwritten
  for (long lo = 0; lo < n; lo += B) {
    const int nc = (int)(n - lo < B ? n - lo : B);
    const double* x = xs + lo * d;
    NPGP_TRY(svgp_row_field(p, nc, x, theta, st));
    int nsplit;
    double* mu_part = svgp_ku_parts(p, nc, &nsplit);
    NPGP_TRY(svgp_kxz_digits(p, nc, x, theta, mu_part, nc, st));
    NPGP_TRY(npgp_o8_rowquad_digits(nc, M, p->Ad, nullptr, p->scal, b.Gd, b.gexp, nullptr, 0, nullptr, M, p->q_part, nc,
                                    nullptr, nullptr, st));  // k^T G k
    NPGP_TRY(npgp_o8_gemm_digits(nc, Sp, M, p->Ad, nullptr, p->scal, b.Wd, b.wexp, b.F, Sp, st));  // F = K W
    svgp_sample_finish_kernel<<<ceil_div(nc, 32), dim3(32, 8), 0, st>>>(nc, S, mu_part, nsplit, p->q_part, nq, p->scal,
                                                                        c.jitter_xx, noise, b.F, Sp, p->sample_seed,
                                                                        row_offset + lo, out + lo, ldo);
    NPGP_LAUNCH_CHECK();
  }
  return NPGP_OK;
}

/* device pointers into the plan's workspace, for inspection / prediction: which = 0 mu (B), 1 T (B,M), 2 P (M,M), 3 C (M,M),
 * 4 u (M), 5 gmu (B), 6 gv (B), 7 acc4 (4), 8 info (ints) */
extern "C" const void* npgp_svgp_buffer(npgp_svgp_plan* p, int which) {
  if (!p) return nullptr;
  switch (which) {
    case 0: return p->mu;
    case 1: return p->T;
    case 2: return p->P;
    case 3: return p->C;
    case 4: return p->u;
    case 5: return p->gmu;
    case 6: return p->gv;
    case 7: return p->acc4;
    case 8: return p->info;
    default: return nullptr;
  }
}
