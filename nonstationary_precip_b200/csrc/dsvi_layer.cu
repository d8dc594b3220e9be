// One output dimension of a deep-GP layer behind the C ABI: npgp_dsvi_layer_fwd / npgp_dsvi_layer_bwd.
//
// Replaces, for a whitened SVGP layer with an RBF-ARD * Scale kernel (reference models/dgps.py:15-46 through GPyTorch's
// VariationalStrategy / DeepGPLayer.__call__, SURVEY.md Appendix B.2/B.5), the marginal predictive distribution at the rows
// X (which are S x B samples of the previous layer, or the B data rows for the first layer) and its analytic backward:
//     Kzz = os RBF(Z,Z; ls) + jitter I,  L = chol(Kzz),  P = L^-1,  u = P^T m,  C = sym(P^T (Ls Ls^T - I) P)
//     K = os RBF(X,Z; ls),   mean = K u,   var = max(os + add_var + rowdot(K C, K), min_var)
// (the mean function and the reparameterised sample h = mean + sqrt(var) eps stay with the caller: npgp_dsvi_sample).
// RBF-ARD is the constant-lengthscale case of the diagonal Gibbs kernel, so the tile kernels of gibbs_diag.cu serve, with
// analytic gradients to X, Z, ls and os; T = K C runs on the int8 tensor cores (exact, npgp_rowquad_i8) when the width
// allows; dC = K^T diag(dvar) K runs there too when all weights are equal (the last layer under a Gaussian likelihood),
// decided on the device, and on the FP64 tensor pipe otherwise (hidden layers: the weights come from the sampling chain).
// One stream, one caller-supplied workspace that carries K, T and the Z-side factors from the forward to the backward.
#include <cstring>

#include "common.cuh"
#include "svgp_glue.cuh"
#include "../../include/npgp.h"

namespace npgp {

// var_i = max(os + add_var + q_i, min_var), written as a comparison so that a NaN (a row with a missing coordinate) stays NaN
static __global__ void dsvi_var_kernel(int n, const double* __restrict__ q, const double* __restrict__ os, double add_var,
                                       double min_var, double* __restrict__ var) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < n) {
    const double v = *os + add_var + q[i];
    var[i] = (v < min_var) ? min_var : v;
  }
}

// gv_i = dvar_i where the variance was not clamped, else 0; gv2 = 2 gv; cnt += #(gv_i == gv_0); sum += gv_i
static __global__ void __launch_bounds__(256) dsvi_seed_kernel(int n, const double* __restrict__ dvar, const double* __restrict__ var,
                                                               double min_var, double* __restrict__ gv, double* __restrict__ gv2,
                                                               double* __restrict__ cnt_sum) {
  __shared__ double red[32];
  const int i = blockIdx.x * 256 + threadIdx.x;
  const double g0 = (var[0] > min_var) ? dvar[0] : 0.0;
  double c = 0.0, sgv = 0.0;
  if (i < n) {
    const double g = (var[i] > min_var) ? dvar[i] : 0.0;
    gv[i] = g;
    gv2[i] = 2.0 * g;
    c = (g == g0) ? 1.0 : 0.0;
    sgv = g;
  }
  double t = block_sum(c, red);
  if (threadIdx.x == 0) atomicAdd(&cnt_sum[0], t);  // integer-valued: exact in any order
  t = block_sum(sgv, red);
  if (threadIdx.x == 0) atomicAdd(&cnt_sum[1], t);
}

// part[k * nblk + b] = sum over block b's slice of row k of A (d x n)
static __global__ void __launch_bounds__(256) dsvi_rowsum_part_kernel(int d, long n, const double* __restrict__ A,
                                                                     double* __restrict__ part) {
  __shared__ double red[32];
  const int k = blockIdx.y, nblk = gridDim.x;
  const long per = (n + nblk - 1) / nblk;
  const long i0 = blockIdx.x * per, i1 = (i0 + per < n) ? i0 + per : n;
  double a = 0.0;
  for (long i = i0 + threadIdx.x; i < i1; i += 256) a += A[(long)k * n + i];
  const double t = block_sum(a, red);
  if (threadIdx.x == 0) part[k * nblk + blockIdx.x] = t;
  (void)d;
}

// dls[k] = sum_b partX[k][b] + sum_j (dez[k][j]);  dos = ds_acc + sum gv
static __global__ void __launch_bounds__(256) dsvi_finish_kernel(int d, int M, int nblk, const double* __restrict__ partX,
                                                                const double* __restrict__ dez, const double* __restrict__ ds_acc,
                                                                const double* __restrict__ cnt_sum, double* __restrict__ dls,
                                                                double* __restrict__ dos) {
  __shared__ double red[32];
  for (int k = 0; k < d; ++k) {
    double a = 0.0;
    for (int b = threadIdx.x; b < nblk; b += 256) a += partX[k * nblk + b];
    for (int j = threadIdx.x; j < M; j += 256) a += dez[(long)k * M + j];
    const double t = block_sum(a, red);
    if (threadIdx.x == 0) dls[k] = t;
  }
  if (threadIdx.x == 0) dos[0] = ds_acc[0] + cnt_sum[1];
}

// out = tril(A) (M x M)
static __global__ void dsvi_tril_out_kernel(int M, const double* __restrict__ A, double* __restrict__ out) {
  const int c = blockIdx.x * 32 + threadIdx.x, r = blockIdx.y * 8 + threadIdx.y;
  if (r < M && c < M) out[(long)r * M + c] = (c <= r) ? A[(long)r * M + c] : 0.0;
}

struct DsviWs {
  double *lam, *lamx, *Kzz, *P, *Ls_t, *E, *EP, *C, *Cs, *u, *K, *T, *q;
  double *gv, *gv2, *cnt_sum, *du, *dC, *W2, *dE, *dLs, *X2, *Y, *dK, *dKzz, *dex, *dez, *ds_acc, *partX;
  int* flags;
  void* i8;
  long i8_bytes, flags_bytes, total;
};

static int dsvi_layout(int n, int M, int d, void* base, DsviWs* w) {
  if (n <= 0 || M <= 0 || d < 1 || d > 6) return NPGP_EINVAL;
  if (M & 1) return NPGP_EUNSUPPORTED;  // even leading dimensions throughout
  char* b = static_cast<char*>(base);
  long off = 0;
  auto take = [&](long bytes) {
    off = (off + 255) & ~255L;
    char* p = b ? b + off : nullptr;
    off += bytes;
    return p;
  };
  const long MM = (long)M * M, D8 = sizeof(double);
  w->lam = (double*)take(D8 * d * M), w->lamx = (double*)take(D8 * d * (long)n);
  w->Kzz = (double*)take(D8 * MM), w->P = (double*)take(D8 * MM), w->Ls_t = (double*)take(D8 * MM);
  w->E = (double*)take(D8 * MM), w->EP = (double*)take(D8 * MM), w->C = (double*)take(D8 * MM), w->Cs = (double*)take(D8 * MM);
  w->u = (double*)take(D8 * M);
  w->K = (double*)take(D8 * (long)n * M), w->T = (double*)take(D8 * (long)n * M), w->q = (double*)take(D8 * n);
  w->gv = (double*)take(D8 * n), w->gv2 = (double*)take(D8 * n), w->cnt_sum = (double*)take(D8 * 2);
  w->du = (double*)take(D8 * M), w->dC = (double*)take(D8 * MM), w->W2 = (double*)take(D8 * MM), w->dE = (double*)take(D8 * MM);
  w->dLs = (double*)take(D8 * MM), w->X2 = (double*)take(D8 * MM), w->Y = (double*)take(D8 * MM), w->dK = (double*)take(D8 * MM);
  w->dKzz = (double*)take(D8 * MM);
  w->dex = (double*)take(D8 * d * (long)n), w->dez = (double*)take(D8 * d * M), w->ds_acc = (double*)take(D8 * 2);
  w->partX = (double*)take(D8 * d * 256);
  w->flags_bytes = npgp_potrf_flow_workspace_bytes(M);
  w->flags = (int*)take(w->flags_bytes);
  long i8 = 0;
  if (M % 64 == 0) i8 = npgp_rowquad_i8_workspace_bytes(n, M);
  if (M % 128 == 0) {
    const long s8 = npgp_syrk_i8_workspace_bytes(n, M);
    if (s8 > i8) i8 = s8;
  }
  w->i8_bytes = i8;
  w->i8 = take(i8 > 0 ? i8 : 8);
  w->total = off + 256;
  return NPGP_OK;
}

#define NPGP_TRY(call)     \
  do {                     \
    int rc__ = (call);     \
    if (rc__) return rc__; \
  } while (0)

static inline dim3 g2(int M) { return dim3(ceil_div(M, 32), ceil_div(M, 8)); }
static const dim3 kB2(32, 8);
constexpr int kI8MinRows = 4096;  // below this the slicing passes of the int8 path cost more than they save

}  // namespace npgp

using namespace npgp;

extern "C" long npgp_dsvi_layer_workspace_bytes(int n, int M, int d) {
  DsviWs w;
  if (dsvi_layout(n, M, d, nullptr, &w)) return -1;
  return w.total;
}

/* X (n,d), Z (M,d), ls (d) and os (1): constrained lengthscales / outputscale on the device, m (M), Ls (M,M; lower part used).
 * mean (n) = K u (the caller adds the mean function), var (n); *info (device) = 0 or the Cholesky's failure code.
 * work (256-byte aligned, npgp_dsvi_layer_workspace_bytes) must reach npgp_dsvi_layer_bwd unchanged. */
extern "C" int npgp_dsvi_layer_fwd(int n, int M, int d, const double* X, const double* Z, const double* ls, const double* os,
                                   const double* m, const double* Ls, double jitter, double add_var, double min_var,
                                   double* mean, double* var, int* info, void* work, long work_bytes, cudaStream_t st) {
  if (!X || !Z || !ls || !os || !m || !Ls || !mean || !var || !info || !work) return NPGP_EINVAL;
  if (reinterpret_cast<uintptr_t>(work) & 255) return NPGP_EUNSUPPORTED;
  DsviWs w;
  NPGP_TRY(dsvi_layout(n, M, d, work, &w));
  if (work_bytes < w.total) return NPGP_EWORKSPACE;
  svgp_bcast_rows_kernel<<<ceil_div(M, 256), 256, 0, st>>>(d, M, ls, w.lam);
  NPGP_LAUNCH_CHECK();
  svgp_bcast_rows_kernel<<<ceil_div(n, 256), 256, 0, st>>>(d, n, ls, w.lamx);
  NPGP_LAUNCH_CHECK();
  // ---- Z side: Kzz -> L, P -> u, C
  NPGP_TRY(npgp_gibbs_diag_fwd(d, M, M, Z, w.lam, Z, w.lam, os, w.Kzz, M, nullptr, nullptr, st));
  svgp_add_diag_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, w.Kzz, M, jitter);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(npgp_potrf_inv_flow(M, w.Kzz, M, w.P, M, w.flags, w.flags_bytes, info, st));
  svgp_tri_skinny_t_kernel<1><<<ceil_div(M, 8), 256, 0, st>>>(M, w.P, m, w.u);
  NPGP_LAUNCH_CHECK();
  svgp_tril_copy_kernel<<<g2(M), kB2, 0, st>>>(M, Ls, w.Ls_t);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(npgp_dgemm(0, 1, M, M, M, 1.0, w.Ls_t, M, w.Ls_t, M, 0.0, w.E, M, 1, 2, 0, st));
  svgp_add_diag_kernel<<<ceil_div(M, 256), 256, 0, st>>>(M, w.E, M, -1.0);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 1.0, w.E, M, w.P, M, 0.0, w.EP, M, 0, 1, 0, st));
  NPGP_TRY(npgp_dgemm(1, 0, M, M, M, 1.0, w.P, M, w.EP, M, 0.0, w.C, M, 2, 0, 0, st));
  svgp_sym_avg_kernel<<<dim3(ceil_div(M, 32), ceil_div(M, 32)), kB2, 0, st>>>(M, w.C, w.Cs);
  NPGP_LAUNCH_CHECK();
  // ---- rows: K (+ K u), T = K C with the row dot, variance
  NPGP_CUDA(cudaMemsetAsync(mean, 0, sizeof(double) * n, st));
  NPGP_TRY(npgp_gibbs_diag_fwd(d, n, M, X, w.lamx, Z, w.lam, os, w.K, M, w.u, mean, st));
  NPGP_CUDA(cudaMemsetAsync(w.q, 0, sizeof(double) * n, st));
  if (M % 64 == 0 && n >= kI8MinRows)
    NPGP_TRY(npgp_rowquad_i8(n, M, w.K, M, w.Cs, M, w.T, M, w.q, w.i8, w.i8_bytes, st));
  else
    NPGP_TRY(npgp_rowquad(n, M, w.K, M, w.Cs, M, w.T, M, w.q, st));
  dsvi_var_kernel<<<ceil_div(n, 256), 256, 0, st>>>(n, w.q, os, add_var, min_var, var);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}

/* Gradients of a scalar whose derivatives w.r.t. this layer's mean / var outputs are dmean / dvar (n each); var: the
 * forward's output (clamped entries pass no gradient).  All outputs are OVERWRITTEN: dX (n,d; may be NULL), dZ (M,d), dls (d),
 * dos (1), dm (M), dLs (M,M; lower triangle, zeros above). */
extern "C" int npgp_dsvi_layer_bwd(int n, int M, int d, const double* X, const double* Z, const double* ls, const double* os,
                                   const double* m, const double* var, double min_var, const double* dmean, const double* dvar,
                                   double* dX, double* dZ, double* dls, double* dos, double* dm, double* dLs, void* work,
                                   long work_bytes, cudaStream_t st) {
  if (!X || !Z || !ls || !os || !m || !var || !dmean || !dvar || !dZ || !dls || !dos || !dm || !dLs || !work) return NPGP_EINVAL;
  if (reinterpret_cast<uintptr_t>(work) & 255) return NPGP_EUNSUPPORTED;
  DsviWs w;
  NPGP_TRY(dsvi_layout(n, M, d, work, &w));
  if (work_bytes < w.total) return NPGP_EWORKSPACE;
  // ---- seeds
  NPGP_CUDA(cudaMemsetAsync(w.cnt_sum, 0, 2 * sizeof(double), st));
  dsvi_seed_kernel<<<ceil_div(n, 256), 256, 0, st>>>(n, dvar, var, min_var, w.gv, w.gv2, w.cnt_sum);
  NPGP_LAUNCH_CHECK();
  // ---- du = K^T dmean,  dC = K^T diag(gv) K
  NPGP_CUDA(cudaMemsetAsync(w.du, 0, sizeof(double) * M, st));
  NPGP_TRY(npgp_colwsum(n, M, w.K, M, dmean, w.du, st));
  if (M % 128 == 0 && n >= kI8MinRows) {
    NPGP_TRY(npgp_wsyrk_weighted_only(n, M, 1.0, w.K, M, w.gv, w.cnt_sum, (double)n, w.dC, M, st));  // unequal weights (else 0)
    NPGP_TRY(npgp_syrk_i8(n, M, 1.0, w.K, M, w.gv, w.cnt_sum, (double)n, 1, 0, w.dC, M, w.i8, w.i8_bytes, st));  // equal: + w0 K^T K
  } else {
    NPGP_TRY(npgp_wsyrk(n, M, 1.0, w.K, M, w.gv, w.dC, M, st));
  }
  // ---- O(M^3) chain to dm, dLs, dKzz (Cholesky + inverse backward folded, as in svgp_step.cu)
  NPGP_TRY(npgp_gemv_n(M, M, w.P, M, w.du, dm, st));
  NPGP_TRY(npgp_dgemm(0, 1, M, M, M, 1.0, w.dC, M, w.P, M, 0.0, w.W2, M, 0, 2, 0, st));
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 1.0, w.P, M, w.W2, M, 0.0, w.dE, M, 1, 0, 0, st));
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 2.0, w.dE, M, w.Ls_t, M, 0.0, w.dLs, M, 0, 1, 0, st));
  dsvi_tril_out_kernel<<<g2(M), kB2, 0, st>>>(M, w.dLs, dLs);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 2.0, w.EP, M, w.W2, M, 0.0, w.X2, M, 0, 0, 0, st));
  svgp_addr_phi_kernel<<<g2(M), kB2, 0, st>>>(M, w.X2, m, dm);
  NPGP_LAUNCH_CHECK();
  NPGP_TRY(npgp_dgemm(1, 0, M, M, M, 1.0, w.P, M, w.X2, M, 0.0, w.Y, M, 2, 1, 0, st));
  NPGP_TRY(npgp_dgemm(0, 0, M, M, M, 1.0, w.Y, M, w.P, M, 0.0, w.dK, M, 0, 1, 0, st));
  svgp_sym_avg_kernel<<<dim3(ceil_div(M, 32), ceil_div(M, 32)), kB2, 0, st>>>(M, w.dK, w.dKzz);
  NPGP_LAUNCH_CHECK();
  // ---- kernel backward: through Kzz and through K(X,Z) (G = dmean u^T + 2 diag(gv) T formed inside the kernel)
  NPGP_CUDA(cudaMemsetAsync(dZ, 0, sizeof(double) * M * d, st));
  NPGP_CUDA(cudaMemsetAsync(w.dez, 0, sizeof(double) * d * M, st));
  NPGP_CUDA(cudaMemsetAsync(w.dex, 0, sizeof(double) * d * (long)n, st));
  NPGP_CUDA(cudaMemsetAsync(w.ds_acc, 0, 2 * sizeof(double), st));
  if (dX) NPGP_CUDA(cudaMemsetAsync(dX, 0, sizeof(double) * (long)n * d, st));
  NPGP_TRY(npgp_gibbs_diag_bwd(d, M, M, Z, w.lam, Z, w.lam, os, w.dKzz, M, nullptr, nullptr, nullptr, w.dez, dZ, w.dez, dZ,
                               w.ds_acc, st));
  NPGP_TRY(npgp_gibbs_diag_bwd(d, n, M, X, w.lamx, Z, w.lam, os, w.T, M, w.gv2, dmean, w.u, w.dex, dX, w.dez, dZ, w.ds_acc, st));
  const int nblk = 128;
  dsvi_rowsum_part_kernel<<<dim3(nblk, d), 256, 0, st>>>(d, (long)n, w.dex, w.partX);
  NPGP_LAUNCH_CHECK();
  dsvi_finish_kernel<<<1, 256, 0, st>>>(d, M, nblk, w.partX, w.dez, w.ds_acc, w.cnt_sum, dls, dos);
  NPGP_LAUNCH_CHECK();
  return NPGP_OK;
}
