/* npgp -- C ABI of the B200-native non-stationary (Gibbs) GP hot path.
 *
 * Every entry point takes raw DEVICE pointers (fp64, row-major), explicit sizes / leading dimensions and the CUDA
 * stream to run on; nothing allocates device memory, nothing synchronises.  The only process-global state are the debugging
 * switch npgp_rowquad_i8_debug, the diagnostic launch counter and the lazily resolved driver / NCCL entry points; none of
 * them affects results.  Return value:
 * 0 = ok, < 0 = argument error (NPGP_E*), > 0 = a cudaError_t from the launch.  All calls are asynchronous.
 * Outputs documented as "accumulated" are added to with atomics and must be zeroed by the caller.
 *
 * The reference (Stansfash/nonstationary-precip) has no native code and no FFI: the interfaces replaced here are the
 * Python methods cited per function (file:line into the reference), which the host-side mirror in
 * nonstationary_precip_b200/ re-implements on top of this library.  INTEGRATION.md shows the ctypes binding.
 */
#ifndef NPGP_H_
#define NPGP_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* npgp_stream_t; /* == cudaStream_t */

#define NPGP_OK 0
#define NPGP_EINVAL (-1)
#define NPGP_EUNSUPPORTED (-2)
#define NPGP_EWORKSPACE (-3)

int npgp_version(void);
/* diagnostic: kernels launched through this library so far in this process (bench.py's "gpu_launches") */
long npgp_launch_count(void);
/* measurement aid: buf[slot] = GPU nanosecond timer when the stream reaches this point (capturable in a CUDA graph, unlike
 * a timing event): the real timeline of a replayed multi-stream step */
int npgp_timestamp(long long* buf, int slot, npgp_stream_t stream);

/* ---- (a) fused Gibbs cross-covariance tiles ------------------------------------------------------------------------
 * Diagonal Gibbs kernel, replaces GibbsKernel.forward (models/gibbs_kernels.py:135-162).
 *   x1 (n1,D), x2 (n2,D) row-major; ell1 (D,n1), ell2 (D,n2) dim-major (layout of nonstationary_models.py:31-34);
 *   scale: optional device scalar (outputscale, GibbsSafeScaleKernel gibbs_kernels.py:164-168); K (n1,n2), ld = ldk.
 *   Optional fused mat-vec: Ku[i] += sum_j K_ij u_j (accumulated).  D = 1..6. */
int npgp_gibbs_diag_fwd(int D, int n1, int n2, const double* x1, const double* ell1, const double* x2,
                        const double* ell2, const double* scale, double* K, long ldk, const double* u, double* Ku,
                        npgp_stream_t stream);
/* Analytic backward (replaces the autograd graph of the same lines).  Upstream gradient
 *   G_ij = rowscale_i * G[i,j] + rowvec_i * colvec_j   (G or the rank-1 part may be NULL; rowscale NULL = 1).
 * Accumulated outputs: d_ell1 (D,n1), d_ell2 (D,n2), optional d_x1 (n1,D), d_x2 (n2,D), d_scale (scalar). */
int npgp_gibbs_diag_bwd(int D, int n1, int n2, const double* x1, const double* ell1, const double* x2,
                        const double* ell2, const double* scale, const double* G, long ldg, const double* rowscale,
                        const double* rowvec, const double* colvec, double* d_ell1, double* d_x1, double* d_ell2,
                        double* d_x2, double* d_scale, npgp_stream_t stream);

/* Full-matrix (Paciorek-Schervish) Gibbs kernel, d = 2 or 3; replaces MultivariateGibbsKernel.forward
 * (models/multivariate_gibbs_kernel.py:101-150) and SparseMultivariateGibbsKernel.forward
 * (models/sparse_multivariate_gibbs_kernel.py:105-154).  S1 (n1,P), S2 (n2,P): packed symmetric per-point matrices,
 * P = d(d+1)/2, d=2 [00,01,11], d=3 [00,01,02,11,12,22].  jitter: the reference's 1e-5 on the inverse only. */
int npgp_gibbs_full_fwd(int d, int n1, int n2, const double* x1, const double* S1, const double* x2, const double* S2,
                        double jitter, const double* scale, double* K, long ldk, const double* u, double* Ku,
                        npgp_stream_t stream);
/* d_S1 (n1,P), d_S2 (n2,P) accumulated: entries of the SYMMETRIC matrix dL/dSigma in the same packing. */
int npgp_gibbs_full_bwd(int d, int n1, int n2, const double* x1, const double* S1, const double* x2, const double* S2,
                        double jitter, const double* scale, const double* G, long ldg, const double* rowscale,
                        const double* rowvec, const double* colvec, double* d_S1, double* d_x1, double* d_S2,
                        double* d_x2, double* d_scale, npgp_stream_t stream);

/* Sigma(h) = softplus((h h^T)o(h h^T)) + DoD (models/multivariate_gibbs_kernel.py:98); H (n,d), Dm (d,d) -> S (n,P).
 * Backward: dH (n,d) and dDm (d,d) accumulated (dDm may be NULL). */
int npgp_sigma_from_h_fwd(int d, int n, const double* H, const double* Dm, double* S, npgp_stream_t stream);
int npgp_sigma_from_h_bwd(int d, int n, const double* H, const double* Dm, const double* dS, double* dH, double* dDm,
                          npgp_stream_t stream);

/* ---- (b) matrix-free / tensor-core contractions ---------------------------------------------------------------------
 * Lengthscale-field interpolation, matrix free:
 *   out[b,i,c] = f( bias_b + sum_j os_b exp(-0.5 |(x_i - z_j)/lam_b|^2) V[b,j,c] ),  f = exp if apply_exp else identity
 * x (n,d), z (m,d), lam (nb,d), os (nb) or NULL, V (nb,m,nv), bias (nb) or NULL, out (nb,n,nv).
 * Replaces LogNormalPriorProcess.conditional_sample's K_xg @ alpha (models/gibbs_kernels.py:85-100; nb = D, nv = 1) and
 * expectation_conditional_matrix_variate_dist (models/sparse_multivariate_gibbs_kernel.py:67-80; nb = 1, nv = d).
 * Backward (w.r.t. the pre-f value): dV (nb,m,nv) and dz (m,d, may be NULL) accumulated. */
int npgp_rbf_matvec_fwd(int d, int nb, int nv, int n, int m, const double* x, const double* z, const double* lam,
                        const double* os, const double* V, const double* bias, int apply_exp, double* out,
                        npgp_stream_t stream);
int npgp_rbf_matvec_bwd(int d, int nb, int nv, int n, int m, const double* x, const double* z, const double* lam,
                        const double* os, const double* V, const double* dOut, double* dV, double* dz,
                        npgp_stream_t stream);

/* FP64 tensor-core GEMM (DMMA), row-major: C = alpha op(A) op(B) + beta C.  tri_a / tri_b: structure of op(A) (MxK) /
 * op(B) (KxN): 0 dense, 1 lower, 2 upper (zero blocks are skipped); out_tri: 0 all, 1 lower tiles only, 2 upper only.
 * lda, ldb must be even and A, B 16-byte aligned. */
int npgp_dgemm(int transA, int transB, int M, int N, int K, double alpha, const double* A, long lda, const double* B,
               long ldb, double beta, double* C, long ldc, int tri_a, int tri_b, int out_tri, npgp_stream_t stream);
/* T = K C and q_i = sum_j T_ij K_ij (q accumulated, may be NULL): the A^T (S - I) A term of the whitened predictive
 * variance (GPyTorch VariationalStrategy.forward as driven by models/dgps.py:25-35) with C = L^-T (S - I) L^-1. */
int npgp_rowquad(int n, int M, const double* K, long ldk, const double* C, long ldc, double* T, long ldt, double* q,
                 npgp_stream_t stream);
/* Out = alpha K^T diag(w) K (symmetric, overwritten); w NULL = ones.  dL/dC of the SVGP ELBO and the SGPR
 * Phi = Kzx Kxz (models/gibbs_kernels.py:222-225). */
int npgp_wsyrk(int n, int M, double alpha, const double* K, long ldk, const double* w, double* Out, long ldo,
               npgp_stream_t stream);
/* Same with a device-side hint: if *uniform_count == uniform_target all weights equal w[0] and the unweighted inner
 * loop is taken (SVGP-Gibbs: w = g_v is constant unless a variance was clamped; npgp_gauss_ell counts unclamped rows). */
int npgp_wsyrk_hint(int n, int M, double alpha, const double* K, long ldk, const double* w, const double* uniform_count,
                    double uniform_target, double* Out, long ldo, npgp_stream_t stream);
int npgp_symmetrize(int M, double* C, long ldc, int from_upper, npgp_stream_t stream);
/* Triangular solve through the inverse factor P = L^-1 of npgp_potrf_inv_*: X = P B (trans 0) or P^T B (trans 1), one
 * triangular-aware product -- the reference's inv_root = triangular_solve(eye, chol); k_ux1.matmul(inv_root)
 * (models/gibbs_kernels.py:205-208,222-225).  B, X (M,k). */
int npgp_trsm(int trans, int M, int k, const double* P, long ldp, const double* B, long ldb, double* X, long ldx,
              npgp_stream_t stream);

/* ---- (c) blocked Cholesky + inverse factor --------------------------------------------------------------------------
 * A = L L^T in place (upper zeroed), P = L^-1; *info = 0 or 1-based index of the first non-positive pivot.
 * Replaces psd_safe_cholesky + triangular_solve(eye, chol) (models/gibbs_kernels.py:197-208). */
long npgp_potrf_workspace_bytes(int M);
int npgp_potrf_inv_lower(int M, double* A, long lda, double* P, long ldp, void* work, long work_bytes, int* info,
                         npgp_stream_t stream);
/* Same contract in ONE kernel launch (csrc/chol_flow.cu): every 64 x 64 tile of L and of L^-1 is a resident CTA that waits
 * on per-tile flags, so a dependent panel step costs an L2 round trip instead of a kernel boundary and the inverse is
 * assembled while the factorisation proceeds.  *info = -1 if a (bounded) dataflow wait timed out.  work: flags only. */
long npgp_potrf_flow_workspace_bytes(int M);
int npgp_potrf_inv_flow(int M, double* A, long lda, double* P, long ldp, void* work, long work_bytes, int* info,
                        npgp_stream_t stream);
/* n <= 4 independent matrices of the same order in ONE launch (tasks interleaved: all matrices advance together; two
 * separate launches on two streams cost 0.62 ms at M = 1024, the batch 0.45).  A, P, work, info: HOST arrays of n device
 * pointers (work[i]: npgp_potrf_flow_workspace_bytes(M) bytes of flags per matrix). */
int npgp_potrf_inv_flow_batch(int n, int M, double* const* A, long lda, double* const* P, long ldp, void* const* work,
                              long work_bytes, int* const* info, npgp_stream_t stream);

/* ---- SVGP-Gibbs ELBO step: small kernels (GPyTorch VariationalELBO + GaussianLikelihood.expected_log_prob semantics
 * as driven by experiments/deepgp_spatial_bench.py:61,84-87; SURVEY.md Appendix B.4) -------------------------------
 * out[j] += sum_i w_i K[i,j] (w NULL = ones; accumulated): K_zx y of SGPR, K_xz^T g_mu of the ELBO backward. */
int npgp_colwsum(int n, int M, const double* K, long ldk, const double* w, double* out, npgp_stream_t stream);
/* out[i] = sum_j A[i,j] v[j] (overwritten): predictive mean K_xz u, P du of the backward. */
int npgp_gemv_n(int n, int M, const double* A, long lda, const double* v, double* out, npgp_stream_t stream);
/* Gaussian expected log-likelihood over n rows.  v_i = max(*kdiag + jitter_xx + q_i, min_var);
 * acc3[0] += sum_i E_q log N(y_i | f_i, *noise); acc3[1] += sum_i ((y_i-mu_i)^2 + v_i); acc3[2] += #rows not clamped;
 * gmu_i = wscale (y_i-mu_i)/noise, gv_i = -0.5 wscale/noise (0 where clamped); var_out (may be NULL) = v. */
int npgp_gauss_ell(int n, const double* y, const double* mu, const double* q, const double* kdiag, double jitter_xx,
                   double min_var, const double* noise, double wscale, double* var_out, double* gmu, double* gv,
                   double* acc3, npgp_stream_t stream);
/* X <- alpha * Phi(X): lower triangle, diagonal halved, upper zeroed (Cholesky backward). */
int npgp_phi_mask(int M, double* X, long ldx, double alpha, npgp_stream_t stream);
/* Fused Adam over a flat parameter buffer (torch.optim.Adam semantics as used by experiments/spatial_exp.py:193);
 * g is scaled by gscale first; entries with mask[i] == 0 are frozen (mask may be NULL). */
int npgp_adam_step(long n, double* p, const double* g, double* m, double* v, const double* mask, double lr,
                   double beta1, double beta2, double eps, int step, double gscale, npgp_stream_t stream);

/* Same update with the step counter kept on the device (step_dev[0] = steps taken so far, incremented here), so that a
 * captured CUDA graph of the training step replays with the correct bias correction. */
int npgp_adam_step_dev(long n, double* p, const double* g, double* m, double* v, const double* mask, double lr,
                       double beta1, double beta2, double eps, double* step_dev, double gscale, npgp_stream_t stream);

/* Failure handling inside a captured step.  The reference raises from psd_safe_cholesky (models/gibbs_kernels.py:201) after
 * its jitter ladder; a replayed CUDA graph cannot raise, so: npgp_status_update ORs bit 0 into the sticky device flag
 * *status when *info != 0 (bad pivot / dataflow time-out) and bit 1 when *loss is not finite (either pointer may be NULL);
 * npgp_adam_step_guarded is npgp_adam_step_dev that leaves parameters, moments and step counter untouched while
 * *status != 0.  The host polls status every few steps and re-runs with the next jitter of the ladder. */
int npgp_status_update(int* status, const int* info, const double* loss, npgp_stream_t stream);
int npgp_adam_step_guarded(long n, double* p, const double* g, double* m, double* v, const double* mask, double lr,
                           double beta1, double beta2, double eps, double* step_dev, double gscale, const int* status,
                           npgp_stream_t stream);

/* ---- (d) doubly-stochastic deep GP (models/dgps.py:53-111 through GPyTorch DeepGPLayer.__call__ and
 * DeepApproximateMLL(VariationalELBO); SURVEY.md Appendix B.4/B.5) ----------------------------------------------------
 * Marginal reparameterised layer sample h = mu + sqrt(var) * eps over n elements.  eps_in NULL: eps ~ N(0,1) from
 * Philox4x32-10 keyed by (seed, index_offset + element index) -- independent of how samples / rows are sharded;
 * eps_out (may be NULL) receives the draws (needed by the backward). */
int npgp_dsvi_sample(long n, const double* mu, const double* var, const double* eps_in, unsigned long long seed,
                     unsigned long long index_offset, double* h, double* eps_out, npgp_stream_t stream);
int npgp_dsvi_sample_bwd(long n, const double* var, const double* eps, const double* dh, double* dmu, double* dvar,
                         npgp_stream_t stream);
/* Per-sample Gaussian expected log-likelihood: mu, var (S,n), y (n); sums[s] += sum_i E log N(y_i | f_si, *noise)
 * (warp-shuffle + block reduction); sq[s] += sum_i ((y-mu)^2 + var) (may be NULL); gmu, gvar (S,n) (may be NULL) =
 * wscale * d/dmu, d/dvar of the per-element term. */
int npgp_gauss_ell_batched(int S, int n, const double* y, const double* mu, const double* var, const double* noise,
                           double wscale, double* sums, double* sq, double* gmu, double* gvar, npgp_stream_t stream);

/* One output dimension of a deep-GP layer (csrc/dsvi_layer.cu): the whitened-SVGP marginals at the rows X for an RBF-ARD * Scale
 * kernel (reference models/dgps.py:15-46 through GPyTorch's VariationalStrategy / DeepGPLayer.__call__) and their analytic
 * backward.  X (n,d): S x B samples of the previous layer (or the B data rows); Z (M,d); ls (d), os (1): constrained
 * lengthscales / outputscale on the device; m (M), Ls (M,M, lower part used).  fwd: mean = K u (the caller adds the mean
 * function), var = max(os + add_var + rowdot(K C, K), min_var), *info = the Cholesky's code.  bwd: all outputs OVERWRITTEN
 * (dX (n,d) may be NULL; dLs lower triangle).  work: npgp_dsvi_layer_workspace_bytes(n, M, d) bytes, 256-byte aligned, passed
 * unchanged from fwd to bwd (it carries K, T = K C and the Z-side factors).  M even, d <= 6.  T = K C and, when all
 * variance seeds are equal (decided on the device), K^T diag(dvar) K run on the int8 tensor cores. */
long npgp_dsvi_layer_workspace_bytes(int n, int M, int d);
int npgp_dsvi_layer_fwd(int n, int M, int d, const double* X, const double* Z, const double* ls, const double* os,
                        const double* m, const double* Ls, double jitter, double add_var, double min_var, double* mean,
                        double* var, int* info, void* work, long work_bytes, npgp_stream_t stream);
int npgp_dsvi_layer_bwd(int n, int M, int d, const double* X, const double* Z, const double* ls, const double* os,
                        const double* m, const double* var, double min_var, const double* dmean, const double* dvar,
                        double* dX, double* dZ, double* dls, double* dos, double* dm, double* dLs, void* work, long work_bytes,
                        npgp_stream_t stream);

/* ---- temporal kernel of the spatio-temporal model (models/spatio_temporal_models.py:42):
 * K[i,j] = s exp(-0.5 tau^2/l_r^2) exp(-2 sin^2(pi |tau|/p)/l_p), tau = t1[i] - t2[j]; hyp (device) = [l_r, l_p, p, s].
 * Backward: out4 += dL/d[l_r, l_p, p, s]; dt2 (n2, may be NULL) += dL/dt2. */
int npgp_rbfper_fwd(int n1, int n2, const double* t1, const double* t2, const double* hyp, double* K, long ldk,
                    npgp_stream_t stream);
int npgp_rbfper_bwd(int n1, int n2, const double* t1, const double* t2, const double* hyp, const double* G, long ldg,
                    double* out4, double* dt2, npgp_stream_t stream);

/* ---- exact FP64 contractions on the integer tensor cores (csrc/oz8.cu, csrc/oz8.cuh) ----------------------------------
 * Replaces the reference's dense n x M x M products: k_ux1.matmul(inv_root) and the Woodbury terms
 * (models/gibbs_kernels.py:222-232), A^T (S - I) A of the whitened VariationalStrategy (models/dgps.py:25-35 through
 * GPyTorch) and Phi = Kzx Kxz of the SGPR objective.  Every operand entry is the integer rint(x 2^(54-e)) written as 7
 * signed base-256 digits, e a power-of-two exponent per row or per matrix; the 28 digit products with p + q <= 6 are
 * accumulated exactly in int32 by tcgen05.mma kind::i8 (S8 x S8) and recombined in the epilogue.
 * Results equal the FP64 product to its own rounding bound and are bit-exact on integer-valued data.  Exception: a row
 * (or column) whose largest magnitude is below 2^-961 has its exponent clamped at -960, so its entries carry an absolute
 * error of up to 2^-1015 rather than a relative one.
 *
 * General operands (contract of npgp_rowquad / npgp_wsyrk): C symmetric, M % 64 == 0 (SYRK: M % 128 == 0), M <= 16384,
 * T 16-byte aligned with even ldt.  work: the *_workspace_bytes(n, M) bytes of device memory (digit planes, exponents,
 * SYRK chunk partials).  The SYRK adds its row chunks in a fixed order: bitwise reproducible. */
long npgp_rowquad_i8_workspace_bytes(int n, int M);
void npgp_rowquad_i8_debug(long long* dev_counters); /* debugging aid: 8 cycle counters written by CTA 0 (NULL = off) */
int npgp_rowquad_i8(int n, int M, const double* K, long ldk, const double* C, long ldc, double* T, long ldt, double* q,
                    void* work, long work_bytes, npgp_stream_t stream);
/* alpha * w0 * K^T K (symmetric M x M): the equal-weights case of npgp_wsyrk (w0 = *w0_dev, NULL: 1).  uniform_count /
 * uniform_target (optional): device-side gate as in npgp_wsyrk_hint, the kernels only run when *uniform_count ==
 * uniform_target; accumulate != 0 adds to Out.  npgp_wsyrk_weighted_only is the complementary half: Out = alpha K^T diag(w) K
 * when the weights are NOT all equal, else untouched. */
long npgp_syrk_i8_workspace_bytes(int n, int M);
int npgp_syrk_i8(int n, int M, double alpha, const double* K, long ldk, const double* w0_dev, const double* uniform_count,
                 double uniform_target, int accumulate, double* Out, long ldo, void* work, long work_bytes,
                 npgp_stream_t stream);
int npgp_wsyrk_weighted_only(int n, int M, double alpha, const double* K, long ldk, const double* w,
                             const double* uniform_count, double uniform_target, double* Out, long ldo,
                             npgp_stream_t stream);

/* Digit-plane level (the SVGP step's path: K(X,Z) is never materialised in FP64).
 * npgp_o8_digits_bytes: size of the planes of a rows x Kd matrix (block_rows 128: A operand, 64: symmetric B operand).
 * npgp_o8_slice_rows:   planes + per-row exponents (ceil(R / block_rows) * block_rows ints) of an arbitrary FP64 matrix. */
long npgp_o8_digits_bytes(int rows, int Kd, int block_rows);
int npgp_o8_slice_rows(int R, int Kd, const double* X, long ldx, int block_rows, void* digits, int* expo,
                       npgp_stream_t stream);
/* Gibbs kernels emitted as digit planes: the same arithmetic as npgp_gibbs_diag_fwd / npgp_gibbs_full_fwd (same reference
 * lines), 7 bytes per pair instead of 8, scale (device scalar, required) bounds the entries and fixes the matrix-wide
 * exponent.  n2 % 32 == 0.  Optional fused K u: Ku_part (npgp_gibbs_digits_splits(n1, n2) x ku_stride) receives per-column-
 * split partial sums (plain stores; add them in index order, e.g. npgp_mu_gmu_parts). */
int npgp_gibbs_digits_splits(int n1, int n2);
int npgp_gibbs_diag_fwd_digits(int D, int n1, int n2, const double* x1, const double* ell1, const double* x2,
                               const double* ell2, const double* scale, void* digits, const double* u, double* Ku_part,
                               long ku_stride, npgp_stream_t stream);
int npgp_gibbs_full_fwd_digits(int d, int n1, int n2, const double* x1, const double* S1, const double* x2, const double* S2,
                               double jitter, const double* scale, void* digits, const double* u, double* Ku_part,
                               long ku_stride, npgp_stream_t stream);
/* T = K C from planes.  a_expo NULL: matrix-wide exponent from *a_scale.  Kmat (optional): FP64 K for the row dot, else K is
 * rebuilt from the planes.  T may be NULL when q is given: only the row dot is formed (bitwise the q of the same call with T),
 * T is not stored; T and q both NULL is NPGP_EINVAL.  q (optional): q_stride == 0 -> q[i] += rowdot (atomics);
 * q_stride >= n -> q[cb * q_stride + i] = partial of column block cb (M / 64 blocks; deterministic).  gvec / du_part
 * (optional): du_part[rb * M + j] = sum over the rows of row block rb (128 rows) of gvec_i K_ij -- K^T g_mu of the ELBO
 * backward from the K tiles the kernel holds anyway. */
int npgp_o8_rowquad_digits(int n, int M, const void* a_digits, const int* a_expo, const double* a_scale,
                           const void* c_digits, const int* c_expo, const double* Kmat, long ldk, double* T, long ldt,
                           double* q, long q_stride, const double* gvec, double* du_part, npgp_stream_t stream);
/* T (n x N) = A B^T from planes, T stored only (no row dot, no column sums): A (n x Kd, block_rows 128; a_expo NULL ->
 * matrix-wide exponent from *a_scale), B (N x Kd, block_rows 64) with per-row exponents b_expo.  N % 64 == 0, Kd % 32 == 0,
 * Kd <= 16384, T 16-byte aligned with even ldt >= N.  Same arithmetic and rounding bound as npgp_o8_rowquad_digits. */
int npgp_o8_gemm_digits(int n, int N, int Kd, const void* a_digits, const int* a_expo, const double* a_scale,
                        const void* b_digits, const int* b_expo, double* T, long ldt, npgp_stream_t stream);
/* Row norms of a triangular contraction from planes: q[cb * q_stride + i] = sum_{j in column block cb} (A B^T)_ij^2, T never
 * stored.  A (n x Kd, block_rows 128; a_expo NULL -> matrix-wide exponent from *a_scale), B (N x Kd, block_rows 64, per-row
 * exponents b_expo as npgp_o8_slice_rows writes them) lower triangular: column block cb (64 rows of B) contracts over
 * k < 64 (cb + 1) only.  Ms > 0 splits B block-diagonally at column Ms: blocks with 64 cb >= Ms also start at k = Ms (the zero
 * quadrant of blockdiag(P_t, P_s) costs nothing).  The skipped k-steps of B are never read.  Deterministic per-block
 * partials (plain stores), N / 64 of them per row.  N % 64 == 0, Kd % 32 == 0, 0 < Kd <= 16384, Ms % 64 == 0, Ms == 0 or
 * Ms < Kd, q_stride >= n; anything else (and NULL operands) is NPGP_EINVAL. */
int npgp_o8_trinorm_digits(int n, int N, int Kd, int Ms, const void* a_digits, const int* a_expo, const double* a_scale,
                           const void* b_digits, const int* b_expo, double* q, long q_stride, npgp_stream_t stream);
int npgp_o8_sum_partials(int nb, int N, const double* part, double* out, npgp_stream_t stream); /* out[j] = sum_b part[b*N+j] */
/* Out (+)= alpha * w0 * (K^T K - sum_{i in skip} k_i k_i^T) from the ROW-layout planes of K (n x M, matrix-wide scale
 * *x_scale), read MN-major: no transposed copy.  skip_count / skip_rows (optional): rows of weight 0 (clamped variances).
 * part: npgp_o8_syrk_part_bytes(n, M) bytes.  M % 128 == 0. */
long npgp_o8_syrk_part_bytes(int n, int M);
int npgp_o8_syrk_digits(int n, int M, const void* x_digits, const double* x_scale, double alpha, const double* w0_dev,
                        const int* skip_count, const int* skip_rows, int accumulate, double* Out, long ldo, void* part,
                        long part_bytes, npgp_stream_t stream);

/* Deterministic (two-stage, fixed order) variants of the ELBO reductions used with the digit-plane path. */
int npgp_mu_gmu_parts(int n, const double* y, const double* mu_part, int nparts, long stride, const double* noise,
                      double wscale, double* mu, double* gmu, npgp_stream_t stream);
long npgp_gauss_ell_parts_workspace_bytes(int n);
int npgp_gauss_ell_parts(int n, const double* y, const double* mu, const double* q_part, int nq, long q_stride,
                         const double* kdiag, double jitter_xx, double min_var, const double* noise, double wscale,
                         double* var_out, double* gmu, double* gv, double* acc4, int* skip_count, int* skip_rows, void* work,
                         long work_bytes, npgp_stream_t stream);

/* ---- the whole SVGP-Gibbs ELBO step behind one call (csrc/svgp_step.cu) -----------------------------------------------
 * Composition of the reference's parts as in SURVEY.md Appendix B: the inducing-point field handling of InducingGibbsKernel
 * (models/gibbs_kernels.py:210-223) / SparseMultivariateGibbsKernel (models/sparse_multivariate_gibbs_kernel.py:67-154),
 * GPyTorch's whitened VariationalStrategy + VariationalELBO as driven by models/dgps.py:25-35 and
 * experiments/deepgp_spatial_bench.py:61,84-87, Adam as in experiments/spatial_exp.py:193.
 * A plan holds the shapes, the carve-up of ONE caller-supplied workspace (npgp_svgp_workspace_bytes; 256-byte aligned), two
 * side streams and a few events; calls on the same plan must not overlap.  Every call enqueues on `stream` (plus the plan's
 * side streams, joined again before it returns: capturable into a CUDA graph) and returns without synchronising.
 * theta / grad layout (doubles), n_pad = npgp_svgp_theta_size (even):
 *   variant 1 (full-matrix Gibbs): [Z (M,d) | H (M,d) | D (d,d) | m (M) | Ls (M,M) | raw_outputscale | raw_noise]
 *   variant 0 (diagonal Gibbs)   : [Z (M,d) | log_ell_z (d,M)   | m (M) | Ls (M,M) | raw_outputscale | raw_noise]
 * grad has n_pad + 2 entries: grad[n_pad] = this rank's share of -ELBO, so ONE all-reduce of grad carries gradient and loss.
 * M % 128 == 0; variant 1: d = 2 or 3; variant 0: d <= 6. */
typedef struct {
  int variant;           /* 0 = diagonal Gibbs kernel with a log-normal lengthscale field, 1 = full-matrix kernel, field (H, D) */
  int d, M, B_local;     /* input dimension, inducing points, rows of this rank's share of the minibatch */
  long N_total;          /* size of the data set (scaling of the KL / prior terms) */
  int B_global;          /* rows of the global minibatch */
  int world_size;        /* ranks: the replicated KL / prior terms are weighted 1 / world_size on every rank */
  double jitter_zz, jitter_xx, kernel_jitter, min_var; /* GPyTorch's 1e-6 / 1e-4, the reference's 1e-5, variance floor 1e-6 */
  double extra_jitter;   /* psd_safe_cholesky ladder on top of jitter_zz (npgp_svgp_set_extra_jitter) */
  int learn_z, include_prior;
  const double* row_os;  /* variant 1: device scalar, outputscale of the row kernel of the matrix-normal field prior */
  const double* row_lam; /* variant 1: (d) its lengthscales */
  const double* prior_c; /* variant 0: (d) prior means of log ell, */
  const double* prior_os;  /*          (d) prior outputscales, */
  const double* prior_lam; /*          (d,d) prior lengthscales, one row per output dimension */
  long long* timeline;   /* optional: 2 * npgp_svgp_num_sections() GPU-timer stamps (start, end per section); NULL = off */
} npgp_svgp_config;
typedef struct npgp_svgp_plan npgp_svgp_plan;
long npgp_svgp_theta_size(const npgp_svgp_config* cfg);
long npgp_svgp_workspace_bytes(const npgp_svgp_config* cfg);
int npgp_svgp_plan_create(npgp_svgp_plan** plan, const npgp_svgp_config* cfg, void* workspace, long workspace_bytes);
int npgp_svgp_plan_destroy(npgp_svgp_plan* plan);
int npgp_svgp_set_extra_jitter(npgp_svgp_plan* plan, double extra);
int npgp_svgp_num_sections(void);
const char* npgp_svgp_section_name(int i);
/* x (B_local,d), y (B_local).  fwd: everything up to the loss (grad[n_pad] = this rank's share of -ELBO); K(X_B,Z) (digit
 * planes), T = K C, the gradient seeds and the Z-side factors stay in the workspace.  status (optional, device, sticky): bit 0
 * is set when a Cholesky fails.  bwd: grad[0 .. n_pad) of the forward that ran last on this plan (same x, theta). */
int npgp_svgp_elbo_fwd(npgp_svgp_plan* plan, const double* x, const double* y, const double* theta, double* grad, int* status,
                       npgp_stream_t stream);
int npgp_svgp_elbo_bwd(npgp_svgp_plan* plan, const double* x, const double* theta, double* grad, npgp_stream_t stream);
/* fwd + bwd + all-reduce of grad (comm: npgp_comm_create handle, NULL = single rank) + npgp_status_update on the reduced loss
 * + npgp_adam_step_guarded on theta */
int npgp_svgp_step(npgp_svgp_plan* plan, const double* x, const double* y, double* theta, double* grad, double* adam_m,
                   double* adam_v, const double* mask, double* step_dev, int* status, double lr, double beta1, double beta2,
                   double eps, void* comm, npgp_stream_t stream);
/* Posterior prediction with a fitted theta (SVGPGibbs.predict semantics, the reference's model.predict through GPyTorch's
 * whitened VariationalStrategy).  Both calls reuse the plan's workspace (no allocation) and are capturable.
 * prepare: Z-side factors of the posterior for this theta: Kzz -> Cholesky + inverse, u = P^T m, C = P^T (Ls Ls^T - I) P and
 * its digit planes, the field's prior-kernel factorisations and interpolation weights (alpha / W).  status (optional,
 * sticky): bit 0 on a failed factorisation, as in npgp_svgp_elbo_fwd.  Invalidates the saved forward (npgp_svgp_elbo_bwd then
 * returns NPGP_EINVAL until the next npgp_svgp_elbo_fwd). */
int npgp_svgp_predict_prepare(npgp_svgp_plan* plan, const double* theta, int* status, npgp_stream_t stream);
/* Posterior marginals at n rows xs (n,d), in chunks of B_local rows, with the theta of the last prepare on this plan (theta:
 * the same buffer, read for Z and D):
 *   mean (n), var_f (n) = max(s + jitter_xx + k^T C k, min_var)                 required
 *   var_y (n) = var_f + noise, noise = 1e-4 + softplus(raw_noise)               optional (NULL)
 *   field: variant 0 (d,n) dim-major ell(x) = exp(c + K^p alpha); variant 1 (n, d(d+1)/2) Sigma(x) packed as
 *          npgp_sigma_from_h_fwd                                                optional
 *   lpd (n) = log N(y_i | mean_i, var_y_i)                                      optional, needs ys
 *   sums (3), ACCUMULATED: += [sum (y-mean)^2, sum -lpd, n]                     optional, needs ys
 * Every reduction of this call has a fixed order: bitwise reproducible for a fixed plan, n and prepared factors (prepare, like
 * the step's forward, splits its M x M products over K with FP64 atomics from M = 512 on).  Rows may be sharded across ranks
 * with no collective; one npgp_allreduce_f64 of the 3 sums gives the global RMSE / NLPD.  NPGP_EINVAL without a prepare since the
 * last fwd / step / set_extra_jitter on this plan.  Invalidates the saved forward like prepare. */
int npgp_svgp_predict(npgp_svgp_plan* plan, long n, const double* xs, const double* ys, const double* theta, double* mean,
                      double* var_f, double* var_y, double* field, double* lpd, double* sums, npgp_stream_t stream);
/* Posterior sample fields at any number of rows, correlated across rows, with the factors of the last predict_prepare
 * (L = chol(Kzz + (jitter_zz + extra) I), P = L^-1, outputscale s).  The draws are the modified predictive process under q(u)
 * (Finley, Sang, Banerjee & Gelfand, CSDA 2009):
 *   f_s(x) = mean(x) + k(x)^T W_s + sqrt(r(x)) xi_s(x),   W = P^T Ls E (M x S),   r(x) = max(s + jitter_xx - k^T P^T P k, 0)
 * with E and xi independent standard normals; noise != 0 draws y instead, with sqrt(r(x) + noise) in place of sqrt(r(x)).
 * mean(x) is bitwise the mean npgp_svgp_predict returns for the same plan and chunking.  The covariance of the draws is
 * k^T P^T S P k' + delta_xx' r(x) (S = Ls Ls^T): each marginal equals var_f = s + jitter_xx + k^T C k wherever neither clamp
 * is active.  The only departure from the exact SVGP posterior k(x,x') + k^T C k' is that the off-diagonal residual
 * k(x,x') - k^T P^T P k' is set to zero.
 * Normals: E[j, s] = normal_from_index(seed, (s << 32) + j), xi_s(row) = normal_from_index(seed, 2^63 + (s << 48) + row_offset
 * + i) (Philox as npgp_dsvi_sample with mu = 0, var = 1): every rank draws the same E, so rows sharded over ranks with their
 * global row_offset are parts of one joint draw, and draw s does not depend on S.
 * workspace_bytes: size of `work` (256-byte aligned) for S draws, -1 on a bad cfg or S outside 1 .. 1024; it grows with
 *   64 ceil(S / 64): G = P^T P and its digit planes, W^T padded to that many rows and its planes, a B_local-row chunk of K W.
 * prepare: G, W and their planes into work.  NPGP_EINVAL unless npgp_svgp_predict_prepare has run since the last fwd / step /
 *   set_extra_jitter (theta: that prepare's buffer).
 * sample: out (S, n), leading dimension ldo >= n, rows xs (n, d) streamed in chunks of B_local through the plan (it overwrites
 *   what npgp_svgp_predict overwrites; P, C and their planes stay, so npgp_svgp_predict still works).  NPGP_EINVAL unless
 *   prepare ran on this work since the last fwd / step / set_extra_jitter / predict_prepare.
 * Both calls run on `stream` only, allocate nothing and are capturable; both invalidate the saved forward like predict.  For a
 * fixed plan and prepared factors the draws are bitwise reproducible (the prepares split their M x M products over K with FP64
 * atomics from M = 512 on). */
long npgp_svgp_sample_workspace_bytes(const npgp_svgp_config* cfg, int S);
/* E^T of S draws of width W, the one generator of both samplers' row-independent normals: Et (Sp x W, contiguous)
 * Et[s * W + j] = E[j, s] = normal_from_index(seed, (s << 32) + j) for s < S, 0 for S <= s < Sp.  Sp >= S. */
int npgp_sample_normals(int W, int S, int Sp, unsigned long long seed, double* Et, npgp_stream_t stream);
int npgp_svgp_sample_prepare(npgp_svgp_plan* plan, const double* theta, int S, unsigned long long seed, void* work,
                             long work_bytes, npgp_stream_t stream);
int npgp_svgp_sample(npgp_svgp_plan* plan, long n, const double* xs, long row_offset, const double* theta, int noise,
                     double* out, long ldo, void* work, long work_bytes, npgp_stream_t stream);
/* Posterior of weighted regional sums t_r = sum_{i in r} w_i f_i (basin totals, area means, block averages), exact under q(u),
 * with the factors of the last predict_prepare.  With k_i = K(x_i, Z) (scaled by s as the plan scales it), kappa the unscaled
 * Gibbs kernel (kappa(x, x) = 1) and C = P^T (Ls Ls^T - I) P:
 *   Cov(f_i, f_j) = s kappa(x_i, x_j) + delta_ij jitter_xx + k_i^T C k_j        (var_f on the diagonal, before its clamp)
 *   mean_R[r]    = Y[:, r]^T u,   Y (M x R), Y[:, r] = sum_{i in r} w_i k_i
 *   cov_R[r, r'] = s G[r, r'] + delta_rr' (jitter_xx [+ noise]) sum_{i in r} w_i^2 + (Y^T C Y)[r, r']
 *   G[r, r']     = sum_{i in r} sum_{j in r'} w_i w_j kappa(x_i, x_j)
 * Rows xs (n, d) are sorted by region: region r is rows [seg[r], seg[r+1]) (seg: R + 1 device offsets, non-decreasing from 0 to
 * n); w (n) optional (NULL = ones).  Every row belongs to exactly one region: nested basins may repeat rows in xs, but then
 * jitter_xx is counted only for identical indices, not for repeated points.
 * Pair sums (the new hot path, csrc/gibbs_segsum.cu): G is never formed as an n x n matrix.  Only pairs i < j are evaluated (a
 * same-row pair contributes exactly w_i^2), so the variances cost sum_r n_r^2 / 2 pairs and the full R x R matrix n^2 / 2.
 *   npgp_gibbs_diag_segsum: x (n, D), ell (D, n) dim-major, D = 1..6;  npgp_gibbs_full_segsum: x (n, d), S (n, P) packed, d = 2, 3,
 *   jitter as npgp_gibbs_full_fwd.  kappa is bitwise the entry npgp_gibbs_*_fwd(x, x) computes with scale NULL.
 *   Gdiag[r] = scale * G[r, r] always (scale: device scalar, NULL = 1); G (R x R, leading dimension ldg >= R) only with full,
 *   which evaluates r <= r' and mirrors.  Items (pairs of 256-row tiles) each write one partial to work, a finishing kernel adds
 *   every entry's partials in a fixed order: bitwise reproducible for fixed (n, seg, part, nparts), and with full = 0 Gdiag is
 *   bitwise that of full = 1 (nparts = 1).  part / nparts (0 <= part < nparts) split the item list: each part OVERWRITES the
 *   outputs with its share, and the sum over parts (one all-reduce of R + R^2 doubles) is the single-part result up to the order
 *   of that sum.  seg is validated on the device: a seg that is not non-decreasing from 0 to n gives NaN outputs, return 0.
 *   workspace_bytes: size of `work` (256-byte aligned) for any valid seg of n rows and R regions, -1 for n < 0, n >= 2^31 or
 *   R < 1.  Errors before any launch: NPGP_EINVAL for R < 1, n < 0, n >= 2^31, D / d out of range, NULL operands, part outside
 *   [0, nparts), full with ldg < R; NPGP_EUNSUPPORTED for a misaligned work; NPGP_EWORKSPACE for a small one.
 * Segmented column sums (the Y of one chunk, csrc/gibbs_segsum.cu): K (n x M, ldk >= M) holds the rows row0 .. row0 + n - 1 of
 *   the sorted set:  out[r * ldo + j] += sum_{i in r, row0 <= i < row0 + n} w_i K[i - row0, j]  (w: the chunk's n weights, NULL =
 *   ones).  Each (region, column) has one owner per launch, which adds its rows in index order (in 256-row slices, the slices
 *   in order): deterministic, and chunks add in stream order.  work: npgp_segment_colwsum_workspace_bytes(n, M) bytes, 8-byte
 *   aligned.  seg is not validated here (a bad one gives wrong sums, never an access outside K, w, seg or out's R rows).
 * Plan call (csrc/svgp_step.cu): rows streamed through the plan in chunks of B_local: the row field (kept in work: the pair sums
 *   need every row), K(x, Z) in FP64 into the plan's T buffer (neither predict nor sample uses it) and the chunk's Y columns;
 *   then mean_R = Y^T u, C Y and Y^T C Y with npgp_dgemm (only the diagonal, by a row-dot kernel, without cov_R), the pair sums
 *   with scale = s, and (jitter_xx [+ noise]) sum w_i^2 with noise = 1e-4 + softplus(raw_noise).  var_R (R) required; cov_R
 *   (R x R, leading dimension ldc >= R) optional: NULL costs the variances' pairs only.  With both, var_R is bitwise
 *   diag(cov_R), and cov_R is symmetric bitwise.  The marginals' clamp max(var, min_var) has no joint counterpart: a one-row
 *   region with w = 1 reproduces var_f wherever that clamp is inactive.  part / nparts go to the pair sums; the mean, low-rank
 *   and jitter / noise terms come from part 0 only (other parts write mean 0), so one all-reduce of the outputs gives the
 *   single-call answer.  State rules as npgp_svgp_sample: NPGP_EINVAL unless npgp_svgp_predict_prepare ran since the last
 *   fwd / step / set_extra_jitter; invalidates the saved forward; leaves P, C, u and their planes intact, so predict and
 *   sample give bitwise the same results after it.  One stream, no allocation, capturable.  Bitwise reproducible for a fixed
 *   plan, n, seg, part and nparts, except that from M = 512 on with few regions npgp_dgemm splits the low-rank products over
 *   K with FP64 atomics (as the prepares do).
 *   region_workspace_bytes: size of `work` (256-byte aligned), -1 on a bad cfg, n < 0, n >= 2^31 or R < 1; full: with cov_R. */
long npgp_segsum_workspace_bytes(long n, int R, int full);
int npgp_gibbs_diag_segsum(int D, long n, const double* x, const double* ell, const double* w, int R, const long* seg, int full,
                           int part, int nparts, const double* scale, double* Gdiag, double* G, long ldg, void* work,
                           long work_bytes, npgp_stream_t stream);
int npgp_gibbs_full_segsum(int d, long n, const double* x, const double* S, double jitter, const double* w, int R,
                           const long* seg, int full, int part, int nparts, const double* scale, double* Gdiag, double* G,
                           long ldg, void* work, long work_bytes, npgp_stream_t stream);
long npgp_segment_colwsum_workspace_bytes(int n, int M);
int npgp_segment_colwsum(int n, int M, const double* K, long ldk, const double* w, long row0, int R, const long* seg,
                         double* out, long ldo, void* work, long work_bytes, npgp_stream_t stream);
long npgp_svgp_region_workspace_bytes(const npgp_svgp_config* cfg, long n, int R, int full);
int npgp_svgp_region_moments(npgp_svgp_plan* plan, long n, const double* xs, const double* w, int R, const long* seg,
                             const double* theta, int noise, int part, int nparts, double* mean_R, double* var_R,
                             double* cov_R, long ldc, void* work, long work_bytes, npgp_stream_t stream);
/* device pointers into the workspace (inspection): 0 mu (B), 1 T (B,M), 2 P (M,M), 3 C (M,M), 4 u (M), 5 g_mu (B), 6 g_v (B),
 * 7 acc4, 8 info (ints: Kzz, then the prior-kernel factorisations) */
const void* npgp_svgp_buffer(npgp_svgp_plan* plan, int which);

/* ---- streamed SGPR posterior (sgpr.py posterior().predictive()): row-side kernels (csrc/sgpr_predict.cu) ---- */
/* Finishing kernel of one chunk of n rows, one launch.  qn: per-column-block partials of |P k(x)|^2 (row c * qn_stride + i),
 * the first nb_t blocks of the temporal component (0 for the diagonal model), the next nb_s of the Gibbs one; qv: the nb_v
 * partials of |V k(x)|^2.  Each component's partials are added in index order.  Device scalars s, noise, os_t (os_t only
 * with nb_t > 0):
 *   var_f (n) = [nb_t > 0] max(os_t - q_t, 0) + s max(1 - q_s, 0) + q_v      required
 *   var_y (n) = var_f + noise                                                 optional
 *   lpd (n) = log N(y | mean, var_y)                                          optional, needs y and mean
 *   sums (3), ACCUMULATED: += [sum (y - mean)^2, sum -lpd, n]                 optional, needs y and mean (fixed order)
 * work: npgp_sgpr_predict_workspace_bytes(n) bytes, zeroed before its first use (the kernel leaves it so); needed with sums.
 * Same sums contract as npgp_svgp_predict: one all-reduce of 3 doubles gives the global RMSE / NLPD. */
long npgp_sgpr_predict_workspace_bytes(int n);
int npgp_sgpr_predict_finish(int n, const double* qn, long qn_stride, int nb_t, int nb_s, const double* qv, long qv_stride,
                             int nb_v, const double* mean, const double* y, const double* s, const double* noise,
                             const double* os_t, double* var_f, double* var_y, double* lpd, double* sums, void* work,
                             long work_bytes, npgp_stream_t stream);
/* Finishing kernel of the exact Gibbs GP's predictive (models/nonstationary_models.py DiagonalExactGP.posterior()) for one
 * chunk of n rows, one launch.  qn: the nb per-column-block partials of |P_y k(x)|^2 (row c * qn_stride + i), added in index
 * order; P_y = chol(K + tau I)^-1 of the unscaled training kernel.  Device scalars s, noise; host scalar add_var:
 *   var_f (n) = s max(1 - q, 0) + add_var                                     required
 *   var_y, lpd, sums                                                          as npgp_sgpr_predict_finish
 * work: npgp_sgpr_predict_workspace_bytes(n) bytes, zeroed before its first use (the kernel leaves it so); needed with sums.
 * n, nb >= 0; anything else (and NULL required operands) is NPGP_EINVAL. */
int npgp_exact_predict_finish(int n, const double* qn, long qn_stride, int nb, const double* mean, const double* y,
                              const double* s, const double* noise, double add_var, double* var_f, double* var_y, double* lpd,
                              double* sums, void* work, long work_bytes, npgp_stream_t stream);
/* FP64 per-column-block row norms q[cb * q_stride + i] = sum_{j in [64 cb, min(64 cb + 64, W))} G_ij^2 (one warp per row,
 * fixed order): the partials npgp_o8_trinorm_digits gives, for widths the digit path does not take. */
int npgp_sgpr_rownorm_parts(int n, int W, const double* G, long ldg, double* q, long q_stride, npgp_stream_t stream);
/* Finishing kernel of the SGPR posterior draws (sgpr.py posterior().sample()) for one chunk of n rows, one launch: with the
 * residual r_i = [nb_t > 0] max(os_t - q_t, 0) + s max(1 - q_s, 0) of the partials qn (as npgp_sgpr_predict_finish, no V term)
 *   out[s * ldo + i] = mean[i] + F[i * ldf + s] + sqrt(r_i (+ *noise if add_noise)) xi_s(row0 + i),   s < S, i < n
 * xi_s(row) = normal_from_index(seed, 2^63 + (s << 48) + row) as in npgp_svgp_sample.  F (n x ldf, ldf >= S) = K V^T E, its
 * columns s >= S are never read.  Device scalars s, noise (with add_noise), os_t (with nb_t > 0).  S in 1 .. 1024, ldo >= n,
 * row0 >= 0, row0 + n <= 2^48; anything else (and NULL operands) is NPGP_EINVAL. */
int npgp_sgpr_sample_finish(int n, int S, const double* mean, const double* qn, long qn_stride, int nb_t, int nb_s,
                            const double* F, long ldf, const double* s, const double* noise, const double* os_t, int add_noise,
                            unsigned long long seed, long row0, double* out, long ldo, npgp_stream_t stream);

/* ---- the path's one collective (csrc/comm.cu; SURVEY.md section 8(e)): sum all-reduce of the flat fp64 gradient buffer.
 * NCCL is bound at run time (dlopen), the communicator is an opaque handle.  id128: 128-byte token made on one rank by
 * npgp_comm_unique_id and shipped to the others by any means; npgp_comm_create is collective and binds to the current device. */
int npgp_comm_unique_id(void* id128);
int npgp_comm_create(void** comm, const void* id128, int nranks, int rank);
int npgp_comm_destroy(void* comm);
int npgp_allreduce_f64(void* comm, double* buf, long n, npgp_stream_t stream);
int npgp_allreduce_f64_pair(void* comm, double* buf1, long n1, double* buf2, long n2, npgp_stream_t stream); /* one grouped launch */

/* ---- measurement helpers (csrc/peak.cu): FP64 ceiling probes (mode 0 = DFMA loop, 1 = DMMA.8x8x4 loop) and the int8
 * tensor-core ceiling (blocks x reps x 8 back-to-back tcgen05.mma kind::i8 of 128 x n_tile x 32 from resident shared
 * memory; n_tile 256 = densest shape, 64 = the digit engine's tile; collector = A reuse hints) ---- */
int npgp_fp64_peak_probe(int mode, int blocks, int iters, double* out, npgp_stream_t stream);
int npgp_i8_peak_probe(int n_tile, int collector, int blocks, int reps, npgp_stream_t stream);
/* the same for CTA pairs (tcgen05.mma.cta_group::2, 256 x n_tile x 32 per MMA; blocks even) */
int npgp_i8_peak_probe_pair(int n_tile, int collector, int blocks, int reps, npgp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NPGP_H_ */
