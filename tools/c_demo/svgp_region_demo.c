/* A C caller that trains the SVGP-Gibbs model and then returns the posterior of regional sums (basin totals, area means): no
 * Python, no torch.  Reads a problem written by the test (tests/test_svgp_region_gpu.py), runs `iters` calls of npgp_svgp_step
 * on the default stream, then npgp_svgp_predict_prepare and npgp_svgp_region_moments with the full covariance.
 *
 *   gcc -O2 -I include -I /usr/local/cuda/include tools/c_demo/svgp_region_demo.c -o svgp_region_demo \
 *       -L nonstationary_precip_b200 -lnpgp -L /usr/local/cuda/lib64 -lcudart -lm -Wl,-rpath,$PWD/nonstationary_precip_b200
 *   ./svgp_region_demo problem.bin out.bin
 *
 * problem.bin: int header[8] = {variant, d, M, B, N_total, learn_z, include_prior, iters}; doubles x (B,d), y (B), theta (n_pad),
 *   mask (n_pad), the config constants (variant 1: row_os, row_lam (d); variant 0: prior_c (d), prior_os (d), prior_lam (d,d));
 *   int n, R; doubles xs (n,d) sorted by region, w (n); int64 seg (R + 1).
 * out.bin: doubles mean_R (R), var_R (R), cov_R (R*R), theta (n_pad) after training. */
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "npgp.h"

#define CK(call)                                                                      \
  do {                                                                                \
    int rc__ = (int)(call);                                                           \
    if (rc__ != 0) {                                                                  \
      fprintf(stderr, "%s:%d: %s failed with %d\n", __FILE__, __LINE__, #call, rc__); \
      exit(1);                                                                        \
    }                                                                                 \
  } while (0)

static void* to_device(const void* h, long bytes) {
  void* d = NULL;
  CK(cudaMalloc(&d, bytes > 0 ? bytes : 8));
  if (bytes > 0) CK(cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice));
  return d;
}

static double* device_zeros(long n) {
  double* d = NULL;
  CK(cudaMalloc((void**)&d, sizeof(double) * (n > 0 ? n : 1)));
  CK(cudaMemset(d, 0, sizeof(double) * (n > 0 ? n : 1)));
  return d;
}

static void* read_bytes(FILE* f, long bytes) {
  void* h = malloc(bytes > 0 ? bytes : 8);
  if (!h || fread(h, 1, bytes, f) != (size_t)bytes) exit(2);
  return h;
}

int main(int argc, char** argv) {
  if (argc < 3) {
    fprintf(stderr, "usage: %s problem.bin out.bin\n", argv[0]);
    return 2;
  }
  FILE* f = fopen(argv[1], "rb");
  if (!f) return 2;
  int hdr[8];
  if (fread(hdr, sizeof(int), 8, f) != 8) return 2;
  const int variant = hdr[0], d = hdr[1], M = hdr[2], B = hdr[3], iters = hdr[7];
  npgp_svgp_config cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.variant = variant, cfg.d = d, cfg.M = M, cfg.B_local = B, cfg.N_total = hdr[4], cfg.B_global = B, cfg.world_size = 1;
  cfg.jitter_zz = 1e-6, cfg.jitter_xx = 1e-4, cfg.kernel_jitter = 1e-5, cfg.min_var = 1e-6;
  cfg.learn_z = hdr[5], cfg.include_prior = hdr[6];
  const long n_pad = npgp_svgp_theta_size(&cfg);
  if (n_pad <= 0) return 3;
  const long n_const = variant == 1 ? 1 + d : 2 * d + d * d;
  const long nh = (long)B * d + B + 2 * n_pad + n_const;
  double* h = (double*)read_bytes(f, 8 * nh);
  int nr[2];
  if (fread(nr, sizeof(int), 2, f) != 2 || nr[0] <= 0 || nr[1] <= 0) return 2;
  const int n = nr[0], R = nr[1];
  double* hrows = (double*)read_bytes(f, 8L * ((long)n * d + n));
  long* hseg = (long*)read_bytes(f, 8L * (R + 1));
  fclose(f);
  const double *hx = h, *hy = hx + (long)B * d, *htheta = hy + B, *hmask = htheta + n_pad, *hconst = hmask + n_pad;
  double *x = (double*)to_device(hx, 8L * B * d), *y = (double*)to_device(hy, 8L * B);
  double *theta = (double*)to_device(htheta, 8 * n_pad), *mask = (double*)to_device(hmask, 8 * n_pad);
  double* consts = (double*)to_device(hconst, 8 * n_const);
  double* xs = (double*)to_device(hrows, 8L * n * d);
  double* w = (double*)to_device(hrows + (long)n * d, 8L * n);
  long* seg = (long*)to_device(hseg, 8L * (R + 1));
  if (variant == 1) cfg.row_os = consts, cfg.row_lam = consts + 1;
  else cfg.prior_c = consts, cfg.prior_os = consts + d, cfg.prior_lam = consts + 2 * d;

  // ---- training: the plan, its workspace and the optimiser state, as in svgp_step_demo.c
  double *grad = device_zeros(n_pad + 2), *adam_m = device_zeros(n_pad), *adam_v = device_zeros(n_pad), *step = device_zeros(1);
  int* status;
  void* ws;
  const long ws_bytes = npgp_svgp_workspace_bytes(&cfg);
  CK(cudaMalloc((void**)&status, sizeof(int)));
  CK(cudaMemset(status, 0, sizeof(int)));
  CK(cudaMalloc(&ws, ws_bytes));
  npgp_svgp_plan* plan = NULL;
  CK(npgp_svgp_plan_create(&plan, &cfg, ws, ws_bytes));
  for (int it = 0; it < iters; ++it)
    CK(npgp_svgp_step(plan, x, y, theta, grad, adam_m, adam_v, mask, step, status, 0.01, 0.9, 0.999, 1e-8, NULL, 0));

  // ---- regional sums on the same plan: mean, variances and the R x R covariance (rows streamed in chunks of B)
  const long n_out = 2L * R + (long)R * R;
  double* out = device_zeros(n_out);
  const long rw_bytes = npgp_svgp_region_workspace_bytes(&cfg, n, R, 1);
  if (rw_bytes <= 0) return 3;
  void* rw;
  CK(cudaMalloc(&rw, rw_bytes)); /* cudaMalloc returns 256-byte aligned memory */
  CK(npgp_svgp_predict_prepare(plan, theta, status, 0));
  CK(npgp_svgp_region_moments(plan, n, xs, w, R, seg, theta, 0, 0, 1, out, out + R, out + 2 * R, R, rw, rw_bytes, 0));
  double* hout = (double*)malloc(sizeof(double) * (n_out + n_pad));
  CK(cudaMemcpy(hout, out, sizeof(double) * n_out, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hout + n_out, theta, sizeof(double) * n_pad, cudaMemcpyDeviceToHost));
  int hstatus = -1;
  CK(cudaMemcpy(&hstatus, status, sizeof(int), cudaMemcpyDeviceToHost));
  f = fopen(argv[2], "wb");
  if (!f) return 2;
  fwrite(hout, sizeof(double), n_out + n_pad, f);
  fclose(f);
  CK(npgp_svgp_plan_destroy(plan));
  CK(cudaFree(rw));
  printf("npgp %d: %d steps, status %d, %d regions over %d rows; region 0: mean %.6g, sd %.6g\n", npgp_version(), iters,
         hstatus, R, n, hout[0], hout[R] > 0 ? __builtin_sqrt(hout[R]) : -1.0);
  return hstatus == 0 ? 0 : 4;
}
