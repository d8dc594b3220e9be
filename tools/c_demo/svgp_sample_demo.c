/* A C caller that trains the SVGP-Gibbs model and then draws posterior sample fields from it: no Python, no torch.  Reads a
 * problem written by the test (tests/test_svgp_sample_gpu.py), runs `iters` calls of npgp_svgp_step on the default stream,
 * then npgp_svgp_predict_prepare, npgp_svgp_predict (mean and var_f) and npgp_svgp_sample_prepare + npgp_svgp_sample on a
 * block of test rows.
 *
 *   gcc -O2 -I include -I /usr/local/cuda/include tools/c_demo/svgp_sample_demo.c -o svgp_sample_demo \
 *       -L nonstationary_precip_b200 -lnpgp -L /usr/local/cuda/lib64 -lcudart -lm -Wl,-rpath,$PWD/nonstationary_precip_b200
 *   ./svgp_sample_demo problem.bin out.bin [S [seed]]
 *
 * problem.bin: the format of svgp_predict_demo.c (the test targets ys are read and not used).
 * out.bin: doubles mean (n), var_f (n), draws (S*n, draw-major), theta (n_pad) after training.  Prints the largest distance
 *   of the draws' average from the mean, in standard errors sqrt(var_f / S). */
#include <cuda_runtime.h>
#include <math.h>
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

static double* to_device(const double* h, long n) {
  double* d = NULL;
  CK(cudaMalloc((void**)&d, sizeof(double) * (n > 0 ? n : 1)));
  if (n > 0) CK(cudaMemcpy(d, h, sizeof(double) * n, cudaMemcpyHostToDevice));
  return d;
}

static double* device_zeros(long n) {
  double* d = NULL;
  CK(cudaMalloc((void**)&d, sizeof(double) * (n > 0 ? n : 1)));
  CK(cudaMemset(d, 0, sizeof(double) * (n > 0 ? n : 1)));
  return d;
}

static double* read_doubles(FILE* f, long n) {
  double* h = (double*)malloc(sizeof(double) * (n > 0 ? n : 1));
  if (!h || fread(h, sizeof(double), n, f) != (size_t)n) exit(2);
  return h;
}

int main(int argc, char** argv) {
  if (argc < 3) {
    fprintf(stderr, "usage: %s problem.bin out.bin [S [seed]]\n", argv[0]);
    return 2;
  }
  const int S = argc > 3 ? atoi(argv[3]) : 64;
  const unsigned long long seed = argc > 4 ? strtoull(argv[4], NULL, 10) : 0ull;
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
  double* h = read_doubles(f, (long)B * d + B + 2 * n_pad + n_const);
  int n = 0;
  if (fread(&n, sizeof(int), 1, f) != 1 || n <= 0) return 2;
  double* ht = read_doubles(f, (long)n * d + n);
  fclose(f);
  const double *hx = h, *hy = hx + (long)B * d, *htheta = hy + B, *hmask = htheta + n_pad, *hconst = hmask + n_pad;
  double *x = to_device(hx, (long)B * d), *y = to_device(hy, B), *theta = to_device(htheta, n_pad), *mask = to_device(hmask, n_pad);
  double *xs = to_device(ht, (long)n * d);
  double* consts = to_device(hconst, n_const);
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

  // ---- the posterior on the same plan: marginals, then S correlated draws (streamed in chunks of B)
  double* out = device_zeros(2L * n + (long)S * n);
  double *mean = out, *var_f = mean + n, *draws = var_f + n;
  CK(npgp_svgp_predict_prepare(plan, theta, status, 0));
  CK(npgp_svgp_predict(plan, n, xs, NULL, theta, mean, var_f, NULL, NULL, NULL, NULL, 0));
  const long sw_bytes = npgp_svgp_sample_workspace_bytes(&cfg, S);
  if (sw_bytes <= 0) return 3;
  void* sw;
  CK(cudaMalloc(&sw, sw_bytes));  /* cudaMalloc returns 256-byte aligned memory */
  CK(npgp_svgp_sample_prepare(plan, theta, S, seed, sw, sw_bytes, 0));
  CK(npgp_svgp_sample(plan, n, xs, 0, theta, 0, draws, n, sw, sw_bytes, 0));
  const long n_out = 2L * n + (long)S * n;
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
  CK(cudaFree(sw));
  double worst = 0.0;
  int finite = 1;
  for (int i = 0; i < n; ++i) {
    double acc = 0.0;
    for (int s = 0; s < S; ++s) {
      const double v = hout[2L * n + (long)s * n + i];
      finite &= isfinite(v) != 0;
      acc += v;
    }
    const double z = fabs(acc / S - hout[i]) / sqrt(hout[n + i] / S);
    if (z > worst) worst = z;
  }
  printf("npgp %d: %d steps, status %d, %d draws at %d rows: %s, largest |average - mean| %.3f standard errors\n",
         npgp_version(), iters, hstatus, S, n, finite ? "finite" : "NOT finite", worst);
  return hstatus == 0 && finite ? 0 : 4;
}
