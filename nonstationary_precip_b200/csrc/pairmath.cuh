// Per-pair arithmetic of the Gibbs kernels, shared by every tile kernel (the host branches only keep the header compilable
// by a host compiler; the product calls these from CUDA kernels, and tests/test_pairmath_range_gpu.py checks them there).
//
// Diagonal kernel  (reference: models/gibbs_kernels.py:154-162):
//     K_ij = prod_d sqrt(2 l_id l_jd / s_d) * exp(-sum_d delta_d^2 / s_d),  s_d = l_id^2 + l_jd^2
//   evaluated in common-denominator form with P = prod_d s_d, r = rsqrt(P):
//     K_ij = c_i c_j r exp(-r^2 sum_d delta_d^2 prod_{e!=d} s_e),   c_i = sqrt(2^{D/2} prod_d l_id)
//   -> one rsqrt + one exp per pair, no division.
// Full-matrix kernel (reference: models/multivariate_gibbs_kernel.py:101-150):
//     K_ij = det(S_i)^(1/4) det(S_j)^(1/4) det(A)^(-1/2) exp(-delta^T (A + eps I)^-1 delta),  A = (S_i + S_j)/2
//   with At = S_i + S_j:  det(A) = det(At)/2^d,  (A + eps I)^-1 = 2 (At + 2 eps I)^-1 = 2 adj(Bt)/det(Bt).
#pragma once
#include <math.h>

#include "exp_table.cuh"

#if defined(__CUDACC__)
#define NPGP_HD __host__ __device__ __forceinline__
#else
#define NPGP_HD inline
#endif

namespace npgp {

// 1/sqrt(x) and 1/x for the tile kernels: hardware seed (MUFU.RSQ64H / MUFU.RCP64H, ~20 bits) + two Newton steps, branch
// free.  The library versions carry special-case paths (BSSY/CALL around every use) that cost ~30 % of the tile kernels'
// issue slots; the arguments here (products of squared lengthscales, determinants of positive definite 2x2 / 3x3
// matrices) are positive normal numbers.  A NaN argument returns NaN (the seed instructions and FMAs propagate it); so do
// 0 and +inf (the Newton step forms 0 * inf) and, for fast_rsqrt, negative numbers.  A singular or indefinite Sigma thus
// shows up as NaN in K, as a failed factorisation would.
NPGP_HD double fast_rsqrt(double x) {
#if defined(__CUDA_ARCH__)
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double h = 0.5 * x;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const double e = fma(-h * y, y, 0.5);
    y = fma(y, e, y);
  }
  return y;
#else
  return 1.0 / sqrt(x);
#endif
}

#if defined(__CUDACC__)
__host__ __device__
#endif
// exp(x) for x <= 0 (the only case on this path: K = prefactor * exp(-Q)).  Table-driven: x = (256 k + j) ln2/256 + r,
// |r| <= ln2/512, exp(x) = 2^k * 2^(j/256) * (1 + r + r^2/2 + r^3/6 + r^4/24)  (remainder r^5/120 < 4e-17).  About 10 FP64
// instructions instead of ~25-30 for the library exp -- the Gibbs / RBF tile kernels are FP64-pipe bound and spend one
// exp per pair.  `tab` is the 256-entry table of 2^(j/256) (in shared memory on the device).
NPGP_HD double exp_neg(double x, const double* tab) {
#if defined(__CUDA_ARCH__)
  // Branch free.  exp(-708) = 3e-308 stands in for the underflowed tail; the clamp is a compare-and-select rather than fmax
  // so that a NaN argument (a missing coordinate) passes through to t, whose high word is >= 0x7ff00000 exactly when x is
  // NaN (or +inf).  The last line returns t then: the exponent-field add would turn a NaN v into a finite number.
  x = (x < -708.0) ? -708.0 : x;
  const double t = fma(x, kInvLn2x256, 6755399441055744.0);  // 2^52 + 2^51: the integer lands in the low mantissa bits
  const int n = __double2loint(t);
  const double nd = t - 6755399441055744.0;
  double r = fma(nd, -kLn2d256Hi, x);
  r = fma(nd, -kLn2d256Lo, r);
  double p = fma(r, 1.0 / 24.0, 1.0 / 6.0);
  p = fma(p, r, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const double v = tab[n & 255] * p;  // in [1, 2) up to rounding
  const double e = __hiloint2double(__double2hiint(v) + ((n >> 8) << 20), __double2loint(v));  // * 2^k via the exponent
  return (static_cast<unsigned>(__double2hiint(t)) >= 0x7ff00000u) ? t : e;
#else
  (void)tab;
  return exp(x);
#endif
}

NPGP_HD double fast_rcp(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
  }
  return r;
#else
  return 1.0 / x;
#endif
}

constexpr int sym_size(int d) { return d * (d + 1) / 2; }

// ---------------------------------------------------------------------------------------------------------------------
// diagonal Gibbs
// ---------------------------------------------------------------------------------------------------------------------
template <int D>
struct DiagPair {
  double k;       // unscaled kernel value
  double is[D];   // 1 / s_d
  double dl[D];   // delta_d = x_id - z_jd
};

// xi, ai = l_i^2, ci as above (row point); zj, bj, cj (column point)
template <int D>
NPGP_HD double gibbs_diag_eval(const double* xi, const double* ai, double ci, const double* zj, const double* bj,
                               double cj, const double* etab, DiagPair<D>* out = nullptr) {
  double s[D], dl[D], pre[D + 1], suf[D + 1];
#pragma unroll
  for (int d = 0; d < D; ++d) {
    s[d] = ai[d] + bj[d];
    dl[d] = xi[d] - zj[d];
  }
  pre[0] = 1.0;
#pragma unroll
  for (int d = 0; d < D; ++d) pre[d + 1] = pre[d] * s[d];
  suf[D] = 1.0;
#pragma unroll
  for (int d = D - 1; d >= 0; --d) suf[d] = suf[d + 1] * s[d];
  const double P = pre[D];
  double num = 0.0;
  double pe[D];
#pragma unroll
  for (int d = 0; d < D; ++d) {
    pe[d] = pre[d] * suf[d + 1];
    num = fma(dl[d] * dl[d], pe[d], num);
  }
  const double r = fast_rsqrt(P);
  const double r2 = r * r;
  const double k = (ci * cj) * r * exp_neg(-num * r2, etab);
  if (out) {
    out->k = k;
#pragma unroll
    for (int d = 0; d < D; ++d) {
      out->is[d] = pe[d] * r2;
      out->dl[d] = dl[d];
    }
  }
  return k;
}

// ---------------------------------------------------------------------------------------------------------------------
// small symmetric matrices, packed row-wise upper triangle: d=2 [00,01,11]; d=3 [00,01,02,11,12,22]
// ---------------------------------------------------------------------------------------------------------------------
template <int d>
NPGP_HD void sym_adj_det(const double* m, double* adj, double& det);

template <>
NPGP_HD void sym_adj_det<2>(const double* m, double* adj, double& det) {
  adj[0] = m[2];
  adj[1] = -m[1];
  adj[2] = m[0];
  det = fma(m[0], m[2], -m[1] * m[1]);
}

template <>
NPGP_HD void sym_adj_det<3>(const double* m, double* adj, double& det) {
  adj[0] = fma(m[3], m[5], -m[4] * m[4]);
  adj[1] = fma(m[2], m[4], -m[1] * m[5]);
  adj[2] = fma(m[1], m[4], -m[2] * m[3]);
  adj[3] = fma(m[0], m[5], -m[2] * m[2]);
  adj[4] = fma(m[1], m[2], -m[0] * m[4]);
  adj[5] = fma(m[0], m[3], -m[1] * m[1]);
  det = fma(m[0], adj[0], fma(m[1], adj[1], m[2] * adj[2]));
}

template <int d>
NPGP_HD double sym_det(const double* m) {
  double adj[sym_size(d)], det;
  sym_adj_det<d>(m, adj, det);
  return det;
}

// y = M v for packed symmetric M
template <int d>
NPGP_HD void sym_matvec(const double* m, const double* v, double* y);
template <>
NPGP_HD void sym_matvec<2>(const double* m, const double* v, double* y) {
  y[0] = fma(m[0], v[0], m[1] * v[1]);
  y[1] = fma(m[1], v[0], m[2] * v[1]);
}
template <>
NPGP_HD void sym_matvec<3>(const double* m, const double* v, double* y) {
  y[0] = fma(m[0], v[0], fma(m[1], v[1], m[2] * v[2]));
  y[1] = fma(m[1], v[0], fma(m[3], v[1], m[4] * v[2]));
  y[2] = fma(m[2], v[0], fma(m[4], v[1], m[5] * v[2]));
}

// packed index helper (compile-time unrolled loops use it)
NPGP_HD int sym_idx(int d, int k, int l) {  // k <= l
  return k * d - (k * (k - 1)) / 2 + (l - k);
}

// adjugate / determinant of Bt = At + lam I from those of At, d = 3: the off-diagonal cofactors differ by -lam * At_p (one
// FMA instead of a product and an FMA); the diagonal ones are recomputed from the shifted diagonal (same cost either way)
template <int d>
NPGP_HD void sym_adj_det_shifted(const double* At, const double* adjA, double lam, double* adjB, double& detB);
template <>
NPGP_HD void sym_adj_det_shifted<2>(const double* At, const double* adjA, double lam, double* adjB, double& detB) {
  (void)adjA;
  const double b0 = At[0] + lam, b2 = At[2] + lam;
  adjB[0] = b2;
  adjB[1] = -At[1];
  adjB[2] = b0;
  detB = fma(b0, b2, -At[1] * At[1]);
}
template <>
NPGP_HD void sym_adj_det_shifted<3>(const double* At, const double* adjA, double lam, double* adjB, double& detB) {
  const double b0 = At[0] + lam, b3 = At[3] + lam, b5 = At[5] + lam;
  adjB[0] = fma(b3, b5, -At[4] * At[4]);
  adjB[1] = fma(-lam, At[1], adjA[1]);
  adjB[2] = fma(-lam, At[2], adjA[2]);
  adjB[3] = fma(b0, b5, -At[2] * At[2]);
  adjB[4] = fma(-lam, At[4], adjA[4]);
  adjB[5] = fma(b0, b3, -At[1] * At[1]);
  detB = fma(b0, adjB[0], fma(At[1], adjB[1], At[2] * adjB[2]));
}

template <int d>
struct FullPair {
  double k;                  // kernel value (scaled as qj is)
  double w[d];               // (A + eps I)^-1 delta
  double adjA[sym_size(d)];  // adj(At), At = S_i + S_j
  double hr2;                // 0.5 / det(At): 0.25 A^-1 = hr2 * adjA
};

// xi, Si (packed), qi = det(Si)^(1/4); column point zj, Sj and qj = 2^(d/2) det(Sj)^(1/4) [* outputscale]: the constant of
// det(A)^(-1/2) = 2^(d/2) rsqrt(det At) is folded into the column factor by the callers (full_col_factor).  jit2 = 2 * jitter.
template <int d>
NPGP_HD double full_col_factor(double det_Sj) {
  return ((d == 2) ? 2.0 : 2.8284271247461900976) * sqrt(sqrt(det_Sj));
}

template <int d>
NPGP_HD double gibbs_full_eval(const double* xi, const double* Si, double qi, const double* zj, const double* Sj,
                               double qj, double jit2, const double* etab, FullPair<d>* out = nullptr) {
  constexpr int P = sym_size(d);
  double At[P], adjA[P], adjB[P], detA, detB, dl[d], v[d];
#pragma unroll
  for (int p = 0; p < P; ++p) At[p] = Si[p] + Sj[p];
#pragma unroll
  for (int k = 0; k < d; ++k) dl[k] = xi[k] - zj[k];
  sym_adj_det<d>(At, adjA, detA);
  sym_adj_det_shifted<d>(At, adjA, jit2, adjB, detB);
  sym_matvec<d>(adjB, dl, v);
  double dv = 0.0;
#pragma unroll
  for (int k = 0; k < d; ++k) dv = fma(dl[k], v[k], dv);
  const double nidetB2 = -2.0 * fast_rcp(detB);  // -(A + eps I)^-1 = nidetB2 * adj(Bt)
  const double r = fast_rsqrt(detA);
  const double k = (qi * qj) * r * exp_neg(dv * nidetB2, etab);
  if (out) {
    out->k = k;
    out->hr2 = 0.5 * r * r;
#pragma unroll
    for (int a = 0; a < d; ++a) out->w[a] = -v[a] * nidetB2;
#pragma unroll
    for (int p = 0; p < P; ++p) out->adjA[p] = adjA[p];
  }
  return k;
}

// softplus with torch's threshold (20): Sigma_kl = softplus(u^2) + D_kl^2, u = h_k h_l
NPGP_HD double softplus20(double t) { return t > 20.0 ? t : log1p(exp(t)); }
NPGP_HD double sigmoid20(double t) { return t > 20.0 ? 1.0 : 1.0 / (1.0 + exp(-t)); }

template <int d>
NPGP_HD void sigma_from_h_row(const double* h, const double* Dm /* d x d row-major */, double* S /* packed */) {
#pragma unroll
  for (int k = 0; k < d; ++k)
#pragma unroll
    for (int l = k; l < d; ++l) {
      const double u = h[k] * h[l];
      S[sym_idx(d, k, l)] = softplus20(u * u) + Dm[k * d + l] * Dm[k * d + l];
    }
}

}  // namespace npgp
