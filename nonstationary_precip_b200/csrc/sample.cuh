// Store loop of the posterior samplers' finishing kernels (svgp_sample_finish_kernel in svgp_step.cu,
// sgpr_sample_finish_kernel in sgpr_predict.cu).  CTA = 32 rows x 8 thread rows; the caller's thread row 0 has put the mean
// and the standard deviation of the independent part of each of the CTA's rows into smean / ssd.  For s < S, i < n:
//   out[s ldo + i] = smean_i + (F[i ldf + s] + ssd_i xi_s(row0 + i)),   xi_s(row) = normal_from_index(seed, 2^63 + (s << 48) + row)
// F is read along s and written along i through a shared-memory tile; its columns s >= S are never read.
#pragma once
#include "philox.cuh"

namespace npgp {

__device__ __forceinline__ void sample_store_rows(int n, int S, const double* __restrict__ F, long ldf, unsigned long long seed,
                                                  long row0, double* __restrict__ out, long ldo, double (&tile)[32][33],
                                                  const double* smean, const double* ssd) {
  const int tx = threadIdx.x, ty = threadIdx.y, i0 = blockIdx.x * 32, i = i0 + tx;
  for (int s0 = 0; s0 < S; s0 += 32) {
    for (int rr = ty; rr < 32; rr += 8) {
      const int s = s0 + tx;
      tile[rr][tx] = (i0 + rr < n && s < S) ? F[(long)(i0 + rr) * ldf + s] : 0.0;
    }
    __syncthreads();
    for (int c = ty; c < 32; c += 8) {
      const int s = s0 + c;
      if (s < S && i < n) {
        const double xi = normal_from_index(seed, (1ull << 63) + ((unsigned long long)s << 48) + (unsigned long long)(row0 + i));
        out[(long)s * ldo + i] = smean[tx] + fma(ssd[tx], xi, tile[tx][c]);
      }
    }
    __syncthreads();
  }
}

}  // namespace npgp
