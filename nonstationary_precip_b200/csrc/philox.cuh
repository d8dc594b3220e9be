// Counter-based standard normals: Philox4x32-10 keyed by (seed, 64-bit element index).  A draw depends only on its seed and
// index, never on how elements are spread over launches, chunks or ranks.  Used by the DSVI samples (dsvi.cu) and the SVGP
// posterior sampler (svgp_step.cu).
#pragma once
#include <cstdint>

namespace npgp {

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t* out) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// one standard normal per element index (Box-Muller on two 32+21-bit uniforms)
__device__ __forceinline__ double normal_from_index(unsigned long long seed, unsigned long long idx) {
  uint32_t r[4];
  philox4x32_10((uint32_t)idx, (uint32_t)(idx >> 32), 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
  const double u1 = ((double)r[0] * 4294967296.0 + (double)r[1] + 0.5) * (1.0 / 18446744073709551616.0);  // (0,1)
  const double u2 = ((double)r[2] * 4294967296.0 + (double)r[3] + 0.5) * (1.0 / 18446744073709551616.0);
  return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

}  // namespace npgp
