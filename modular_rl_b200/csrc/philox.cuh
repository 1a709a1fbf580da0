// Philox4x32-10 (Salmon et al., SC'11; the constants and round of Random123 and curand_philox4x32_x.h) and the
// 53-bit uniform taken from two of its output words.  Every device draw of the project is keyed by a round seed (low
// word, high word) and addressed by a counter whose third word is the PURPOSE of the draw, so the streams of
// different purposes never share a counter.  oracle/rollout.py restates both functions in numpy.
#pragma once
#ifdef __CUDACC_RTC__   // NVRTC (rollout_user.cu) has no <stdint.h>
#include <cuda/std/cstdint>
using cuda::std::uint32_t;
#else
#include <stdint.h>
#endif

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    if (i) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
  }
  return c;
}
// 53-bit uniform in [0, 1) from two words: the high word gives the top 32 bits, the high 21 bits of the low word the rest
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
  return (double)(((unsigned long long)hi << 21) | (lo >> 11)) * 0x1p-53;
}
// counter word 2.  Reset and action draws of a rollout round: (environment, step, purpose, block); the cross-entropy
// search's candidate normals: (member, pair of parameters, purpose, 0), cem_search.cu
enum { RO_PURPOSE_RESET = 0, RO_PURPOSE_ACTION = 1, CEM_PURPOSE_DRAW = 2 };
