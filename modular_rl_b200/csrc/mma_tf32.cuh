// Warp-level tensor-core pieces shared by the fused chain kernels and the layer-by-layer path: mma.sync m16n8k8 TF32 in split
// precision (3xTF32).  x = hi + lo with hi = rna_tf32(x), lo = x - hi (exact in fp32);
// D += lo.hi + hi.lo + hi.hi keeps FP32-class accuracy (north_star: 1e-5) at 1/3 of the TF32 rate.
#pragma once
#include <stdint.h>
#include "common.cuh"

__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  // round-to-nearest TF32 by integer arithmetic on the sign-magnitude bits (cvt.rna.tf32 costs ~4
  // instructions on sm_100a): add half an ulp, then truncate.  hi must be exact for the subtraction;
  // for lo the tensor core's own truncation of the low 13 bits completes the rounding.  Rounding (not
  // truncating) hi matters: with a truncated hi the dropped lo.lo term is one-signed, a 2e-7 relative
  // bias that the CG solve amplifies (measured on the ill-conditioned golden case).
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi)) + 0x1000u;
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// MT x 2 mma tiles, three passes (lo.hi, hi.lo, hi.hi) so that consecutive MMAs hit different accumulators
template <int MT>
__device__ __forceinline__ void mma3_tiles(float (&acc)[MT][2][4], const uint32_t (&ah)[MT][4],
                                           const uint32_t (&al)[MT][4], const uint32_t (&bh)[2][2],
                                           const uint32_t (&bl)[2][2]) {
#pragma unroll
  for (int mi = 0; mi < MT; ++mi)
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) mma_tf32(acc[mi][ni], al[mi], bh[ni]);
#pragma unroll
  for (int mi = 0; mi < MT; ++mi)
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) mma_tf32(acc[mi][ni], ah[mi], bl[ni]);
#pragma unroll
  for (int mi = 0; mi < MT; ++mi)
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) mma_tf32(acc[mi][ni], ah[mi], bh[ni]);
}

// acc[mi][ni] += A^T-tile . B-tile over k in [0,K): A_T[k][r] feature-major activations (ld = MRL_LDT),
// B[k][c] row-major weights (ld = ldb).  Warp tile (16*MT) rows x 16 cols = MT x 2 mma tiles.
template <int MT, bool TAIL>
__device__ __forceinline__ void mma_fwd_step(float (&acc)[MT][2][4], const float* __restrict__ a,
                                             const float* __restrict__ b0, const float* __restrict__ b1, int ldb4,
                                             int krem) {
  // a -> A_T[k0 + t][r0 + g], b0/b1 -> B[k0 + t][c], ldb4 = 4 * ldb ; rows k0+t and k0+t+4
  const bool va = !TAIL || krem > 0, vb = !TAIL || krem > 4;   // krem = K - (k0 + t)
  uint32_t bh[2][2], bl[2][2], ah[MT][4], al[MT][4];
  split_tf32(va ? b0[0] : 0.f, bh[0][0], bl[0][0]);
  split_tf32(vb ? b0[ldb4] : 0.f, bh[0][1], bl[0][1]);
  split_tf32(va ? b1[0] : 0.f, bh[1][0], bl[1][0]);
  split_tf32(vb ? b1[ldb4] : 0.f, bh[1][1], bl[1][1]);
#pragma unroll
  for (int mi = 0; mi < MT; ++mi) {
    split_tf32(va ? a[16 * mi] : 0.f, ah[mi][0], al[mi][0]);
    split_tf32(va ? a[16 * mi + 8] : 0.f, ah[mi][1], al[mi][1]);
    split_tf32(vb ? a[4 * MRL_LDT + 16 * mi] : 0.f, ah[mi][2], al[mi][2]);
    split_tf32(vb ? a[4 * MRL_LDT + 16 * mi + 8] : 0.f, ah[mi][3], al[mi][3]);
  }
  mma3_tiles<MT>(acc, ah, al, bh, bl);
}
template <int MT>
__device__ __forceinline__ void mma_fwd_acc(float (&acc)[MT][2][4], const float* __restrict__ A,
                                            const float* __restrict__ B, int K, int ldb, int r0, int c0,
                                            int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float* a = A + t * MRL_LDT + r0 + g;
  const float* b0 = B + t * ldb + min(c0 + g, ldb - 1);
  const float* b1 = B + t * ldb + min(c0 + 8 + g, ldb - 1);
  const int ldb4 = 4 * ldb, ldb8 = 8 * ldb;
  int k0 = 0;
#pragma unroll 2
  for (; k0 + 8 <= K; k0 += 8) {
    mma_fwd_step<MT, false>(acc, a, b0, b1, ldb4, 8);
    a += 8 * MRL_LDT; b0 += ldb8; b1 += ldb8;
  }
  if (k0 < K) mma_fwd_step<MT, true>(acc, a, b0, b1, ldb4, K - k0 - t);
}
