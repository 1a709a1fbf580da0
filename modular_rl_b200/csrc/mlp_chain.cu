// Layers >= 2 of the MLP as register-resident per-warp chains: forward (losses, activation cache) and
// gradient (trpo.py:37-43,60-63; ppo.py:35-49; core.py:613-617).  The Fisher-vector product runs in
// mlp_fvp_tc.cu.
//
// Backward kernel (gradient): one CTA of 12 warps owns a slab of <= 1024 timesteps and walks it in
// chain tiles of 192 timesteps (3 cache tiles).
//
//   chain phase  Each warp owns 16 timesteps and carries them from the head gradient through the whole
//                reverse sweep WITHOUT block barriers: the m16n8 accumulator fragment of one layer is
//                the A fragment of the next (k-slot t <-> feature 2t, slot t+4 <-> feature 2t+1, so no
//                shuffle is needed), weights are read from shared memory in an 8x8-block layout that is
//                bank-conflict free for both W (forward) and W^T (delta) fragment reads, cached
//                activations come straight from HBM/L2 in fragment order (a thread's two fragment rows are
//                adjacent timesteps: 64-bit accesses).  Every product is 3xTF32 (mma_tf32.cuh).  delta_l
//                (l >= 2) is left in shared memory as fp32 rows, delta_1 goes to HBM as the pre-split
//                tcgen05 operand of l1_grad_tc_kernel.
//   grad phase   After ONE barrier the weight gradients G_l = h_{l-1}^T delta_l (K = the 192 timesteps)
//                are accumulated by a static (layer, m-tile, n-tiles) -> warp assignment: every accumulator
//                block has one owner, lives in shared memory between chain tiles and is flushed once as the
//                fp32 slab partial that reduce_partials_kernel sums in fp64.
//
// Two barriers per 192 timesteps (the job-list kernel in mlp_mid.cu needs ~10 per 64) and ~2x fewer
// issued instructions per timestep; see DESIGN.md section 4 for the measured effect.
#include "common.cuh"
#include "heads.cuh"
#include "kernels.h"
#include "mma_tf32.cuh"
#include <string.h>

#define CH_THREADS (32 * CH_WARPS)   // backward chain kernel: 384 threads, <= 168 registers
#define CH_TILES (CH_WARPS / 4)     // cache tiles (64 timesteps) per chain tile
#define CH_T (16 * CH_WARPS)        // timesteps per chain tile
#define CH_LDE (CH_T + 8)           // floats between consecutive delta rows in shared memory (= 8 mod 32: the
                                    // 64-bit fragment reads of the grad phase are bank-conflict free)
#define FW_WARPS 8                  // forward chain kernel: 256 threads, 2 CTAs per SM
#define FW_THREADS (32 * FW_WARPS)

template <int L_, int N1_, int N2_, int N3_, int N4_>
struct ChainShape {
  static constexpr int L = L_;
  __host__ __device__ static constexpr int nt(int l) { return l == 1 ? N1_ : (l == 2 ? N2_ : (l == 3 ? N3_ : N4_)); }
  // weight blocks of layer l (l >= 2): [in-block][out-block][64]
  __host__ __device__ static constexpr int woff(int l) {
    int s = 0;
    for (int k = 2; k < l; ++k) s += nt(k - 1) * nt(k) * 64;
    return s;
  }
  __host__ __device__ static constexpr int wfloats() { return woff(L_ + 1); }
  __host__ __device__ static constexpr int eoff(int l) {   // first delta row of layer l (l >= 2)
    int s = 0;
    for (int k = 2; k < l; ++k) s += 8 * nt(k);
    return s;
  }
  __host__ __device__ static constexpr int erows() { return eoff(L_ + 1); }
  __host__ __device__ static constexpr int vboff(int l) {  // bias of layer l (l >= 1) in the forward kernel
    int s = 0;
    for (int k = 1; k < l; ++k) s += 8 * nt(k);
    return s;
  }
  __host__ __device__ static constexpr int vbfloats() { return vboff(L_ + 1); }
  // weight-gradient accumulator blocks (m16 x n8, one float4 per lane) of all layers >= 2, upper bound
  __host__ __device__ static constexpr int gblocks() {
    int s = 0;
    for (int k = 2; k <= L_; ++k) s += ((8 * nt(k - 1) + 15) / 16) * nt(k);
    return s;
  }
  __host__ __device__ static constexpr size_t smem_floats() {   // backward kernel
    return (size_t)wfloats() + 16 * nt(L_) + CH_WARPS * 8 * (N1_ + nt(L_)) + (size_t)gblocks() * 128 +
           (size_t)erows() * CH_LDE;
  }
};

// split barriers between the chain and grad phases (one arrive per warp): a warp signals as soon as ITS part is
// done and only waits where it really needs the others' data, so the skew between warps is absorbed by work
__device__ __forceinline__ void warp_arrive(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) return;
    if (++spins > (1u << 26)) __trap();   // a protocol bug becomes an error, never a hung GPU
  }
}

// row of feature j' (0..7) inside an 8x8 weight block: conflict-free for the 64-bit W reads (lanes g = 0..3 /
// 4..7 of a half-warp hit rows with distinct (row mod 4)) and for the 32-bit W^T reads (rows 2t / 2t+1).
__device__ __forceinline__ int blk_row(int j) { return j < 4 ? j : (j ^ 1); }

// A thread's two fragment rows (g and g+8 of the m16 tile) are mapped to ADJACENT timesteps 2g and 2g+1 of the
// warp's 16, so one 64-bit access moves both rows of a feature (p already points at timestep 2g).
__device__ __forceinline__ void ldfrag(float (&v)[4], const float* __restrict__ p, int f0, int dmax, bool ok) {
  const bool k0 = ok && f0 < dmax, k1 = ok && f0 + 1 < dmax;
  const float2 a = k0 ? __ldg(reinterpret_cast<const float2*>(p + f0 * MRL_LDT)) : make_float2(0.f, 0.f);
  const float2 b = k1 ? __ldg(reinterpret_cast<const float2*>(p + (f0 + 1) * MRL_LDT)) : make_float2(0.f, 0.f);
  v[0] = a.x; v[2] = a.y;
  v[1] = b.x; v[3] = b.y;
}
// accumulator-order values (c0..c3) -> A-fragment order (a0 = c0, a1 = c2, a2 = c1, a3 = c3), split
__device__ __forceinline__ void to_frag(const float (&v)[4], uint32_t (&hi)[4], uint32_t (&lo)[4]) {
  split_tf32(v[0], hi[0], lo[0]);
  split_tf32(v[2], hi[1], lo[1]);
  split_tf32(v[1], hi[2], lo[2]);
  split_tf32(v[3], hi[3], lo[3]);
}

// acc[n] += A(k-step ks) . B(block), n-tiles nb .. nb+NT-1.  TRANS = false: B = W_l (K = in features, N = out),
// TRANS = true: B = W_l^T (K = out features, N = in).  ntl = out-blocks of layer l.
template <int NT, bool TRANS>
__device__ __forceinline__ void kstep(float (&acc)[NT][4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                      const float* __restrict__ W, int ks, int nb, int ntl, int lane) {
  const int g = lane >> 2, t = lane & 3;
  // RND independent accumulators per pass: consecutive MMAs on one accumulator are RND issues apart
  constexpr int RND = NT <= 8 ? NT : (NT + 1) / 2;
#pragma unroll
  for (int n0 = 0; n0 < NT; n0 += RND) {
    uint32_t bh[RND][2], bl[RND][2];
#pragma unroll
    for (int q = 0; q < RND; ++q) {
      if (n0 + q < NT) {
        float b0, b1;
        if (!TRANS) {
          const float2 b = *reinterpret_cast<const float2*>(W + (ks * ntl + nb + n0 + q) * 64 + blk_row(g) * 8 + 2 * t);
          b0 = b.x; b1 = b.y;
        } else {
          const float* p = W + ((nb + n0 + q) * ntl + ks) * 64 + g;
          b0 = p[blk_row(2 * t) * 8];
          b1 = p[blk_row(2 * t + 1) * 8];
        }
        split_tf32(b0, bh[q][0], bl[q][0]);
        split_tf32(b1, bh[q][1], bl[q][1]);
      }
    }
#pragma unroll
    for (int q = 0; q < RND; ++q) if (n0 + q < NT) mma_tf32(acc[n0 + q], al, bh[q]);
#pragma unroll
    for (int q = 0; q < RND; ++q) if (n0 + q < NT) mma_tf32(acc[n0 + q], ah, bl[q]);
#pragma unroll
    for (int q = 0; q < RND; ++q) if (n0 + q < NT) mma_tf32(acc[n0 + q], ah, bh[q]);
  }
}

template <int NT>
__device__ __forceinline__ void zero_acc(float (&acc)[NT][4]) {
#pragma unroll
  for (int n = 0; n < NT; ++n)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[n][i] = 0.f;
}

// delta rows of one layer -> shared memory: E[row = feature][timestep] fp32 (accumulator-order values; the
// thread's two rows are adjacent timesteps: one 64-bit store per feature)
template <int NT>
__device__ __forceinline__ void store_E(float* __restrict__ Erow, const float (&d)[NT][4], int warp, int lane) {
  const int g = lane >> 2, t = lane & 3;
  float* base = Erow + (2 * t) * CH_LDE + 16 * warp + 2 * g;
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    float* p = base + n * 8 * CH_LDE;
    *reinterpret_cast<float2*>(p) = make_float2(d[n][0], d[n][2]);            // feature f0
    *reinterpret_cast<float2*>(p + CH_LDE) = make_float2(d[n][1], d[n][3]);   // feature f0 + 1
  }
}
template <int NT>
__device__ __forceinline__ void to_frags(const float (&d)[NT][4], uint32_t (&hi)[NT][4], uint32_t (&lo)[NT][4]) {
#pragma unroll
  for (int n = 0; n < NT; ++n) to_frag(d[n], hi[n], lo[n]);
}

// delta_{l-1} = acc * act'(h_{l-1})
template <int ACT, int NT>
__device__ __forceinline__ void epi_delta(const float (&acc)[NT][4], const float (&h)[NT][4], float (&d)[NT][4]) {
#pragma unroll
  for (int n = 0; n < NT; ++n)
#pragma unroll
    for (int i = 0; i < 4; ++i) d[n][i] = acc[n][i] * dact_from_h<ACT>(h[n][i]);
}

// dL/dz_L of the surrogate / penalised surrogate / squared error at the head (trpo.py:43, ppo.py:47-49,
// core.py:613-617), un-normalised (1/N is applied by the slab reduce).  ho = cached head output (mean | probs |
// value) in accumulator order; auxb = this warp's rows of the side inputs.  Also the logstd gradient partials.
// The per-element terms are those of heads.cuh.  CLIP: the PPO clipped objective (clip range eps), no KL term; a
// gated row gives zeros.
template <int NT, bool CLIP>
__device__ __forceinline__ void head_grad(int head, const float (&ho)[NT][4], const float* __restrict__ auxb, int dL,
                                          const float* __restrict__ sig, const float* __restrict__ ivar, float cs,
                                          float ck, int reverse_kl, bool valid0, bool valid1, bool ok,
                                          float (&gls)[NT][2], float (&d)[NT][4], int lane, float eps) {
  const int t = lane & 3;
#pragma unroll
  for (int n = 0; n < NT; ++n)
#pragma unroll
    for (int i = 0; i < 4; ++i) d[n][i] = 0.f;
  if constexpr (CLIP) { cs = 1.f; ck = 0.f; reverse_kl = 0; }
  if (head == MRL_HEAD_GAUSS) {
    const float adv0 = valid0 ? __ldg(auxb) : 0.f, adv1 = valid1 ? __ldg(auxb + 1) : 0.f;
    float ac[NT][4], m0[NT][4], s0[NT][4];
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      ldfrag(ac[n], auxb + MRL_LDT, 8 * n + 2 * t, dL, ok);
      ldfrag(m0[n], auxb + (1 + dL) * MRL_LDT, 8 * n + 2 * t, dL, ok);
      ldfrag(s0[n], auxb + (1 + 2 * dL) * MRL_LDT, 8 * n + 2 * t, dL, ok);
    }
    float dl0 = 0.f, dl1 = 0.f;
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = 8 * n + 2 * t + (i & 1);
        if (j < dL && ok) {
          const float v = gauss_logratio(ho[n][i], ac[n][i], m0[n][i], s0[n][i], sig[j]);
          if (i < 2) dl0 += v; else dl1 += v;
        }
      }
    dl0 += __shfl_xor_sync(0xffffffffu, dl0, 1); dl0 += __shfl_xor_sync(0xffffffffu, dl0, 2);
    dl1 += __shfl_xor_sync(0xffffffffu, dl1, 1); dl1 += __shfl_xor_sync(0xffffffffu, dl1, 2);
    const float w0 = -expf(dl0) * adv0 * cs, w1 = -expf(dl1) * adv1 * cs;
    if constexpr (CLIP) {   // a gated row takes no gradient
      valid0 = valid0 && !clip_gated(expf(dl0), adv0, eps);
      valid1 = valid1 && !clip_gated(expf(dl1), adv1, eps);
    }
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = 8 * n + 2 * t + (i & 1);
        const bool valid = i < 2 ? valid0 : valid1;
        if (j < dL && valid) {
          float d_ls;
          gauss_grad(ho[n][i], ac[n][i], m0[n][i], s0[n][i], sig[j], ivar[j], i < 2 ? w0 : w1, ck, reverse_kl, d[n][i],
                     d_ls);
          gls[n][i & 1] += d_ls;
        }
      }
  } else if (head == MRL_HEAD_CAT) {
    const float adv0 = valid0 ? __ldg(auxb) : 0.f, adv1 = valid1 ? __ldg(auxb + 1) : 0.f;
    const int ai0 = ok ? (int)__ldg(auxb + MRL_LDT) : -1, ai1 = ok ? (int)__ldg(auxb + MRL_LDT + 1) : -1;
    float p0[NT][4];
#pragma unroll
    for (int n = 0; n < NT; ++n) ldfrag(p0[n], auxb + 2 * MRL_LDT, 8 * n + 2 * t, dL, ok);
    float pa0 = 0.f, pa1 = 0.f, qa0 = 0.f, qa1 = 0.f, kl0 = 0.f, kl1 = 0.f;
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = 8 * n + 2 * t + (i & 1);
        if (j < dL && ok) {
          const float p = ho[n][i], q = p0[n][i];
          if (i < 2) { if (j == ai0) { pa0 = p; qa0 = q; } } else { if (j == ai1) { pa1 = p; qa1 = q; } }
          if (reverse_kl) { const float v = p * logf(p / q); if (i < 2) kl0 += v; else kl1 += v; }
        }
      }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
      pa0 += __shfl_xor_sync(0xffffffffu, pa0, o); pa1 += __shfl_xor_sync(0xffffffffu, pa1, o);
      qa0 += __shfl_xor_sync(0xffffffffu, qa0, o); qa1 += __shfl_xor_sync(0xffffffffu, qa1, o);
      kl0 += __shfl_xor_sync(0xffffffffu, kl0, o); kl1 += __shfl_xor_sync(0xffffffffu, kl1, o);
    }
    const float w0 = valid0 ? -(pa0 / qa0) * adv0 * cs : 0.f, w1 = valid1 ? -(pa1 / qa1) * adv1 * cs : 0.f;
    if constexpr (CLIP) {
      valid0 = valid0 && !clip_gated(pa0 / qa0, adv0, eps);
      valid1 = valid1 && !clip_gated(pa1 / qa1, adv1, eps);
    }
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = 8 * n + 2 * t + (i & 1);
        const bool valid = i < 2 ? valid0 : valid1;
        if (j < dL && valid)
          d[n][i] = cat_grad(ho[n][i], p0[n][i], i < 2 ? w0 : w1, ck, i < 2 ? kl0 : kl1, j == (i < 2 ? ai0 : ai1),
                             reverse_kl);
      }
  } else {   // value head: d/dpred of (y - pred)^2
    if (t == 0) {
      if (valid0) d[0][0] = value_dpred(ho[0][0], __ldg(auxb));
      if (valid1) d[0][2] = value_dpred(ho[0][2], __ldg(auxb + 1));
    }
  }
}

// delta_{l-1} pre-activation = delta_l . W_l^T for in-blocks nb .. nb+NI-1
template <int NI, int NO>
__device__ __forceinline__ void delta_layer(float (&acc)[NI][4], const uint32_t (&dhi)[NO][4],
                                            const uint32_t (&dlo)[NO][4], const float* __restrict__ W, int nb,
                                            int lane) {
  if constexpr (NI <= 4 && NO >= 2) {   // narrow output: even / odd k-steps on separate accumulators
    float acc2[NI][4];
    zero_acc(acc2);
#pragma unroll
    for (int ks = 0; ks < NO; ++ks) {
      if (ks & 1) kstep<NI, true>(acc2, dhi[ks], dlo[ks], W, ks, nb, NO, lane);
      else kstep<NI, true>(acc, dhi[ks], dlo[ks], W, ks, nb, NO, lane);
    }
#pragma unroll
    for (int n = 0; n < NI; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[n][i] += acc2[n][i];
  } else {
#pragma unroll
    for (int ks = 0; ks < NO; ++ks) kstep<NI, true>(acc, dhi[ks], dlo[ks], W, ks, nb, NO, lane);
  }
}

// delta_1 for in-blocks nb .. nb+NH-1: bias partial sums + the tcgen05 operand DG as raw fp32 (l1_dg_offset;
// mlp_l1_tc.cu splits it into (hi, lo))
template <int ACT, int NH, int nb, int N1, int NO>
__device__ __forceinline__ void delta1_block(const uint32_t (&dhi)[NO][4], const uint32_t (&dlo)[NO][4],
                                             const float* __restrict__ W2, const float* __restrict__ hp,
                                             int d1, bool ok, float* __restrict__ gb1w, float* __restrict__ dg, int nu,
                                             int lane) {
  const int g = lane >> 2, t = lane & 3;
  float h1[NH][4];
#pragma unroll
  for (int n = 0; n < NH; ++n) ldfrag(h1[n], hp, 8 * (nb + n) + 2 * t, d1, ok);
  float acc[NH][4];
  zero_acc(acc);
  delta_layer<NH, NO>(acc, dhi, dlo, W2, nb, lane);
#pragma unroll
  for (int n = 0; n < NH; ++n) {
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = acc[n][i] * dact_from_h<ACT>(h1[n][i]);
    {  // bias gradient of layer 1: column sums over the warp's 16 timesteps into the warp's own slot
      float s0 = v[0] + v[2], s1 = v[1] + v[3];
      s0 += __shfl_xor_sync(0xffffffffu, s0, 4); s1 += __shfl_xor_sync(0xffffffffu, s1, 4);
      s0 += __shfl_xor_sync(0xffffffffu, s0, 8); s1 += __shfl_xor_sync(0xffffffffu, s1, 8);
      s0 += __shfl_xor_sync(0xffffffffu, s0, 16); s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
      if (g == 0) {
        float2* q = reinterpret_cast<float2*>(gb1w + 8 * (nb + n) + 2 * t);
        float2 c = *q;
        c.x += s0; c.y += s1;
        *q = c;
      }
    }
    if (ok && 8 * (nb + n) < nu) {
      // dg -> the warp's first timestep group.  This thread's timesteps 2g, 2g+1 are adjacent inside a group of 4:
      // one 64-bit store per feature.
      float* p0 = dg + l1_dg_offset(g >> 2, (g >> 1) & 1, 8 * (nb + n) + 2 * t, nu) + 2 * (g & 1);
#pragma unroll
      for (int b = 0; b < 2; ++b)   // features 2t, 2t+1 of the n-tile
        *reinterpret_cast<float2*>(p0 + b * 4) = make_float2(v[b], v[b + 2]);
    }
  }
}

// G[q] += h_{l-1}^T delta_l over the CH_T timesteps of the chain tile for one (m-tile, CNT n-tiles) entry.
// A = cached activations straight from L2 (k-slot t <-> timestep 2t, slot t+4 <-> 2t+1: one 64-bit load per
// row), B = delta rows from shared memory (one 64-bit load per n-tile and k-step, split here).  The accumulator
// blocks live in shared memory between chain tiles ([n-tile][lane] float4): with 12 warps a thread has 168 registers.
template <int CNT>
__device__ __forceinline__ void grad_entry(float* __restrict__ Gs, const float* __restrict__ A0, size_t tile_stride,
                                           bool ok0, bool ok1, int tiles_here, const float* __restrict__ Eb, int lane) {
  float G[CNT][4];
#pragma unroll
  for (int q = 0; q < CNT; ++q) {
    const float4 v = *reinterpret_cast<const float4*>(Gs + (q * 32 + lane) * 4);
    G[q][0] = v.x; G[q][1] = v.y; G[q][2] = v.z; G[q][3] = v.w;
  }
  float2 xa[4], xb[4];
  auto load_group = [&](int kg, float2 (&a)[4], float2 (&b)[4]) {   // 4 k-steps = 32 timesteps = half a cache tile
    const bool hk = (kg >> 1) < tiles_here;
    const float* Ap = A0 + (size_t)(kg >> 1) * tile_stride + (kg & 1) * 32;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      a[j] = (ok0 && hk) ? __ldg(reinterpret_cast<const float2*>(Ap + 8 * j)) : make_float2(0.f, 0.f);
      b[j] = (ok1 && hk) ? __ldg(reinterpret_cast<const float2*>(Ap + 8 * MRL_LDT + 8 * j)) : make_float2(0.f, 0.f);
    }
  };
  load_group(0, xa, xb);
#pragma unroll 1
  for (int kg = 0; kg < 2 * CH_TILES; ++kg) {
    float2 ca[4], cb[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { ca[j] = xa[j]; cb[j] = xb[j]; }
    if (kg + 1 < 2 * CH_TILES) load_group(kg + 1, xa, xb);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ks = 4 * kg + j;
      uint32_t ah[4], al[4];
      split_tf32(ca[j].x, ah[0], al[0]);
      split_tf32(cb[j].x, ah[1], al[1]);
      split_tf32(ca[j].y, ah[2], al[2]);
      split_tf32(cb[j].y, ah[3], al[3]);
      uint32_t bh[CNT][2], bl[CNT][2];
#pragma unroll
      for (int q = 0; q < CNT; ++q) {
        const float2 b = *reinterpret_cast<const float2*>(Eb + (size_t)q * 8 * CH_LDE + ks * 8);
        split_tf32(b.x, bh[q][0], bl[q][0]);
        split_tf32(b.y, bh[q][1], bl[q][1]);
      }
#pragma unroll
      for (int q = 0; q < CNT; ++q) mma_tf32(G[q], al, bh[q]);
#pragma unroll
      for (int q = 0; q < CNT; ++q) mma_tf32(G[q], ah, bl[q]);
#pragma unroll
      for (int q = 0; q < CNT; ++q) mma_tf32(G[q], ah, bh[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < CNT; ++q)
    *reinterpret_cast<float4*>(Gs + (q * 32 + lane) * 4) = make_float4(G[q][0], G[q][1], G[q][2], G[q][3]);
}

template <class S, int ACT, int MODE>
__global__ void __launch_bounds__(CH_THREADS, 1) chain_bwd_kernel(NetGeom g, MidBwdArgs a, ChainJobs jobs, int n_slabs,
                                                                  float clip_eps) {
  constexpr int L = S::L;
  constexpr int N1 = S::nt(1), N2 = S::nt(2), N3 = S::nt(3);
  constexpr int NL = S::nt(L);
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* ivar = Ws + S::wfloats();
  float* sig = ivar + 8 * NL;
  float* gb1s = sig + 8 * NL;                          // [warp][8 N1] layer-1 bias partials
  float* glss = gb1s + CH_WARPS * 8 * N1;              // [warp][8 NL] logstd partials
  float* Gs = glss + CH_WARPS * 8 * NL;                // weight-gradient accumulator blocks of all entries
  float* E = Gs + S::gblocks() * 128;                  // delta rows [row][CH_LDE]
  __shared__ uint64_t e_full, e_free;   // delta rows of the current chain tile: all stored / all consumed
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int gq = lane >> 2, t = lane & 3;
  const bool cat = g.head == MRL_HEAD_CAT, gauss = g.head == MRL_HEAD_GAUSS;
  if (tid == 0) {
    mbar_init(&e_full, CH_WARPS);
    mbar_init(&e_free, CH_WARPS);
    fence_barrier_init();
  }
  uint32_t tile_no = 0;                 // chain tiles processed by this CTA (barrier phase = tile_no & 1)

  // ---- weights into the 8x8-block layout, sigma, 1/sigma^2
#pragma unroll
  for (int l = 2; l <= L; ++l) {
    const int kin = 8 * S::nt(l - 1), nout = 8 * S::nt(l);
    const float* src = a.img + g.off_W[l];
    float* dw = Ws + S::woff(l);
    for (int e = tid; e < kin * nout; e += CH_THREADS) {
      const int i = e / nout, j = e - i * nout;
      const bool ok = i < g.d[l - 1] && j < g.d[l];
      const int dst = ((i >> 3) * S::nt(l) + (j >> 3)) * 64 + blk_row(j & 7) * 8 + (i & 7);
      dw[dst] = ok ? src[i * g.ldw[l] + j] : 0.f;
    }
  }
  for (int f = tid; f < 8 * NL; f += CH_THREADS) {
    const float ls = (gauss && f < g.d[L]) ? a.img[g.off_pm_logstd + f] : 0.f;
    sig[f] = expf(ls);
    ivar[f] = (gauss && f < g.d[L]) ? expf(-2.f * ls) : 0.f;
  }
  float cs = 1.f, ck = 0.f;
  if (a.coef) { cs = (float)a.coef[0]; ck = (float)a.coef[1]; }

  for (int slab = blockIdx.x; slab < n_slabs; slab += gridDim.x) {   // persistent: weights stay in shared memory
  const int t0 = slab * a.slab_tiles, t1 = min(t0 + a.slab_tiles, a.n_tiles);
  for (int i = tid; i < S::gblocks() * 128; i += CH_THREADS) Gs[i] = 0.f;
  float gls[NL][2];   // logstd gradient partials of this thread's columns (DiagGauss)
#pragma unroll
  for (int n = 0; n < NL; ++n) { gls[n][0] = 0.f; gls[n][1] = 0.f; }
  for (int i = tid; i < CH_WARPS * 8 * N1; i += CH_THREADS) gb1s[i] = 0.f;
  float gbe = 0.f;   // lane j: bias-gradient sum of delta row warp + 8 j
  __syncthreads();

  for (int ct0 = t0; ct0 < t1; ct0 += CH_TILES) {
    // ================= chain phase: this warp's 16 timesteps
    {
      const int ctile = ct0 + (warp >> 2);
      const bool ok = ctile < t1;
      const int rr = ((warp & 3) << 4) + 2 * gq;   // this thread's rows: timesteps rr and rr + 1 of the cache tile
      const long long ts = (long long)ctile * MRL_TILE + rr;
      const bool valid0 = ok && ts < a.N, valid1 = ok && ts + 1 < a.N;
      const float* cb = a.cache + (size_t)ctile * g.act_rows * MRL_LDT + rr;
      if (ct0 + CH_TILES < t1 && lane == 0) {   // pull the next chain tile into L2 while this one computes (bulk prefetch, one share per warp)
        const int nt2 = min(CH_TILES, t1 - ct0 - CH_TILES);
        const unsigned cbytes = (unsigned)(nt2 * g.act_rows * MRL_LDT * 4);
        const unsigned cchunk = (cbytes / CH_WARPS) & ~15u;
        const char* pc = reinterpret_cast<const char*>(a.cache + (size_t)(ct0 + CH_TILES) * g.act_rows * MRL_LDT) + (size_t)warp * cchunk;
        const unsigned cn = warp == CH_WARPS - 1 ? cbytes - (CH_WARPS - 1) * cchunk : cchunk;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(pc), "r"(cn) : "memory");
        const unsigned zbytes = (unsigned)(nt2 * g.naux * MRL_LDT * 4);   // side inputs: adv / actions / old probs
        const unsigned zchunk = (zbytes / CH_WARPS) & ~15u;
        const char* pz = reinterpret_cast<const char*>(a.aux + (size_t)(ct0 + CH_TILES) * g.naux * MRL_LDT) + (size_t)warp * zchunk;
        const unsigned zn = warp == CH_WARPS - 1 ? zbytes - (CH_WARPS - 1) * zchunk : zchunk;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(pz), "r"(zn) : "memory");
      }
      float h2[N2][4];
      float h3[L == 4 ? N3 : 1][4];
      float ph[NL][4];   // cached head output: mean | probs | value
#pragma unroll
      for (int n = 0; n < N2; ++n) ldfrag(h2[n], cb + g.off_act[2] * MRL_LDT, 8 * n + 2 * t, g.d[2], ok);
      if constexpr (L == 4) {
#pragma unroll
        for (int n = 0; n < N3; ++n) ldfrag(h3[n], cb + g.off_act[3] * MRL_LDT, 8 * n + 2 * t, g.d[3], ok);
      }
#pragma unroll
      for (int n = 0; n < NL; ++n) ldfrag(ph[n], cb + g.off_act[L] * MRL_LDT, 8 * n + 2 * t, g.d[L], ok);
      float dL[NL][4];   // delta_L (accumulator order)
      const float* auxb = a.aux + (size_t)ctile * g.naux * MRL_LDT + rr;
      head_grad<NL, MODE == MRL_MODE_GRAD_CLIP>(g.head, ph, auxb, g.d[L], sig, ivar, cs, ck, a.reverse_kl, valid0, valid1,
                                                ok, gls, dL, lane, clip_eps);
      // ---- reverse sweep
      bar_wait(&e_free, (tile_no & 1) ^ 1);   // the previous tile's grad phase has read its delta rows (passes at once for tile 0)
      store_E<NL>(E + (size_t)S::eoff(L) * CH_LDE, dL, warp, lane);
      uint32_t d2h[N2][4], d2l[N2][4];
      {
        uint32_t dLh[NL][4], dLl[NL][4];
        to_frags<NL>(dL, dLh, dLl);
        float acc2[N2][4];
        zero_acc(acc2);
        if constexpr (L == 3) {
          delta_layer<N2, N3>(acc2, dLh, dLl, Ws + S::woff(3), 0, lane);
        } else {
          float acc3[N3][4];
          zero_acc(acc3);
          delta_layer<N3, NL>(acc3, dLh, dLl, Ws + S::woff(4), 0, lane);
          float d3[N3][4];
          epi_delta<ACT, N3>(acc3, h3, d3);
          store_E<N3>(E + (size_t)S::eoff(3) * CH_LDE, d3, warp, lane);
          uint32_t d3h[N3][4], d3l[N3][4];
          to_frags<N3>(d3, d3h, d3l);
          delta_layer<N2, N3>(acc2, d3h, d3l, Ws + S::woff(3), 0, lane);
        }
        float d2[N2][4];
        epi_delta<ACT, N2>(acc2, h2, d2);
        store_E<N2>(E + (size_t)S::eoff(2) * CH_LDE, d2, warp, lane);
        to_frags<N2>(d2, d2h, d2l);
      }
      warp_arrive(&e_full, lane);           // this warp's delta rows are complete; delta_1 below needs nobody else
      float* dg = a.DG + l1_dg_offset(ct0 * 8 + 2 * warp, 0, 0, a.nu);
      constexpr int NA = (N1 + 1) / 2, NB = N1 - NA;
      delta1_block<ACT, NA, 0, N1, N2>(d2h, d2l, Ws + S::woff(2), cb, g.d[1], ok, gb1s + warp * 8 * N1, dg, a.nu, lane);
      if constexpr (NB > 0)
        delta1_block<ACT, NB, NA, N1, N2>(d2h, d2l, Ws + S::woff(2), cb, g.d[1], ok, gb1s + warp * 8 * N1, dg, a.nu, lane);
      if (ok && a.nu > 8 * N1) {   // the one operand n-group beyond the chain's padded width is zeros
#pragma unroll
        for (int k = 0; k < 4; ++k) dg[l1_dg_offset(k >> 1, k & 1, 8 * N1, a.nu) + lane] = 0.f;   // [tg 2][khalf 2] x 32 floats
      }
    }
    bar_wait(&e_full, tile_no & 1);
    // ================= grad phase: G_l += h_{l-1}^T delta_l over the CH_T timesteps of this chain tile
    {
      const int tiles_here = min(CH_TILES, t1 - ct0);
#pragma unroll
      for (int e = 0; e < CH_NE; ++e) {
        const ChainEntry en = jobs.e[warp][e];
        if (!en.on) continue;
        const bool ok0 = gq < en.amax, ok1 = gq + 8 < en.amax;
        const float* A0 = a.cache + ((size_t)ct0 * g.act_rows + en.arow0 + gq) * MRL_LDT + 2 * t;
        const float* Eb = E + (size_t)(en.erow0 + gq) * CH_LDE + 2 * t;
        const size_t tstride = (size_t)g.act_rows * MRL_LDT;
        switch (en.cnt) {   // warp-uniform
          case 4: grad_entry<4>(Gs + en.gsoff, A0, tstride, ok0, ok1, tiles_here, Eb, lane); break;
          case 3: grad_entry<3>(Gs + en.gsoff, A0, tstride, ok0, ok1, tiles_here, Eb, lane); break;
          case 2: grad_entry<2>(Gs + en.gsoff, A0, tstride, ok0, ok1, tiles_here, Eb, lane); break;
          default: grad_entry<1>(Gs + en.gsoff, A0, tstride, ok0, ok1, tiles_here, Eb, lane); break;
        }
      }
      // bias gradients of layers >= 2: row sums of delta
      for (int j = 0; warp + CH_WARPS * j < S::erows(); ++j) {
        const float2* p = reinterpret_cast<const float2*>(E + (size_t)(warp + CH_WARPS * j) * CH_LDE);
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < CH_T / 64; ++i) { const float2 u = p[lane + 32 * i]; s += u.x + u.y; }
        s = warp_sum(s);
        if (lane == j) gbe += s;
      }
    }
    warp_arrive(&e_free, lane);
    ++tile_no;
  }

  // ================= flush the slab partial
  float* part = a.partm + (size_t)slab * g.pmid;
#pragma unroll
  for (int e = 0; e < CH_NE; ++e) {
    const ChainEntry en = jobs.e[warp][e];
    if (!en.on) continue;
    for (int q = 0; q < en.cnt; ++q) {
      const float4 G = *reinterpret_cast<const float4*>(Gs + en.gsoff + (q * 32 + lane) * 4);
      const int n = 8 * q + 2 * t;
      float* pr = part + en.poff + n;
      if (gq < en.amax) {
        if (n < en.nmax) pr[gq * en.ldw] = G.x;
        if (n + 1 < en.nmax) pr[gq * en.ldw + 1] = G.y;
      }
      if (gq + 8 < en.amax) {
        if (n < en.nmax) pr[(gq + 8) * en.ldw] = G.z;
        if (n + 1 < en.nmax) pr[(gq + 8) * en.ldw + 1] = G.w;
      }
    }
  }
  {
    const int r = warp + CH_WARPS * lane;
    if (r < S::erows()) {
#pragma unroll
      for (int l = 2; l <= L; ++l)
        if (r >= S::eoff(l) && r < S::eoff(l + 1)) {
          const int f = r - S::eoff(l);
          if (f < g.d[l]) part[g.off_b[l] + f] = gbe;
        }
    }
  }
  __syncthreads();
  for (int f = tid; f < g.d[1]; f += CH_THREADS) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < CH_WARPS; ++w) s += gb1s[w * 8 * N1 + f];   // fixed order -> deterministic
    part[g.off_b[1] + f] = s;
  }
  if (gauss) {   // logstd gradient: this thread's column sums -> across rows (shuffles) -> across warps (fixed order)
#pragma unroll
    for (int n = 0; n < NL; ++n)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        float v = gls[n][b];
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if (gq == 0) glss[warp * 8 * NL + 8 * n + 2 * t + b] = v;
      }
    __syncthreads();
    for (int j = tid; j < g.d[L]; j += CH_THREADS) {
      float sum = 0.f;
#pragma unroll
      for (int w = 0; w < CH_WARPS; ++w) sum += glss[w * 8 * NL + j];
      part[g.off_pm_logstd + j] = sum;
    }
  } else {
    for (int j = tid; j < g.d[L]; j += CH_THREADS) part[g.off_pm_logstd + j] = 0.f;
  }
  __syncthreads();   // gb1s / glss are reused by the next slab
  }
}

// ------------------------------------------------------------------------------------ host side
// Static (layer, m-tile, n-tiles) -> warp assignment of the weight-gradient blocks: longest job first
// onto the least loaded warp that still has a free entry.
template <class S>
static bool build_jobs(const NetGeom& g, ChainJobs* jobs) {
  struct Job { int l, mt, nt0, cnt; };
  Job list[256];
  int nj = 0;
  for (int l = 2; l <= S::L; ++l) {
    const int mts = (g.d[l - 1] + 15) / 16, nts = (g.d[l] + 7) / 8;
    for (int mt = 0; mt < mts; ++mt) {
      const int groups = (nts + CH_NTJ - 1) / CH_NTJ;
      for (int gi = 0; gi < groups; ++gi) {   // spread the n-tiles evenly over the groups
        const int a0 = nts * gi / groups, a1 = nts * (gi + 1) / groups;
        if (nj == 256) return false;
        list[nj++] = {l, mt, a0, a1 - a0};
      }
    }
  }
  if (nj > CH_WARPS * CH_NE) return false;
  for (int i = 1; i < nj; ++i)
    for (int k = i; k > 0 && list[k].cnt > list[k - 1].cnt; --k) { Job tmp = list[k]; list[k] = list[k - 1]; list[k - 1] = tmp; }
  int load[CH_WARPS] = {0}, used[CH_WARPS] = {0};
  int gs = 0;
  memset(jobs, 0, sizeof(*jobs));
  for (int i = 0; i < nj; ++i) {
    int best = -1;
    for (int w = 0; w < CH_WARPS; ++w)
      if (used[w] < CH_NE && (best < 0 || load[w] < load[best])) best = w;
    if (best < 0) return false;
    const Job& j = list[i];
    ChainEntry& en = jobs->e[best][used[best]++];
    load[best] += j.cnt;
    en.on = 1;
    en.gsoff = gs;
    gs += j.cnt * 128;
    en.arow0 = g.off_act[j.l - 1] + 16 * j.mt;
    en.amax = g.d[j.l - 1] - 16 * j.mt;
    en.erow0 = S::eoff(j.l) + 8 * j.nt0;
    en.cnt = j.cnt;
    en.poff = g.off_W[j.l] + 16 * j.mt * g.ldw[j.l] + 8 * j.nt0;
    en.ldw = g.ldw[j.l];
    en.nmax = g.d[j.l] - 8 * j.nt0;
  }
  return true;
}

template <class S>
static bool shape_fits(const NetGeom& g) {
  if (g.L != S::L || g.act != MRL_ACT_TANH) return false;
  for (int l = 1; l <= S::L; ++l)
    if ((g.d[l] + 7) / 8 > S::nt(l)) return false;
  // the padded layer-1 width must cover every n-group of the layer-1 gradient operand but one
  if (l1tc_nu(g) - 8 * S::nt(1) > 8 || l1tc_nu(g) < 8 * S::nt(1)) return false;
  ChainJobs jobs;
  return build_jobs<S>(g, &jobs);
}

template <class S, int MODE>
static cudaError_t launch_shape_mode(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  ChainJobs jobs;
  if (!build_jobs<S>(g, &jobs)) return cudaErrorInvalidConfiguration;
  const size_t sm = S::smem_floats() * 4;
  {
    cudaError_t e = mrl_func_smem((const void*)chain_bwd_kernel<S, MRL_ACT_TANH, MODE>, sm);
    if (e != cudaSuccess) return e;
  }
  const int sms = mrl_sm_count();
  chain_bwd_kernel<S, MRL_ACT_TANH, MODE><<<n_slabs < sms ? n_slabs : sms, CH_THREADS, sm, st>>>(g, a, jobs, n_slabs, eps);
  return cudaGetLastError();
}
template <class S>
static cudaError_t launch_shape(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  if (a.mode == MRL_MODE_GRAD_CLIP) return launch_shape_mode<S, MRL_MODE_GRAD_CLIP>(g, a, n_slabs, st, eps);
  return launch_shape_mode<S, MRL_MODE_GRAD>(g, a, n_slabs, st, eps);
}

typedef ChainShape<3, 8, 8, 1, 0> ShapeA;     // 64-64 hidden, <= 8 outputs  (Hopper, Walker2d, CartPole, value nets)
typedef ChainShape<3, 8, 8, 3, 0> ShapeB;     // 64-64 hidden, <= 24 outputs (18-action Categorical)
typedef ChainShape<4, 13, 7, 4, 3> ShapeC;    // 100-50-25 hidden, <= 24 outputs (Humanoid policy and value nets)

// 0 = not supported (use the job-list kernel of mlp_mid.cu), else the shape id
int chain_bwd_shape(const NetGeom& g) {
  if (shape_fits<ShapeA>(g)) return 1;
  if (shape_fits<ShapeB>(g)) return 2;
  if (shape_fits<ShapeC>(g)) return 3;
  return 0;
}

cudaError_t launch_chain_backward(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps) {
  if (a.mode == MRL_MODE_FVP) return cudaErrorInvalidValue;   // the chain computes gradients only
  switch (chain_bwd_shape(g)) {
    case 1: return launch_shape<ShapeA>(g, a, n_slabs, st, clip_eps);
    case 2: return launch_shape<ShapeB>(g, a, n_slabs, st, clip_eps);
    case 3: return launch_shape<ShapeC>(g, a, n_slabs, st, clip_eps);
    default: return cudaErrorInvalidConfiguration;
  }
}

// ====================================================================================================
// Forward chain: h1 = act(Z1 + b1), ..., head -> surr / kl / ent (or squared error) sums, activation cache,
// row-major head output (trpo.py:37-42,60-63; core.py:339-365,402-438,613-617).  Same per-warp register
// chain as above (16 timesteps per warp, no block barriers inside a slab), 8 warps = 128 timesteps per pass,
// 2 CTAs per SM.

__device__ __forceinline__ void st_cfrag(float* __restrict__ p, const float (&v)[4], int f0, int dmax, bool ok) {
  if (ok && f0 < dmax) *reinterpret_cast<float2*>(p + f0 * MRL_LDT) = make_float2(v[0], v[2]);
  if (ok && f0 + 1 < dmax) *reinterpret_cast<float2*>(p + (f0 + 1) * MRL_LDT) = make_float2(v[1], v[3]);
}
// hidden-layer epilogue: h = act(acc + b) -> cache, fragments of the next GEMM
template <int ACT, int NT>
__device__ __forceinline__ void epi_hidden(const float (&acc)[NT][4], const float* __restrict__ bl, float* __restrict__ cp,
                                           int dmax, bool ok, uint32_t (&hi)[NT][4], uint32_t (&lo)[NT][4], int lane) {
  const int t = lane & 3;
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    const float2 b = *reinterpret_cast<const float2*>(bl + 8 * n + 2 * t);
    float v[4];
    v[0] = act_fn<ACT>(acc[n][0] + b.x); v[1] = act_fn<ACT>(acc[n][1] + b.y);
    v[2] = act_fn<ACT>(acc[n][2] + b.x); v[3] = act_fn<ACT>(acc[n][3] + b.y);
    if (cp) st_cfrag(cp, v, 8 * n + 2 * t, dmax, ok);
    to_frag(v, hi[n], lo[n]);
  }
}
template <int NI, int NO>
__device__ __forceinline__ void fwd_layer(float (&acc)[NO][4], const uint32_t (&ahi)[NI][4], const uint32_t (&alo)[NI][4],
                                          const float* __restrict__ W, int lane) {
#pragma unroll
  for (int ks = 0; ks < NI; ++ks) kstep<NO, false>(acc, ahi[ks], alo[ks], W, ks, 0, NO, lane);
}

// head of one warp's 16 timesteps: out = acc + b_L -> mean | softmax | value; losses; cache; row-major output
// CLIP: surr takes the clipped objective (clip range eps), s_clip counts the rows outside the clip range
template <int NT, bool CLIP>
__device__ __forceinline__ void head_forward(int head, float (&o)[NT][4], const float* __restrict__ bl,
                                             const float* __restrict__ auxb, int dL, const float* __restrict__ sig,
                                             float ent_row, int reverse_kl, bool valid0, bool valid1, bool ok,
                                             double& s_surr, double& s_kl, double& s_ent, int lane, float eps,
                                             double& s_clip) {
  const int t = lane & 3;
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    const float2 b = *reinterpret_cast<const float2*>(bl + 8 * n + 2 * t);
    o[n][0] += b.x; o[n][1] += b.y; o[n][2] += b.x; o[n][3] += b.y;
  }
  if (head == MRL_HEAD_GAUSS) {
    if (auxb == nullptr) return;
    float dl0 = 0.f, dl1 = 0.f, kl0 = 0.f, kl1 = 0.f;
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      float ac[4], m0[4], s0[4];
      ldfrag(ac, auxb + MRL_LDT, 8 * n + 2 * t, dL, ok);
      ldfrag(m0, auxb + (1 + dL) * MRL_LDT, 8 * n + 2 * t, dL, ok);
      ldfrag(s0, auxb + (1 + 2 * dL) * MRL_LDT, 8 * n + 2 * t, dL, ok);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = 8 * n + 2 * t + (i & 1);
        if (j < dL && ok) {
          const float dlv = gauss_logratio(o[n][i], ac[i], m0[i], s0[i], sig[j]);
          const float klv = gauss_kl(o[n][i], m0[i], s0[i], sig[j], reverse_kl);
          if (i < 2) { dl0 += dlv; kl0 += klv; } else { dl1 += dlv; kl1 += klv; }
        }
      }
    }
#pragma unroll
    for (int q = 1; q <= 2; q <<= 1) {
      dl0 += __shfl_xor_sync(0xffffffffu, dl0, q); dl1 += __shfl_xor_sync(0xffffffffu, dl1, q);
      kl0 += __shfl_xor_sync(0xffffffffu, kl0, q); kl1 += __shfl_xor_sync(0xffffffffu, kl1, q);
    }
    if (t == 0) {
      if constexpr (CLIP) {
        if (valid0) { clip_row(expf(dl0), __ldg(auxb), eps, s_surr, s_clip); s_kl += (double)kl0; s_ent += (double)ent_row; }
        if (valid1) { clip_row(expf(dl1), __ldg(auxb + 1), eps, s_surr, s_clip); s_kl += (double)kl1; s_ent += (double)ent_row; }
      } else {
        if (valid0) { s_surr += (double)(expf(dl0) * __ldg(auxb)); s_kl += (double)kl0; s_ent += (double)ent_row; }
        if (valid1) { s_surr += (double)(expf(dl1) * __ldg(auxb + 1)); s_kl += (double)kl1; s_ent += (double)ent_row; }
      }
    }
  } else if (head == MRL_HEAD_CAT) {
    float m0_ = -INFINITY, m1_ = -INFINITY;
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (8 * n + 2 * t + (i & 1) < dL) { if (i < 2) m0_ = fmaxf(m0_, o[n][i]); else m1_ = fmaxf(m1_, o[n][i]); }
#pragma unroll
    for (int q = 1; q <= 2; q <<= 1) {
      m0_ = fmaxf(m0_, __shfl_xor_sync(0xffffffffu, m0_, q)); m1_ = fmaxf(m1_, __shfl_xor_sync(0xffffffffu, m1_, q));
    }
    float z0 = 0.f, z1 = 0.f;
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool in = 8 * n + 2 * t + (i & 1) < dL;
        const float e = in ? expf(o[n][i] - (i < 2 ? m0_ : m1_)) : 0.f;
        o[n][i] = e;
        if (i < 2) z0 += e; else z1 += e;
      }
#pragma unroll
    for (int q = 1; q <= 2; q <<= 1) { z0 += __shfl_xor_sync(0xffffffffu, z0, q); z1 += __shfl_xor_sync(0xffffffffu, z1, q); }
    const float i0 = 1.f / z0, i1 = 1.f / z1;
#pragma unroll
    for (int n = 0; n < NT; ++n) { o[n][0] *= i0; o[n][1] *= i0; o[n][2] *= i1; o[n][3] *= i1; }
    if (auxb == nullptr) return;
    const int ai0 = ok ? (int)__ldg(auxb + MRL_LDT) : -1, ai1 = ok ? (int)__ldg(auxb + MRL_LDT + 1) : -1;
    float pa0 = 0.f, pa1 = 0.f, qa0 = 0.f, qa1 = 0.f, kl0 = 0.f, kl1 = 0.f, en0 = 0.f, en1 = 0.f;
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      float p0[4];
      ldfrag(p0, auxb + 2 * MRL_LDT, 8 * n + 2 * t, dL, ok);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = 8 * n + 2 * t + (i & 1);
        if (j < dL && ok) {
          const float p = o[n][i];
          const float klv = cat_kl(p, p0[i], reverse_kl);
          const float env = -p * logf(p);
          if (i < 2) { kl0 += klv; en0 += env; if (j == ai0) { pa0 = p; qa0 = p0[i]; } }
          else { kl1 += klv; en1 += env; if (j == ai1) { pa1 = p; qa1 = p0[i]; } }
        }
      }
    }
#pragma unroll
    for (int q = 1; q <= 2; q <<= 1) {
      pa0 += __shfl_xor_sync(0xffffffffu, pa0, q); pa1 += __shfl_xor_sync(0xffffffffu, pa1, q);
      qa0 += __shfl_xor_sync(0xffffffffu, qa0, q); qa1 += __shfl_xor_sync(0xffffffffu, qa1, q);
      kl0 += __shfl_xor_sync(0xffffffffu, kl0, q); kl1 += __shfl_xor_sync(0xffffffffu, kl1, q);
      en0 += __shfl_xor_sync(0xffffffffu, en0, q); en1 += __shfl_xor_sync(0xffffffffu, en1, q);
    }
    if (t == 0) {
      if constexpr (CLIP) {
        if (valid0) { clip_row(pa0 / qa0, __ldg(auxb), eps, s_surr, s_clip); s_kl += (double)kl0; s_ent += (double)en0; }
        if (valid1) { clip_row(pa1 / qa1, __ldg(auxb + 1), eps, s_surr, s_clip); s_kl += (double)kl1; s_ent += (double)en1; }
      } else {
        if (valid0) { s_surr += (double)((pa0 / qa0) * __ldg(auxb)); s_kl += (double)kl0; s_ent += (double)en0; }
        if (valid1) { s_surr += (double)((pa1 / qa1) * __ldg(auxb + 1)); s_kl += (double)kl1; s_ent += (double)en1; }
      }
    }
  } else {   // value head: squared error against the target row
    if (auxb != nullptr && t == 0) {
      if (valid0) s_surr += value_sqerr(__ldg(auxb), o[0][0]);
      if (valid1) s_surr += value_sqerr(__ldg(auxb + 1), o[0][2]);
    }
  }
}

template <class S, int ACT, bool CLIP>
__global__ void __launch_bounds__(FW_THREADS, 2) chain_fwd_kernel(NetGeom g, MidFwdArgs a, int n_slabs, float clip_eps) {
  constexpr int L = S::L;
  constexpr int N1 = S::nt(1), N2 = S::nt(2), N3 = S::nt(3);
  constexpr int NL = S::nt(L);
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* bs = Ws + S::wfloats();      // biases of layers 1..L (vboff layout)
  float* sig = bs + S::vbfloats();
  __shared__ double red[32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int gq = lane >> 2, t = lane & 3;
  const bool gauss = g.head == MRL_HEAD_GAUSS;

#pragma unroll
  for (int l = 2; l <= L; ++l) {
    const int kin = 8 * S::nt(l - 1), nout = 8 * S::nt(l);
    const float* src = a.img + g.off_W[l];
    float* dw = Ws + S::woff(l);
    for (int e = tid; e < kin * nout; e += FW_THREADS) {
      const int i = e / nout, j = e - i * nout;
      const bool ok = i < g.d[l - 1] && j < g.d[l];
      dw[((i >> 3) * S::nt(l) + (j >> 3)) * 64 + blk_row(j & 7) * 8 + (i & 7)] = ok ? src[i * g.ldw[l] + j] : 0.f;
    }
  }
#pragma unroll
  for (int l = 1; l <= L; ++l)
    for (int f = tid; f < 8 * S::nt(l); f += FW_THREADS) bs[S::vboff(l) + f] = f < g.d[l] ? a.img[g.off_b[l] + f] : 0.f;
  float ent_row = 0.f;     // DiagGauss entropy is the same for every row: sum log sigma + d/2 log(2 pi e)
  {
    float sls = 0.f;
    for (int j = 0; j < g.d[L] && gauss; ++j) sls += a.img[g.off_pm_logstd + j];
    ent_row = sls + 0.5f * MRL_LOG_2PIE * g.d[L];
  }
  for (int f = tid; f < 8 * NL; f += FW_THREADS) sig[f] = (gauss && f < g.d[L]) ? expf(a.img[g.off_pm_logstd + f]) : 1.f;
  __syncthreads();

  for (int slab = blockIdx.x; slab < n_slabs; slab += gridDim.x) {
    const int t0 = slab * a.slab_tiles, t1 = min(t0 + a.slab_tiles, a.n_tiles);
    double s_surr = 0.0, s_kl = 0.0, s_ent = 0.0, s_clip = 0.0;
    for (int ct0 = t0; ct0 < t1; ct0 += 2) {
      const int ctile = ct0 + (warp >> 2);
      const bool ok = ctile < t1;
      const int rr = ((warp & 3) << 4) + 2 * gq;   // this thread's rows: timesteps rr and rr + 1 of the cache tile
      const long long ts = (long long)ctile * MRL_TILE + rr;
      const bool valid0 = ok && ts < a.N, valid1 = ok && ts + 1 < a.N;
      const float* zb = a.Zt + (size_t)ctile * g.d[1] * MRL_LDT + rr;
      float* cb = a.cache ? a.cache + (size_t)ctile * g.act_rows * MRL_LDT + rr : nullptr;
      const float* auxb = a.aux ? a.aux + (size_t)ctile * g.naux * MRL_LDT + rr : nullptr;
      if (ct0 + 2 < t1 && lane == 0) {   // next chain tile's layer-1 pre-activations (and side inputs) into L2
        const int nt2 = min(2, t1 - ct0 - 2);
        const unsigned zbytes = (unsigned)(nt2 * g.d[1] * MRL_LDT * 4), zchunk = (zbytes / FW_WARPS) & ~15u;
        const char* pz = reinterpret_cast<const char*>(a.Zt + (size_t)(ct0 + 2) * g.d[1] * MRL_LDT) + (size_t)warp * zchunk;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(pz), "r"(warp == FW_WARPS - 1 ? zbytes - (FW_WARPS - 1) * zchunk : zchunk) : "memory");
        if (a.aux) {
          const unsigned xbytes = (unsigned)(nt2 * g.naux * MRL_LDT * 4), xchunk = (xbytes / FW_WARPS) & ~15u;
          const char* px = reinterpret_cast<const char*>(a.aux + (size_t)(ct0 + 2) * g.naux * MRL_LDT) + (size_t)warp * xchunk;
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(px), "r"(warp == FW_WARPS - 1 ? xbytes - (FW_WARPS - 1) * xchunk : xchunk) : "memory");
        }
      }
      // ---- layer 1 activation streamed per k-step into the layer-2 GEMM
      float acc2[N2][4];
      zero_acc(acc2);
      {
        float zc[4], z1[4];
        ldfrag(zc, zb, 2 * t, g.d[1], ok);
        ldfrag(z1, zb, 8 + 2 * t, g.d[1], ok && N1 > 1);
#pragma unroll 1
        for (int ks = 0; ks < N1; ++ks) {
          float zn[4];
          ldfrag(zn, zb, 8 * (ks + 2) + 2 * t, g.d[1], ok && ks + 2 < N1);
          const float2 b = *reinterpret_cast<const float2*>(bs + S::vboff(1) + 8 * ks + 2 * t);
          float h[4];
          if (L > 1) {
            h[0] = act_fn<ACT>(zc[0] + b.x); h[1] = act_fn<ACT>(zc[1] + b.y);
            h[2] = act_fn<ACT>(zc[2] + b.x); h[3] = act_fn<ACT>(zc[3] + b.y);
          }
          if (cb) st_cfrag(cb, h, 8 * ks + 2 * t, g.d[1], ok);
          uint32_t ah[4], al[4];
          to_frag(h, ah, al);
          kstep<N2, false>(acc2, ah, al, Ws + S::woff(2), ks, 0, N2, lane);
#pragma unroll
          for (int i = 0; i < 4; ++i) { zc[i] = z1[i]; z1[i] = zn[i]; }
        }
      }
      float o[NL][4];
      if constexpr (L == 3) {
        uint32_t h2h[N2][4], h2l[N2][4];
        epi_hidden<ACT, N2>(acc2, bs + S::vboff(2), cb ? cb + g.off_act[2] * MRL_LDT : nullptr, g.d[2], ok, h2h, h2l, lane);
        zero_acc(o);
        fwd_layer<N2, NL>(o, h2h, h2l, Ws + S::woff(3), lane);
      } else {
        uint32_t h2h[N2][4], h2l[N2][4];
        epi_hidden<ACT, N2>(acc2, bs + S::vboff(2), cb ? cb + g.off_act[2] * MRL_LDT : nullptr, g.d[2], ok, h2h, h2l, lane);
        float acc3[N3][4];
        zero_acc(acc3);
        fwd_layer<N2, N3>(acc3, h2h, h2l, Ws + S::woff(3), lane);
        uint32_t h3h[N3][4], h3l[N3][4];
        epi_hidden<ACT, N3>(acc3, bs + S::vboff(3), cb ? cb + g.off_act[3] * MRL_LDT : nullptr, g.d[3], ok, h3h, h3l, lane);
        zero_acc(o);
        fwd_layer<N3, NL>(o, h3h, h3l, Ws + S::woff(4), lane);
      }
      head_forward<NL, CLIP>(g.head, o, bs + S::vboff(L), auxb, g.d[L], sig, ent_row, a.reverse_kl, valid0, valid1, ok,
                             s_surr, s_kl, s_ent, lane, clip_eps, s_clip);
      if (cb) {
#pragma unroll
        for (int n = 0; n < NL; ++n) st_cfrag(cb + g.off_act[L] * MRL_LDT, o[n], 8 * n + 2 * t, g.d[L], ok);
      }
      if (a.head_out) {
        const int dL = g.d[L];
#pragma unroll
        for (int n = 0; n < NL; ++n)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int j = 8 * n + 2 * t + (i & 1);
            if (j < dL && (i < 2 ? valid0 : valid1)) a.head_out[(size_t)(ts + (i < 2 ? 0 : 1)) * dL + j] = o[n][i];
          }
      }
    }
    if (a.loss_part) {
      double v0 = block_sum(s_surr, red);
      double v1 = block_sum(s_kl, red);
      double v2 = block_sum(s_ent, red);
      double v3 = 0.0;
      if constexpr (CLIP) v3 = block_sum(s_clip, red);
      if (tid == 0) {
        double* op = a.loss_part + (size_t)slab * 4;
        op[0] = v0; op[1] = v1; op[2] = v2; op[3] = v3;
      }
    }
  }
}

template <class S>
static bool fwd_shape_fits(const NetGeom& g) {
  if (g.L != S::L || g.act != MRL_ACT_TANH) return false;
  for (int l = 1; l <= S::L; ++l)
    if ((g.d[l] + 7) / 8 > S::nt(l)) return false;
  return true;
}
template <class S, bool CLIP>
static cudaError_t launch_fwd_shape_clip(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  const size_t sm = ((size_t)S::wfloats() + S::vbfloats() + 8 * S::nt(S::L)) * 4;
  {
    cudaError_t e = mrl_func_smem((const void*)chain_fwd_kernel<S, MRL_ACT_TANH, CLIP>, sm);
    if (e != cudaSuccess) return e;
  }
  const int sms = mrl_sm_count();
  chain_fwd_kernel<S, MRL_ACT_TANH, CLIP><<<n_slabs < 2 * sms ? n_slabs : 2 * sms, FW_THREADS, sm, st>>>(g, a, n_slabs, eps);   // 2 CTAs per SM
  return cudaGetLastError();
}
template <class S>
static cudaError_t launch_fwd_shape(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  if (eps > 0.f && g.head != MRL_HEAD_VALUE) return launch_fwd_shape_clip<S, true>(g, a, n_slabs, st, eps);
  return launch_fwd_shape_clip<S, false>(g, a, n_slabs, st, eps);
}
int chain_fwd_shape(const NetGeom& g) {
  if (fwd_shape_fits<ShapeA>(g)) return 1;
  if (fwd_shape_fits<ShapeB>(g)) return 2;
  if (fwd_shape_fits<ShapeC>(g)) return 3;
  return 0;
}
cudaError_t launch_chain_forward(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps) {
  switch (chain_fwd_shape(g)) {
    case 1: return launch_fwd_shape<ShapeA>(g, a, n_slabs, st, clip_eps);
    case 2: return launch_fwd_shape<ShapeB>(g, a, n_slabs, st, clip_eps);
    case 3: return launch_fwd_shape<ShapeC>(g, a, n_slabs, st, clip_eps);
    default: return cudaErrorInvalidConfiguration;
  }
}
