// Fused per-tile MLP chain for layers >= 2, the distribution heads, and the reverse sweeps.
//
// One CTA owns a slab of up to 16 tiles (1024 timesteps).  All weights of layers 2..L (plus
// transposes and the tangent's weights for the R-op) live in shared memory for the CTA's
// lifetime; per tile the activations of all layers are held feature-major in shared memory
// ([feature][68]); every GEMM is a set of 32x16 warp tiles computed with mma.sync TF32 in
// split precision (3xTF32, FP32-class accuracy), and weight gradients accumulate in shared
// memory until the slab is flushed as one fp32 partial.
//
//   mid_forward_kernel : h1 = act(Z1+b1), ..., head -> surr/kl/ent (or MSE) sums, activation cache
//                        trpo.py:37-42,60-63 ; core.py:339-365,402-438 ; core.py:613-617
//                        <CLIP>: the PPO clipped objective for surr, the clipped-row count in loss slot 3
//   mid_backward_kernel<GRAD> : dL/dz_L from the head, reverse sweep         trpo.py:43, ppo.py:47-49
//   mid_backward_kernel<GRAD_CLIP> : the same for the PPO clipped objective
//   mid_backward_kernel<FVP>  : R-forward (Pearlmutter), Fisher metric, reverse sweep  trpo.py:45-58
#include "common.cuh"
#include "heads.cuh"
#include "kernels.h"
#include "mma_tf32.cuh"

#ifndef MRL_BWD_THREADS
#define MRL_BWD_THREADS 512   // reverse-sweep kernel: 16 warps hide the LDS/MMA latencies of the small tiles
#endif

struct Lane {
  int warp, lane, rg, cg;
  __device__ Lane() {
    warp = threadIdx.x >> 5;
    lane = threadIdx.x & 31;
    rg = lane & 7;
    cg = lane >> 3;
  }
};

// ---- warp-level tensor-core GEMM pieces (mma.sync m16n8k8 TF32, split-precision 3xTF32) ----------
// The fused chain cannot feed tcgen05: its operands would need the UMMA core-matrix layout in shared
// memory with separate hi/lo copies of every activation and weight (2x the 219 KB this kernel already
// uses at Humanoid sizes).  mma.sync takes fragments from registers, so the split x = hi + lo is done
// on the fly after a plain LDS and the shared-memory layouts stay as they are.  hi = rna_tf32(x),
// lo = x - hi (exact in fp32; the tensor core drops its low 13 bits, a 2^-21 relative effect);
// D += lo.hi + hi.lo + hi.hi keeps FP32-class accuracy (north_star: 1e-5) at 1/3 of the TF32 rate,
// with ~3x fewer issued instructions than the FFMA formulation (the chain is issue-bound).
// One warp job of  OUT[c][r] = epi(c, r, sum_k A1[k][r] B1[k][c] (+ sum_k A2[k][r] B2[k][c])).
// job -> (16*MT) rows x 16 cols; epi(c, r, value) is called once per output element.  MT = 1 doubles
// the number of jobs of a phase that would otherwise leave warps idle.
template <int MT, class Epi>
__device__ __forceinline__ void fwd_job(int job, const Lane& ln, const float* A1, const float* B1, int K1,
                                        const float* A2, const float* B2, int K2, int ldb, int n_out,
                                        Epi epi) {
  constexpr int RB = MRL_TILE / (16 * MT);
  const int r0 = (job % RB) * 16 * MT, c0 = (job / RB) * 16;
  float acc[MT][2][4];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;
  mma_fwd_acc<MT>(acc, A1, B1, K1, ldb, r0, c0, ln.lane);
  if (A2 != nullptr) mma_fwd_acc<MT>(acc, A2, B2, K2, ldb, r0, c0, ln.lane);
  const int g = ln.lane >> 2, t = ln.lane & 3;
#pragma unroll
  for (int mi = 0; mi < MT; ++mi)
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) {
      const int r = r0 + 16 * mi + g, c = c0 + 8 * ni + 2 * t;
      if (c < n_out) { epi(c, r, acc[mi][ni][0]); epi(c, r + 8, acc[mi][ni][2]); }
      if (c + 1 < n_out) { epi(c + 1, r, acc[mi][ni][1]); epi(c + 1, r + 8, acc[mi][ni][3]); }
    }
}
__device__ __forceinline__ int fwd_jobs(int n_out, int mt) { return (MRL_TILE / (16 * mt)) * ((n_out + 15) >> 4); }
// 16-row jobs when 32-row jobs would not give every warp work
__device__ __forceinline__ int pick_mt(int n_out, int nwarps) { return fwd_jobs(n_out, 2) < nwarps ? 1 : 2; }

// One warp job of  G[m][n] += sum_r A[m][r] * D[n][r]   ((16*MT) m x 16 n per job, K = the 64 timesteps)
template <int MT>
__device__ __forceinline__ void grad_job(int job, int n_nblk, const Lane& ln, const float* __restrict__ A,
                                         int M, const float* __restrict__ D, int Nn, float* G, int ldg) {
  const int m0 = (job / n_nblk) * 16 * MT, n0 = (job % n_nblk) * 16;
  const int g = ln.lane >> 2, t = ln.lane & 3;
  const float* ap[2 * MT];   // rows m0+g, +8, ... (clamped; out-of-range rows are never stored)
  const float* dp[2];        // rows n0+g, +8
#pragma unroll
  for (int q = 0; q < 2 * MT; ++q) ap[q] = A + min(m0 + g + 8 * q, M - 1) * MRL_LDT + t;
#pragma unroll
  for (int q = 0; q < 2; ++q) dp[q] = D + min(n0 + g + 8 * q, Nn - 1) * MRL_LDT + t;
  float acc[MT][2][4];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;
#pragma unroll 2
  for (int k0 = 0; k0 < MRL_TILE; k0 += 8) {
    uint32_t bh[2][2], bl[2][2];
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) {
      split_tf32(dp[ni][k0], bh[ni][0], bl[ni][0]);
      split_tf32(dp[ni][k0 + 4], bh[ni][1], bl[ni][1]);
    }
    uint32_t ah[MT][4], al[MT][4];
#pragma unroll
    for (int mi = 0; mi < MT; ++mi) {
      split_tf32(ap[2 * mi][k0], ah[mi][0], al[mi][0]);
      split_tf32(ap[2 * mi + 1][k0], ah[mi][1], al[mi][1]);
      split_tf32(ap[2 * mi][k0 + 4], ah[mi][2], al[mi][2]);
      split_tf32(ap[2 * mi + 1][k0 + 4], ah[mi][3], al[mi][3]);
    }
    mma3_tiles<MT>(acc, ah, al, bh, bl);
  }
#pragma unroll
  for (int mi = 0; mi < MT; ++mi)
#pragma unroll
    for (int ni = 0; ni < 2; ++ni) {
      const int m = m0 + 16 * mi + g, n = n0 + 8 * ni + 2 * t;
      if (m < M) {
        if (n < Nn) G[m * ldg + n] += acc[mi][ni][0];
        if (n + 1 < Nn) G[m * ldg + n + 1] += acc[mi][ni][1];
      }
      if (m + 8 < M) {
        if (n < Nn) G[(m + 8) * ldg + n] += acc[mi][ni][2];
        if (n + 1 < Nn) G[(m + 8) * ldg + n + 1] += acc[mi][ni][3];
      }
    }
}

// gb[j] += sum_r D[j][r] for 8 features per job
__device__ __forceinline__ void bias_job(int job, const Lane& ln, const float* __restrict__ D, int Nn, float* gb) {
  for (int q = 0; q < 8; ++q) {
    const int j = job * 8 + q;
    if (j >= Nn) break;
    float s = D[j * MRL_LDT + ln.lane] + D[j * MRL_LDT + 32 + ln.lane];
    s = warp_sum(s);
    if (ln.lane == 0) gb[j] += s;
  }
}

// pull the next tile's lines into L2 while this tile computes (the working set is far larger than L2)
__device__ __forceinline__ void prefetch_l2(const float* src, int nfloats) {
  const char* p = reinterpret_cast<const char*>(src);
  for (int off = threadIdx.x * 128; off < nfloats * 4; off += blockDim.x * 128)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p + off));
}

__device__ __forceinline__ void copy_f4(float* dst, const float* src, int nfloats) {
  const float4* s = reinterpret_cast<const float4*>(src);
  float4* d = reinterpret_cast<float4*>(dst);
  for (int i = threadIdx.x; i < (nfloats >> 2); i += blockDim.x) d[i] = s[i];
}

// =====================================================================================
template <int HEAD, int ACT, bool CLIP>
__global__ void __launch_bounds__(MRL_MID_THREADS, 1) mid_forward_kernel(NetGeom g, MidFwdArgs a, float clip_eps) {
  extern __shared__ __align__(16) float smem[];
  float* img = smem;
  float* act = img + g.bw_floats;
  __shared__ double red[32];
  __shared__ float sig[MRL_MAX_DOUT], logsig[MRL_MAX_DOUT];
  const Lane ln;
  const int tid = threadIdx.x;
  const int L = g.L, dL = g.d[L];
  const int slab = blockIdx.x;
  const int t0 = slab * a.slab_tiles, t1 = min(t0 + a.slab_tiles, a.n_tiles);

  copy_f4(img, a.img, g.bw_floats);
  __syncthreads();
  if (HEAD == MRL_HEAD_GAUSS && tid < dL) {
    const float ls = img[g.off_pm_logstd + tid];
    logsig[tid] = ls;
    sig[tid] = expf(ls);
  }
  double s_surr = 0.0, s_kl = 0.0, s_ent = 0.0, s_clip = 0.0;
  float* headbuf = act + g.off_act[L] * MRL_LDT;

  for (int tile = t0; tile < t1; ++tile) {
    const int nvalid = (int)min((long long)MRL_TILE, a.N - (long long)tile * MRL_TILE);
    {  // h1 = act(Z1 + b1)   (or the head pre-activation when L == 1)
      const float4* zs = reinterpret_cast<const float4*>(a.Zt + (size_t)tile * g.d[1] * MRL_LDT);
      float4* dst = reinterpret_cast<float4*>(act);
      const float* b1 = img + g.off_b[1];
      const int n4 = g.d[1] * (MRL_LDT / 4);
      for (int i = tid; i < n4; i += MRL_MID_THREADS) {
        float4 z = zs[i];
        const float b = b1[i / (MRL_LDT / 4)];
        if (L > 1) {
          z.x = act_fn<ACT>(z.x + b); z.y = act_fn<ACT>(z.y + b);
          z.z = act_fn<ACT>(z.z + b); z.w = act_fn<ACT>(z.w + b);
        } else {
          z.x += b; z.y += b; z.z += b; z.w += b;
        }
        dst[i] = z;
      }
    }
    __syncthreads();
    for (int l = 2; l <= L; ++l) {
      const float* A = act + g.off_act[l - 1] * MRL_LDT;
      float* O = act + g.off_act[l] * MRL_LDT;
      const float* W = img + g.off_W[l];
      const float* b = img + g.off_b[l];
      const bool last = (l == L);
      auto epi = [&](int c, int r, float v) {
        v += b[c];
        O[c * MRL_LDT + r] = last ? v : act_fn<ACT>(v);
      };
      const int mt = pick_mt(g.d[l], MRL_MID_THREADS / 32);
      const int nj = fwd_jobs(g.d[l], mt);
      for (int job = ln.warp; job < nj; job += MRL_MID_THREADS / 32) {
        if (mt == 1) fwd_job<1>(job, ln, A, W, g.d[l - 1], nullptr, nullptr, 0, g.ldw[l], g.d[l], epi);
        else fwd_job<2>(job, ln, A, W, g.d[l - 1], nullptr, nullptr, 0, g.ldw[l], g.d[l], epi);
      }
      __syncthreads();
    }
    // ---- head: one thread per timestep
    if (tid < MRL_TILE) {
      const float* aux = a.aux ? a.aux + (size_t)tile * g.naux * MRL_LDT + tid : nullptr;
      head_fwd_row<HEAD, CLIP>(headbuf, aux, tid, dL, tid < nvalid, a.reverse_kl, sig, logsig, s_surr, s_kl, s_ent,
                               clip_eps, s_clip);
    }
    __syncthreads();
    if (a.cache) copy_f4(a.cache + (size_t)tile * g.act_rows * MRL_LDT, act, g.act_rows * MRL_LDT);
    if (a.head_out) {
      for (int i = tid; i < MRL_TILE * dL; i += MRL_MID_THREADS) {
        const int r = i / dL, j = i % dL;
        if (r < nvalid) a.head_out[((size_t)tile * MRL_TILE + r) * dL + j] = headbuf[j * MRL_LDT + r];
      }
    }
    __syncthreads();
  }
  if (a.loss_part) {
    double v0 = block_sum(s_surr, red);
    double v1 = block_sum(s_kl, red);
    double v2 = block_sum(s_ent, red);
    double v3 = 0.0;
    if constexpr (CLIP) v3 = block_sum(s_clip, red);
    if (tid == 0) {
      double* o = a.loss_part + (size_t)slab * 4;
      o[0] = v0; o[1] = v1; o[2] = v2; o[3] = v3;
    }
  }
}

// =====================================================================================
template <int HEAD, int ACT, int MODE>
__global__ void __launch_bounds__(MRL_BWD_THREADS, 1) mid_backward_kernel(NetGeom g, MidBwdArgs a, float clip_eps) {
  extern __shared__ __align__(16) float smem[];
  float* img = smem;
  float* imgv = img + g.img_floats;
  float* G = imgv + (MODE == MRL_MODE_FVP ? g.bw_floats : 0);
  float* GL = G + g.bw_floats;
  const int gl_floats = (MODE != MRL_MODE_FVP && HEAD == MRL_HEAD_GAUSS) ? g.d[g.L] * MRL_TILE : 0;
  float* H = GL + gl_floats;
  float* E = H + g.act_rows * MRL_LDT;
  __shared__ float sig[MRL_MAX_DOUT], ivar[MRL_MAX_DOUT];
  const Lane ln;
  const int tid = threadIdx.x;
  const int L = g.L, dL = g.d[L];
  const int slab = blockIdx.x;
  const int t0 = slab * a.slab_tiles, t1 = min(t0 + a.slab_tiles, a.n_tiles);
  constexpr int NW = MRL_BWD_THREADS / 32;

  copy_f4(img, a.img, g.img_floats);
  if (MODE == MRL_MODE_FVP) copy_f4(imgv, a.imgv, g.bw_floats);
  for (int i = tid; i < g.bw_floats + gl_floats; i += MRL_BWD_THREADS) G[i] = 0.f;
  __syncthreads();
  if (HEAD == MRL_HEAD_GAUSS && tid < dL) {
    const float ls = img[g.off_pm_logstd + tid];
    sig[tid] = expf(ls);
    ivar[tid] = expf(-2.f * ls);
  }
  double c_s = 1.0, c_k = 0.0;
  if (MODE != MRL_MODE_FVP && a.coef) { c_s = a.coef[0]; c_k = a.coef[1]; }
  const float cs = (float)c_s, ck = (float)c_k;
  float* Hh = H + g.off_act[L] * MRL_LDT;   // cached head output (mean | probs | value)
  float* EH = E + g.off_act[L] * MRL_LDT;   // Rz_L, then delta_L
  __syncthreads();

  for (int tile = t0; tile < t1; ++tile) {
    const int nvalid = (int)min((long long)MRL_TILE, a.N - (long long)tile * MRL_TILE);
    copy_f4(H, a.cache + (size_t)tile * g.act_rows * MRL_LDT, g.act_rows * MRL_LDT);
    if (tile + 1 < t1) {
      prefetch_l2(a.cache + (size_t)(tile + 1) * g.act_rows * MRL_LDT, g.act_rows * MRL_LDT);
      if (MODE == MRL_MODE_FVP) prefetch_l2(a.Zt + (size_t)(tile + 1) * g.d[1] * MRL_LDT, g.d[1] * MRL_LDT);
    }
    if (MODE == MRL_MODE_FVP) {
      // R-forward, layer 1: Rh1 = act'(h1) * (x.V1 + vb1).  Same thread wrote H[i] just above.
      const float4* zs = reinterpret_cast<const float4*>(a.Zt + (size_t)tile * g.d[1] * MRL_LDT);
      const float4* hs = reinterpret_cast<const float4*>(H);
      float4* dst = reinterpret_cast<float4*>(E);
      const float* vb1 = imgv + g.off_b[1];
      const int n4 = g.d[1] * (MRL_LDT / 4);
      for (int i = tid; i < n4; i += MRL_BWD_THREADS) {
        float4 z = zs[i];
        const float b = vb1[i / (MRL_LDT / 4)];
        if (L > 1) {
          const float4 h = hs[i];
          z.x = dact_from_h<ACT>(h.x) * (z.x + b); z.y = dact_from_h<ACT>(h.y) * (z.y + b);
          z.z = dact_from_h<ACT>(h.z) * (z.z + b); z.w = dact_from_h<ACT>(h.w) * (z.w + b);
        } else {
          z.x += b; z.y += b; z.z += b; z.w += b;
        }
        dst[i] = z;
      }
    }
    __syncthreads();
    if (MODE == MRL_MODE_FVP) {
      for (int l = 2; l <= L; ++l) {  // Rz_l = Rh_{l-1} W_l + h_{l-1} V_l + vb_l
        const float* RA = E + g.off_act[l - 1] * MRL_LDT;
        const float* HA = H + g.off_act[l - 1] * MRL_LDT;
        const float* Hl = H + g.off_act[l] * MRL_LDT;
        float* O = E + g.off_act[l] * MRL_LDT;
        const float* W = img + g.off_W[l];
        const float* V = imgv + g.off_W[l];
        const float* vb = imgv + g.off_b[l];
        const bool last = (l == L);
        const bool fold = last && HEAD == MRL_HEAD_GAUSS;   // Fisher metric of DiagGauss folded into the epilogue
        auto epi = [&](int c, int r, float v) {
          v += vb[c];
          if (!last) v *= dact_from_h<ACT>(Hl[c * MRL_LDT + r]);
          if (fold) v = (r < nvalid) ? v * ivar[c] : 0.f;
          O[c * MRL_LDT + r] = v;
        };
        const int mt = pick_mt(g.d[l], NW);
        const int nj = fwd_jobs(g.d[l], mt);
        for (int job = ln.warp; job < nj; job += NW) {
          if (mt == 1) fwd_job<1>(job, ln, RA, W, g.d[l - 1], HA, V, g.d[l - 1], g.ldw[l], g.d[l], epi);
          else fwd_job<2>(job, ln, RA, W, g.d[l - 1], HA, V, g.d[l - 1], g.ldw[l], g.d[l], epi);
        }
        __syncthreads();
      }
    }
    // ---- head: delta_L (un-normalised; 1/N is applied by the slab reduce)
    const bool head_folded = (MODE == MRL_MODE_FVP && HEAD == MRL_HEAD_GAUSS && L > 1);
    if (!head_folded && tid < MRL_TILE) {
      const float* aux = a.aux ? a.aux + (size_t)tile * g.naux * MRL_LDT + tid : nullptr;
      head_bwd_row<HEAD, MODE>(Hh, EH, GL, aux, tid, dL, tid < nvalid, a.reverse_kl, cs, ck, sig, ivar, clip_eps);
    }
    if (!head_folded) __syncthreads();
    // ---- reverse sweep: layers L..2 (weights in shared memory)
    for (int l = L; l >= 2; --l) {
      const float* D = E + g.off_act[l] * MRL_LDT;
      const float* Hp = H + g.off_act[l - 1] * MRL_LDT;
      float* Ep = E + g.off_act[l - 1] * MRL_LDT;
      const int M = g.d[l - 1], Nn = g.d[l];
      const int n_nblk = (Nn + 15) >> 4;
      const int n_bias = (Nn + 7) >> 3;
      // 16-row / 16-feature jobs when the 32-wide ones would leave warps without work
      const int mt = (fwd_jobs(M, 2) + ((M + 31) >> 5) * n_nblk + n_bias) < NW ? 1 : 2;
      const int n_delta = fwd_jobs(M, mt);
      const int n_grad = ((M + 16 * mt - 1) / (16 * mt)) * n_nblk;
      const float* WT = img + g.off_WT[l];
      auto epi = [&](int c, int r, float v) { Ep[c * MRL_LDT + r] = v * dact_from_h<ACT>(Hp[c * MRL_LDT + r]); };
      for (int job = ln.warp; job < n_delta + n_grad + n_bias; job += NW) {
        if (job < n_delta) {       // delta_{l-1} = (delta_l W_l^T) * act'(h_{l-1})
          if (mt == 1) fwd_job<1>(job, ln, D, WT, Nn, nullptr, nullptr, 0, g.ldt[l], M, epi);
          else fwd_job<2>(job, ln, D, WT, Nn, nullptr, nullptr, 0, g.ldt[l], M, epi);
        } else if (job < n_delta + n_grad) {
          if (mt == 1) grad_job<1>(job - n_delta, n_nblk, ln, Hp, M, D, Nn, G + g.off_W[l], g.ldw[l]);
          else grad_job<2>(job - n_delta, n_nblk, ln, Hp, M, D, Nn, G + g.off_W[l], g.ldw[l]);
        } else {
          bias_job(job - n_delta - n_grad, ln, D, Nn, G + g.off_b[l]);
        }
      }
      __syncthreads();
    }
    {  // layer 1: bias gradient here; delta_1 goes out as the tensor-core operand of l1_grad_tc_kernel
      const float* D1 = E;  // off_act[1] == 0
      const int n1 = g.d[1];
      for (int job = ln.warp; job < ((n1 + 7) >> 3); job += NW) bias_job(job, ln, D1, n1, G + g.off_b[1]);
      if (a.DG) {   // tensor-core operand (raw fp32, split by l1_grad_tc_kernel): 4 consecutive timesteps of one column per thread
        const int nu = a.nu;
        for (int i = tid; i < 16 * nu; i += MRL_BWD_THREADS) {
          const int tq = i / nu, n = i % nu;       // timesteps 4*tq .. +3 of this tile
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (n < n1) v = *reinterpret_cast<const float4*>(D1 + n * MRL_LDT + 4 * tq);
          *reinterpret_cast<float4*>(a.DG + l1_dg_offset((size_t)tile * 8 + (tq >> 1), tq & 1, n, nu)) = v;
        }
      }
    }
    __syncthreads();
  }
  if (gl_floats) {  // logstd gradient: reduce the per-timestep columns
    for (int j = ln.warp; j < dL; j += NW) {
      float s = GL[j * MRL_TILE + ln.lane] + GL[j * MRL_TILE + 32 + ln.lane];
      s = warp_sum(s);
      if (ln.lane == 0) G[g.off_pm_logstd + j] = s;
    }
    __syncthreads();
  }
  copy_f4(a.partm + (size_t)slab * g.pmid, G, g.bw_floats);
}

// =====================================================================================
size_t mid_forward_smem(const NetGeom& g) { return ((size_t)g.bw_floats + (size_t)g.act_rows * MRL_LDT) * 4; }
size_t mid_backward_smem(const NetGeom& g, int mode) {
  size_t f = (size_t)g.img_floats + g.bw_floats + 2 * (size_t)g.act_rows * MRL_LDT;
  if (mode == MRL_MODE_FVP) f += g.bw_floats;
  if (mode != MRL_MODE_FVP && g.head == MRL_HEAD_GAUSS) f += (size_t)g.d[g.L] * MRL_TILE;
  return f * 4;
}

template <int HEAD, int ACT, bool CLIP>
static cudaError_t launch_fwd_clip(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  const size_t sm = mid_forward_smem(g);
  cudaError_t e = cudaFuncSetAttribute(mid_forward_kernel<HEAD, ACT, CLIP>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (e != cudaSuccess) return e;
  mid_forward_kernel<HEAD, ACT, CLIP><<<n_slabs, MRL_MID_THREADS, sm, st>>>(g, a, eps);
  return cudaGetLastError();
}
template <int HEAD, int ACT>
static cudaError_t launch_fwd_t(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  if constexpr (HEAD != MRL_HEAD_VALUE) {
    if (eps > 0.f) return launch_fwd_clip<HEAD, ACT, true>(g, a, n_slabs, st, eps);
  }
  return launch_fwd_clip<HEAD, ACT, false>(g, a, n_slabs, st, eps);
}
template <int HEAD, int ACT, int MODE>
static cudaError_t launch_bwd_t(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  const size_t sm = mid_backward_smem(g, MODE);
  cudaError_t e = cudaFuncSetAttribute(mid_backward_kernel<HEAD, ACT, MODE>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (e != cudaSuccess) return e;
  mid_backward_kernel<HEAD, ACT, MODE><<<n_slabs, MRL_BWD_THREADS, sm, st>>>(g, a, eps);
  return cudaGetLastError();
}

#define DISPATCH_ACT(FN, HEADV, ...)                                     \
  switch (g.act) {                                                       \
    case MRL_ACT_TANH: return FN<HEADV, MRL_ACT_TANH>(__VA_ARGS__);      \
    case MRL_ACT_RELU: return FN<HEADV, MRL_ACT_RELU>(__VA_ARGS__);      \
    default: return FN<HEADV, MRL_ACT_SIGMOID>(__VA_ARGS__);             \
  }

cudaError_t launch_mid_forward(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps) {
  switch (g.head) {
    case MRL_HEAD_GAUSS: DISPATCH_ACT(launch_fwd_t, MRL_HEAD_GAUSS, g, a, n_slabs, st, clip_eps)
    case MRL_HEAD_CAT: DISPATCH_ACT(launch_fwd_t, MRL_HEAD_CAT, g, a, n_slabs, st, clip_eps)
    default: DISPATCH_ACT(launch_fwd_t, MRL_HEAD_VALUE, g, a, n_slabs, st, clip_eps)
  }
}

template <int HEAD, int ACT>
static cudaError_t launch_bwd_mode(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float eps) {
  if (a.mode == MRL_MODE_FVP) return launch_bwd_t<HEAD, ACT, MRL_MODE_FVP>(g, a, n_slabs, st, eps);
  if (a.mode == MRL_MODE_GRAD_CLIP) {
    if constexpr (HEAD != MRL_HEAD_VALUE) return launch_bwd_t<HEAD, ACT, MRL_MODE_GRAD_CLIP>(g, a, n_slabs, st, eps);
    return cudaErrorInvalidValue;   // a value net has no clipped objective
  }
  return launch_bwd_t<HEAD, ACT, MRL_MODE_GRAD>(g, a, n_slabs, st, eps);
}

cudaError_t launch_mid_backward(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps) {
  switch (g.head) {
    case MRL_HEAD_GAUSS: DISPATCH_ACT(launch_bwd_mode, MRL_HEAD_GAUSS, g, a, n_slabs, st, clip_eps)
    case MRL_HEAD_CAT: DISPATCH_ACT(launch_bwd_mode, MRL_HEAD_CAT, g, a, n_slabs, st, clip_eps)
    default: DISPATCH_ACT(launch_bwd_mode, MRL_HEAD_VALUE, g, a, n_slabs, st, clip_eps)
  }
}
