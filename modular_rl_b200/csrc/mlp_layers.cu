// Layer-by-layer path for layers >= 2 of the nets that the fused mid_* kernels cannot hold in shared memory
// (hidden layers up to 256 units, up to 6 layers; mrl_net_create picks it from the geometry).
//
// Same contract as mlp_mid.cu (MidFwdArgs / MidBwdArgs): Z1 from the layer-1 forward kernel in, the activation
// cache, the row-major head output, loss_part[n_slabs][4], the partm[n_slabs][pmid] slab partials in image order
// and delta_1 in the DG order of l1_grad_tc_kernel out.  Instead of one fused kernel per slab, a pass is a
// sequence of launches over all tiles, one per layer and step:
//
//   forward  : h1 = act(Z1 + b1); Z_l = H_{l-1} W_l + b_l, H_l = act(Z_l) for l = 2..L (cache); head
//   gradient : dL/dz_L from the head; for l = L..2: delta_{l-1} = (delta_l W_l^T) . act'(h_{l-1}),
//              W_l partial H_{l-1}^T delta_l, b_l partial; delta_1 -> DG, b_1 partial
//   Fvp      : Rh1 = act'(h1) (x.V1 + vb1); Rz_l = Rh_{l-1} W_l + h_{l-1} V_l + vb_l; Fisher metric at the
//              head; then the reverse sweep of the gradient mode
//
// Every product is 3xTF32 mma.sync on 32x16 warp tiles (mma_tf32.cuh), with the operands in the tile-major
// layout of Z1 / cache.  A GEMM CTA stages a 64-column panel of the weights (and of the tangent) in shared
// memory once and applies it to its share of the tiles, so weight traffic does not grow with the batch.  The
// deltas and R-activations live in two ping-pong buffers of [n_tiles + 1][max width][LDT].  All sums run in a
// fixed order (no atomics), so a repeated call is bit-identical.
//
// The heads are the row functions of heads.cuh that mid_forward_kernel / mid_backward_kernel call.
#include "common.cuh"
#include "heads.cuh"
#include "kernels.h"
#include "mma_tf32.cuh"

#define LW_THREADS 256   // 8 warps: a 64-timestep x 64-column block, one 32 x 16 job per warp
#define LW_COLS 64       // output columns per GEMM CTA (one weight panel)
#define LW_LDP 72        // panel row stride in shared memory: conflict-free B-fragment loads
#define LW_KCHUNK 64     // products per tensor-core accumulator chain (one tile of timesteps in the gradient)

// O[c][r] = f(sum_k A[k][r] B[k][c] (+ sum_k A2[k][r] B2[k][c])), per tile; f adds the bias, applies the
// activation and / or multiplies by act'(H[c][r]) when those are given (in that order)
struct LwGemm {
  const float* A; long long lda;     // tile-major operands: X + tile * ldx + feature * MRL_LDT + r
  const float* A2; long long lda2;   // nullptr: one product
  const float* B; const float* B2;   // weights [K][ldb] (theta / tangent image)
  int ldb, K, N;
  const float* bias;                 // [N] or nullptr
  int apply_act;
  const float* H; long long ldh;     // nullptr: no act' factor
  float* O; long long ldo;
  int n_tiles;
};

template <int ACT>
__global__ void __launch_bounds__(LW_THREADS, 2) lw_gemm_kernel(LwGemm p) {
  extern __shared__ __align__(16) float panel[];
  const int c0 = blockIdx.x * LW_COLS;
  const int npanel = p.A2 ? 2 : 1, kp = round_up(p.K, 8);   // zero rows up to a whole k-step
  for (int q = 0; q < npanel; ++q) {
    const float* B = q ? p.B2 : p.B;
    float* S = panel + q * kp * LW_LDP;
    for (int i = threadIdx.x; i < kp * LW_COLS; i += LW_THREADS) {
      const int k = i / LW_COLS, c = i % LW_COLS;
      S[k * LW_LDP + c] = k < p.K && c0 + c < p.N ? B[(size_t)k * p.ldb + c0 + c] : 0.f;
    }
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = (warp & 1) * 32, cw = (warp >> 1) * 16;
  if (c0 + cw >= p.N) return;   // warp-uniform, no barrier below
  const int g = lane >> 2, t = lane & 3;
  for (int tile = blockIdx.y; tile < p.n_tiles; tile += gridDim.y) {
    float acc[2][2][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;
    // the tensor core accumulates with less than fp32 care: at most LW_KCHUNK products per accumulator chain,
    // the chains added with FADD
    for (int q = 0; q < npanel; ++q) {
      const float* A = (q ? p.A2 + (size_t)tile * p.lda2 : p.A + (size_t)tile * p.lda);
      const float* S = panel + q * kp * LW_LDP;
      for (int k0 = 0; k0 < p.K; k0 += LW_KCHUNK) {
        float part[2][2][4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) part[i][j][e] = 0.f;
        mma_fwd_acc<2>(part, A + (size_t)k0 * MRL_LDT, S + k0 * LW_LDP, min(LW_KCHUNK, p.K - k0), LW_LDP, r0, cw, lane);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] += part[i][j][e];
      }
    }
    float* O = p.O + (size_t)tile * p.ldo;
    const float* H = p.H ? p.H + (size_t)tile * p.ldh : nullptr;
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
      for (int ni = 0; ni < 2; ++ni)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c = c0 + cw + 8 * ni + 2 * t + (q & 1), r = r0 + 16 * mi + g + 8 * (q >> 1);
          if (c < p.N) {
            float v = acc[mi][ni][q];
            if (p.bias) v += p.bias[c];
            if (p.apply_act) v = act_fn<ACT>(v);
            if (H) v *= dact_from_h<ACT>(H[c * MRL_LDT + r]);
            O[c * MRL_LDT + r] = v;
          }
        }
  }
}

// Weight-gradient partial of one slab: part[slab][m * ldw + n] = sum over the slab's timesteps of
// H[m][r] D[n][r].  CTA: a 64 x 64 block of the matrix and one slab; warp: 32 m x 16 n, accumulated in
// registers over the slab's tiles in order.
struct LwGrad {
  const float* H; long long ldh;   // H_{l-1}, tile-major
  const float* D; long long ldd;   // delta_l, tile-major
  int M, N, ldw;
  float* part; int pstride;        // partm + off_W[l], pmid
  int n_tiles, slab_tiles;
};
__global__ void __launch_bounds__(LW_THREADS, 2) lw_wgrad_kernel(LwGrad p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nb = (p.N + LW_COLS - 1) / LW_COLS;
  const int m0 = (blockIdx.x / nb) * 64 + (warp & 1) * 32, n0 = (blockIdx.x % nb) * LW_COLS + (warp >> 1) * 16;
  if (m0 >= p.M || n0 >= p.N) return;
  const int g = lane >> 2, t = lane & 3;
  const int slab = blockIdx.y;
  const int t0 = slab * p.slab_tiles, t1 = min(t0 + p.slab_tiles, p.n_tiles);
  int ar[4], dr[2];   // rows m0+g, +8, ... and n0+g, +8 (clamped; out-of-range rows are never stored)
#pragma unroll
  for (int q = 0; q < 4; ++q) ar[q] = min(m0 + g + 8 * q, p.M - 1) * MRL_LDT + t;
#pragma unroll
  for (int q = 0; q < 2; ++q) dr[q] = min(n0 + g + 8 * q, p.N - 1) * MRL_LDT + t;
  float acc[2][2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;
  for (int tile = t0; tile < t1; ++tile) {   // one tile per accumulator chain, the tiles added with FADD
    const float* __restrict__ A = p.H + (size_t)tile * p.ldh;
    const float* __restrict__ D = p.D + (size_t)tile * p.ldd;
    float part[2][2][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) part[i][j][q] = 0.f;
#pragma unroll 2
    for (int k0 = 0; k0 < MRL_TILE; k0 += 8) {
      uint32_t bh[2][2], bl[2][2], ah[2][4], al[2][4];
#pragma unroll
      for (int ni = 0; ni < 2; ++ni) {
        split_tf32(D[dr[ni] + k0], bh[ni][0], bl[ni][0]);
        split_tf32(D[dr[ni] + k0 + 4], bh[ni][1], bl[ni][1]);
      }
#pragma unroll
      for (int mi = 0; mi < 2; ++mi) {
        split_tf32(A[ar[2 * mi] + k0], ah[mi][0], al[mi][0]);
        split_tf32(A[ar[2 * mi + 1] + k0], ah[mi][1], al[mi][1]);
        split_tf32(A[ar[2 * mi] + k0 + 4], ah[mi][2], al[mi][2]);
        split_tf32(A[ar[2 * mi + 1] + k0 + 4], ah[mi][3], al[mi][3]);
      }
      mma3_tiles<2>(part, ah, al, bh, bl);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i][j][q] += part[i][j][q];
  }
  float* G = p.part + (size_t)slab * p.pstride;
#pragma unroll
  for (int mi = 0; mi < 2; ++mi)
#pragma unroll
    for (int ni = 0; ni < 2; ++ni)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int m = m0 + 16 * mi + g + 8 * (q >> 1), n = n0 + 8 * ni + 2 * t + (q & 1);
        if (m < p.M && n < p.N) G[m * p.ldw + n] = acc[mi][ni][q];
      }
}

// Bias partial of one slab: part[slab][j] = sum over the slab's tiles of the tile's column sum of D[j][.]
// (one warp per (slab, feature); per tile as bias_job of mlp_mid.cu)
__global__ void lw_colsum_kernel(const float* __restrict__ D, long long ldd, int n, float* part, int pstride,
                                 int n_tiles, int slab_tiles, int n_slabs) {
  const int gw = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  const int slab = gw / n, j = gw % n;
  if (slab >= n_slabs) return;
  const int t0 = slab * slab_tiles, t1 = min(t0 + slab_tiles, n_tiles);
  float acc = 0.f;
  for (int tile = t0; tile < t1; ++tile) {
    const float* d = D + (size_t)tile * ldd + j * MRL_LDT;
    acc += warp_sum(d[lane] + d[32 + lane]);
  }
  if (lane == 0) part[(size_t)slab * pstride + j] = acc;
}

// Layer 1, elementwise over [tile][d1][LDT]: forward O = act(Z + b); R-forward (H given) O = act'(H) (Z + b)
template <int ACT>
__global__ void lw_layer1_kernel(const float* __restrict__ Z, const float* __restrict__ b, const float* H,
                                 long long ldh, float* O, long long ldo, int d1, int n_tiles) {
  const long long per = (long long)d1 * MRL_LDT;
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= per * n_tiles) return;
  const long long tile = i / per, e = i % per;
  const float z = Z[i] + b[e / MRL_LDT];
  O[tile * ldo + e] = H ? dact_from_h<ACT>(H[tile * ldh + e]) * z : act_fn<ACT>(z);
}

// delta_1 -> DG (the raw fp32 operand of l1_grad_tc_kernel, l1_dg_offset)
__global__ void lw_dg_kernel(const float* __restrict__ D1, long long ldd, int n1, int nu, float* DG, int n_tiles) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)n_tiles * 16 * nu) return;
  const long long tile = i / (16 * nu);
  const int rem = (int)(i % (16 * nu)), tq = rem / nu, n = rem % nu;   // timesteps 4*tq .. +3, column n
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (n < n1) v = *reinterpret_cast<const float4*>(D1 + tile * ldd + n * MRL_LDT + 4 * tq);
  *reinterpret_cast<float4*>(DG + l1_dg_offset((size_t)tile * 8 + (tq >> 1), tq & 1, n, nu)) = v;
}

// ---- heads (heads.cuh): one thread per timestep, one CTA per slab; sigma, log sigma and 1/sigma^2 staged per CTA
template <int HEAD, bool CLIP>
__global__ void __launch_bounds__(MRL_TILE, 1) lw_head_fwd_kernel(NetGeom g, MidFwdArgs a, float clip_eps) {
  __shared__ double red[32];
  __shared__ float sig[MRL_MAX_DOUT], logsig[MRL_MAX_DOUT];
  const int r = threadIdx.x, L = g.L, dL = g.d[L];
  const int slab = blockIdx.x;
  const int t0 = slab * a.slab_tiles, t1 = min(t0 + a.slab_tiles, a.n_tiles);
  if (HEAD == MRL_HEAD_GAUSS && r < dL) {
    const float ls = a.img[g.off_pm_logstd + r];
    logsig[r] = ls;
    sig[r] = expf(ls);
  }
  __syncthreads();
  double s_clip = 0.0;   // declared first: the other instances' register assignment stays as it was
  double s_surr = 0.0, s_kl = 0.0, s_ent = 0.0;
  for (int tile = t0; tile < t1; ++tile) {
    const bool valid = (long long)tile * MRL_TILE + r < a.N;
    float* headbuf = a.cache + ((size_t)tile * g.act_rows + g.off_act[L]) * MRL_LDT;
    const float* aux = a.aux ? a.aux + (size_t)tile * g.naux * MRL_LDT + r : nullptr;
    head_fwd_row<HEAD, CLIP>(headbuf, aux, r, dL, valid, a.reverse_kl, sig, logsig, s_surr, s_kl, s_ent, clip_eps,
                             s_clip);
    if (a.head_out && valid)
      for (int j = 0; j < dL; ++j) a.head_out[((size_t)tile * MRL_TILE + r) * dL + j] = headbuf[j * MRL_LDT + r];
  }
  if (a.loss_part) {
    const double v0 = block_sum(s_surr, red);
    const double v1 = block_sum(s_kl, red);
    const double v2 = block_sum(s_ent, red);
    double v3 = 0.0;
    if constexpr (CLIP) v3 = block_sum(s_clip, red);
    if (r == 0) {
      double* o = a.loss_part + (size_t)slab * 4;
      o[0] = v0; o[1] = v1; o[2] = v2; o[3] = v3;
    }
  }
}

// delta_L (Fvp: the metric applied to Rz_L) into E, the logstd partial (gradient mode, DiagGauss)
template <int HEAD, int MODE>
__global__ void __launch_bounds__(MRL_TILE, 1) lw_head_bwd_kernel(NetGeom g, MidBwdArgs a, float* E, long long lde,
                                                                float clip_eps) {
  __shared__ float GL[MRL_MAX_DOUT * MRL_TILE];
  __shared__ float sig[MRL_MAX_DOUT], ivar[MRL_MAX_DOUT];
  const int r = threadIdx.x, L = g.L, dL = g.d[L];
  const int slab = blockIdx.x;
  const int t0 = slab * a.slab_tiles, t1 = min(t0 + a.slab_tiles, a.n_tiles);
  const bool gl_on = MODE != MRL_MODE_FVP && HEAD == MRL_HEAD_GAUSS;
  if (gl_on)
    for (int j = 0; j < dL; ++j) GL[j * MRL_TILE + r] = 0.f;
  if (HEAD == MRL_HEAD_GAUSS && r < dL) {
    const float ls = a.img[g.off_pm_logstd + r];
    sig[r] = expf(ls);
    ivar[r] = expf(-2.f * ls);
  }
  __syncthreads();
  double c_s = 1.0, c_k = 0.0;
  if (MODE != MRL_MODE_FVP && a.coef) { c_s = a.coef[0]; c_k = a.coef[1]; }
  const float cs = (float)c_s, ck = (float)c_k;
  for (int tile = t0; tile < t1; ++tile) {
    const bool valid = (long long)tile * MRL_TILE + r < a.N;
    const float* Hh = a.cache + ((size_t)tile * g.act_rows + g.off_act[L]) * MRL_LDT;
    const float* aux = a.aux ? a.aux + (size_t)tile * g.naux * MRL_LDT + r : nullptr;
    head_bwd_row<HEAD, MODE>(Hh, E + (size_t)tile * lde, GL, aux, r, dL, valid, a.reverse_kl, cs, ck, sig, ivar,
                             clip_eps);
  }
  if (HEAD == MRL_HEAD_GAUSS) {   // logstd partial: the per-timestep columns summed (zero in Fvp mode)
    __syncthreads();
    const int warp = r >> 5, lane = r & 31;
    for (int j = warp; j < dL; j += MRL_TILE / 32) {
      float s = 0.f;
      if (gl_on) s = warp_sum(GL[j * MRL_TILE + lane] + GL[j * MRL_TILE + 32 + lane]);
      if (lane == 0) a.partm[(size_t)slab * g.pmid + g.off_pm_logstd + j] = s;
    }
  }
}

// =====================================================================================
static int max_width(const NetGeom& g) {
  int w = 0;
  for (int l = 1; l <= g.L; ++l) w = max(w, g.d[l]);
  return w;
}
size_t layers_ws_floats(const NetGeom& g, long long n_tiles) {
  return (size_t)(n_tiles + 1) * max_width(g) * MRL_LDT;
}

template <int ACT>
static cudaError_t gemm(const LwGemm& p, cudaStream_t st) {
  const size_t sm = (size_t)(p.A2 ? 2 : 1) * round_up(p.K, 8) * LW_LDP * 4;
  cudaError_t e = mrl_func_smem((const void*)lw_gemm_kernel<ACT>, sm);
  if (e != cudaSuccess) return e;
  const int gx = (p.N + LW_COLS - 1) / LW_COLS;
  // CTAs per SM that the panel leaves room for (at most 2, the launch bound); each CTA takes every gy-th tile
  const int per_sm = max(1, min(2, (int)((227 * 1024) / (sm + 1024))));
  const int gy = max(1, min(p.n_tiles, (per_sm * mrl_sm_count() + gx - 1) / gx));
  lw_gemm_kernel<ACT><<<dim3(gx, gy), LW_THREADS, sm, st>>>(p);
  return cudaGetLastError();
}

static cudaError_t wgrad(const NetGeom& g, int l, const float* H, long long ldh, const float* D, long long ldd,
                         float* partm, int n_tiles, int slab_tiles, int n_slabs, cudaStream_t st) {
  LwGrad p;
  p.H = H; p.ldh = ldh; p.D = D; p.ldd = ldd;
  p.M = g.d[l - 1]; p.N = g.d[l]; p.ldw = g.ldw[l];
  p.part = partm + g.off_W[l]; p.pstride = g.pmid;
  p.n_tiles = n_tiles; p.slab_tiles = slab_tiles;
  const int blocks = ((p.M + 63) / 64) * ((p.N + LW_COLS - 1) / LW_COLS);
  lw_wgrad_kernel<<<dim3(blocks, n_slabs), LW_THREADS, 0, st>>>(p);
  return cudaGetLastError();
}

static cudaError_t colsum(const float* D, long long ldd, int n, float* part, int pstride, int n_tiles, int slab_tiles,
                          int n_slabs, cudaStream_t st) {
  const long long threads = (long long)n_slabs * n * 32;
  lw_colsum_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(D, ldd, n, part, pstride, n_tiles, slab_tiles, n_slabs);
  return cudaGetLastError();
}

template <int ACT>
static cudaError_t layer1(const NetGeom& g, const float* Z, const float* b, const float* H, long long ldh, float* O,
                          long long ldo, int n_tiles, cudaStream_t st) {
  const long long n = (long long)n_tiles * g.d[1] * MRL_LDT;
  lw_layer1_kernel<ACT><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(Z, b, H, ldh, O, ldo, g.d[1], n_tiles);
  return cudaGetLastError();
}

#define LW_TRY(call)                         \
  do {                                       \
    cudaError_t _e = (call);                 \
    if (_e != cudaSuccess) return _e;        \
  } while (0)

template <int HEAD, int ACT>
static cudaError_t forward_t(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, int* launches,
                             float eps) {
  const long long ldc = (long long)g.act_rows * MRL_LDT;
  LW_TRY(layer1<ACT>(g, a.Zt, a.img + g.off_b[1], nullptr, 0, a.cache, ldc, a.n_tiles, st));
  for (int l = 2; l <= g.L; ++l) {
    LwGemm p = {};
    p.A = a.cache + (size_t)g.off_act[l - 1] * MRL_LDT; p.lda = ldc;
    p.B = a.img + g.off_W[l]; p.ldb = g.ldw[l]; p.K = g.d[l - 1]; p.N = g.d[l];
    p.bias = a.img + g.off_b[l]; p.apply_act = l < g.L;
    p.O = a.cache + (size_t)g.off_act[l] * MRL_LDT; p.ldo = ldc;
    p.n_tiles = a.n_tiles;
    LW_TRY(gemm<ACT>(p, st));
  }
  if (HEAD != MRL_HEAD_VALUE && eps > 0.f) lw_head_fwd_kernel<HEAD, HEAD != MRL_HEAD_VALUE><<<n_slabs, MRL_TILE, 0, st>>>(g, a, eps);
  else lw_head_fwd_kernel<HEAD, false><<<n_slabs, MRL_TILE, 0, st>>>(g, a, eps);
  *launches = g.L + 1;
  return cudaGetLastError();
}

template <int HEAD, int ACT, int MODE>
static cudaError_t backward_t(const NetGeom& g, const MidBwdArgs& a, float* R0, float* R1, int n_slabs,
                              cudaStream_t st, int* launches, float eps) {
  const long long ldc = (long long)g.act_rows * MRL_LDT, ldr = (long long)max_width(g) * MRL_LDT;
  const float* H = a.cache;
  float* cur = R0;
  float* nxt = R1;
  int nl = 0;
  if (MODE == MRL_MODE_FVP) {   // R-forward: Rh1, then Rz_l = Rh_{l-1} W_l + h_{l-1} V_l + vb_l
    LW_TRY(layer1<ACT>(g, a.Zt, a.imgv + g.off_b[1], H, ldc, cur, ldr, a.n_tiles, st));
    ++nl;
    for (int l = 2; l <= g.L; ++l) {
      LwGemm p = {};
      p.A = cur; p.lda = ldr;
      p.A2 = H + (size_t)g.off_act[l - 1] * MRL_LDT; p.lda2 = ldc;
      p.B = a.img + g.off_W[l]; p.B2 = a.imgv + g.off_W[l]; p.ldb = g.ldw[l]; p.K = g.d[l - 1]; p.N = g.d[l];
      p.bias = a.imgv + g.off_b[l];
      if (l < g.L) { p.H = H + (size_t)g.off_act[l] * MRL_LDT; p.ldh = ldc; }
      p.O = nxt; p.ldo = ldr;
      p.n_tiles = a.n_tiles;
      LW_TRY(gemm<ACT>(p, st));
      ++nl;
      float* s = cur; cur = nxt; nxt = s;
    }
  }
  lw_head_bwd_kernel<HEAD, MODE><<<n_slabs, MRL_TILE, 0, st>>>(g, a, cur, ldr, eps);
  LW_TRY(cudaGetLastError());
  ++nl;
  for (int l = g.L; l >= 2; --l) {
    LwGemm p = {};   // delta_{l-1} = (delta_l W_l^T) * act'(h_{l-1})
    p.A = cur; p.lda = ldr;
    p.B = a.img + g.off_WT[l]; p.ldb = g.ldt[l]; p.K = g.d[l]; p.N = g.d[l - 1];
    p.H = H + (size_t)g.off_act[l - 1] * MRL_LDT; p.ldh = ldc;
    p.O = nxt; p.ldo = ldr;
    p.n_tiles = a.n_tiles;
    LW_TRY(gemm<ACT>(p, st));
    LW_TRY(wgrad(g, l, H + (size_t)g.off_act[l - 1] * MRL_LDT, ldc, cur, ldr, a.partm, a.n_tiles, a.slab_tiles, n_slabs, st));
    LW_TRY(colsum(cur, ldr, g.d[l], a.partm + g.off_b[l], g.pmid, a.n_tiles, a.slab_tiles, n_slabs, st));
    nl += 3;
    float* s = cur; cur = nxt; nxt = s;
  }
  LW_TRY(colsum(cur, ldr, g.d[1], a.partm + g.off_b[1], g.pmid, a.n_tiles, a.slab_tiles, n_slabs, st));
  const long long n = (long long)a.n_tiles * 16 * a.nu;
  lw_dg_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cur, ldr, g.d[1], a.nu, a.DG, a.n_tiles);
  *launches = nl + 2;
  return cudaGetLastError();
}

template <int HEAD>
static auto forward_fn(const NetGeom& g) {
  switch (g.act) {
    case MRL_ACT_TANH: return forward_t<HEAD, MRL_ACT_TANH>;
    case MRL_ACT_RELU: return forward_t<HEAD, MRL_ACT_RELU>;
    default: return forward_t<HEAD, MRL_ACT_SIGMOID>;
  }
}
template <int HEAD, int MODE>
static auto backward_fn(const NetGeom& g) {
  switch (g.act) {
    case MRL_ACT_TANH: return backward_t<HEAD, MRL_ACT_TANH, MODE>;
    case MRL_ACT_RELU: return backward_t<HEAD, MRL_ACT_RELU, MODE>;
    default: return backward_t<HEAD, MRL_ACT_SIGMOID, MODE>;
  }
}

cudaError_t launch_layers_forward(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, int* launches,
                                  float clip_eps) {
  if (g.L < 2 || a.cache == nullptr) return cudaErrorInvalidValue;
  switch (g.head) {
    case MRL_HEAD_GAUSS: return forward_fn<MRL_HEAD_GAUSS>(g)(g, a, n_slabs, st, launches, clip_eps);
    case MRL_HEAD_CAT: return forward_fn<MRL_HEAD_CAT>(g)(g, a, n_slabs, st, launches, clip_eps);
    default: return forward_fn<MRL_HEAD_VALUE>(g)(g, a, n_slabs, st, launches, clip_eps);
  }
}

template <int MODE>
static cudaError_t backward_mode(const NetGeom& g, const MidBwdArgs& a, float* R0, float* R1, int n_slabs,
                                 cudaStream_t st, int* launches) {
  switch (g.head) {
    case MRL_HEAD_GAUSS: return backward_fn<MRL_HEAD_GAUSS, MODE>(g)(g, a, R0, R1, n_slabs, st, launches, 0.f);
    case MRL_HEAD_CAT: return backward_fn<MRL_HEAD_CAT, MODE>(g)(g, a, R0, R1, n_slabs, st, launches, 0.f);
    default: return backward_fn<MRL_HEAD_VALUE, MODE>(g)(g, a, R0, R1, n_slabs, st, launches, 0.f);
  }
}
cudaError_t launch_layers_backward(const NetGeom& g, const MidBwdArgs& a, float* R0, float* R1, int n_slabs,
                                   cudaStream_t st, int* launches, float clip_eps) {
  if (g.L < 2 || a.DG == nullptr) return cudaErrorInvalidValue;
  if (a.mode == MRL_MODE_FVP) return backward_mode<MRL_MODE_FVP>(g, a, R0, R1, n_slabs, st, launches);
  if (a.mode == MRL_MODE_GRAD_CLIP) {
    switch (g.head) {   // a value net has no clipped objective
      case MRL_HEAD_GAUSS:
        return backward_fn<MRL_HEAD_GAUSS, MRL_MODE_GRAD_CLIP>(g)(g, a, R0, R1, n_slabs, st, launches, clip_eps);
      case MRL_HEAD_CAT:
        return backward_fn<MRL_HEAD_CAT, MRL_MODE_GRAD_CLIP>(g)(g, a, R0, R1, n_slabs, st, launches, clip_eps);
      default: return cudaErrorInvalidValue;
    }
  }
  return backward_mode<MRL_MODE_GRAD>(g, a, R0, R1, n_slabs, st, launches);
}
