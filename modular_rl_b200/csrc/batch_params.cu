// Parameter packing, batch repacking and the fp64 slab reduce.
//
// theta (the reference's flat vector, core.py:518-557) is expanded once per set_params into the
// shared-memory image the fused chain loads ([biases | logstd | W2..WL | W2^T..WL^T]) and into the
// split-precision tensor-core operand of layer 1 (see mlp_l1_tc.cu).  Side inputs of the batch
// (advantages, actions, old probabilities, value targets) are repacked into the tile-major layout.
#include <cstdlib>
#include "common.cuh"
#include "kernels.h"
#include "comm.h"

// ------------------------------------------------------------------------------------
// theta (flat, reference order) -> the shared-memory image and the layer-1 tensor-core operand
// WB (l1_wb_offset: K-major UMMA core-matrix order, hi = rna_tf32(x), lo = rna_tf32(x - hi)).
__global__ void pack_params_kernel(NetGeom g, const float* __restrict__ theta, float* __restrict__ img,
                                   float* __restrict__ WB, int nu) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n_wb = g.d0p * nu;
  if (i < n_wb) {
    const int k = i / nu, n = i % nu;
    const float x = (k < g.d[0] && n < g.d[1]) ? theta[g.off_flat_W[1] + k * g.d[1] + n] : 0.f;
    const float h = tf32_rna(x);
    float* base = WB + l1_wb_offset(k >> 3, (k & 7) >> 2, n, nu) + (k & 3);
    base[0] = h;
    base[nu * 8] = tf32_rna(x - h);
    return;
  }
  const int j = i - n_wb;
  if (j >= g.img_floats) return;
  float v = 0.f;
  if (j < g.bias_floats) {
    if (j >= g.off_pm_logstd) {
      const int q = j - g.off_pm_logstd;
      if (g.off_flat_logstd >= 0 && q < g.d[g.L]) v = theta[g.off_flat_logstd + q];
    } else {
      for (int l = g.L; l >= 1; --l)
        if (j >= g.off_b[l]) {
          const int q = j - g.off_b[l];
          if (q < g.d[l]) v = theta[g.off_flat_b[l] + q];
          break;
        }
    }
  } else if (j < g.bw_floats) {
    for (int l = g.L; l >= 2; --l)
      if (j >= g.off_W[l]) {
        const int q = j - g.off_W[l];
        const int row = q / g.ldw[l], col = q % g.ldw[l];
        if (col < g.d[l]) v = theta[g.off_flat_W[l] + row * g.d[l] + col];
        break;
      }
  } else {
    for (int l = g.L; l >= 2; --l)
      if (j >= g.off_WT[l]) {
        const int q = j - g.off_WT[l];
        const int row = q / g.ldt[l], col = q % g.ldt[l];  // row = output unit, col = input unit
        if (col < g.d[l - 1]) v = theta[g.off_flat_W[l] + col * g.d[l] + row];
        break;
      }
  }
  img[j] = v;
}

// ------------------------------------------------------------------------------------
// flat[i] = scale * sum_slabs(partials) (+ l2c2 * theta[i]); on the logstd block an Fvp is vls * v[i]
// (fvp[logstd] = 2 v_logstd is data independent, SURVEY A.3)
// fp64 accumulation in a fixed slab order -> deterministic.
// Data-parallel with the peer-memory transport (push.world > 0): phase 1 writes this rank's sums into its exported
// vector and the last CTA to finish raises this rank's flag on every peer; the last RED_GATHER_CTAS CTAs to finish
// (by arrival ticket) stay for phase 2: they wait for all ranks' flags, read the peers' vectors over NVLink - thread
// row sy reads rank sy, batches of reads in flight - and write the sum over ranks (rank order: identical bits
// everywhere).  At most RED_GATHER_CTAS CTAs ever spin (two per SM), every other CTA leaves after phase 1,
// so the CTAs that have not started yet always find SM slots: no residency requirement on the grid (round 2 first
// sized the grid to be resident and let every CTA spin - slower phase 1, and two such kernels on one GPU could have
// starved each other), and phase 1 keeps its full one-chunk-per-CTA grid.
#define RED_PX 32
#define RED_SY 8
#define RED_UN 8
#define RED_GATHER_CTAS 296   // CTAs that stay for the exchange phase (two per SM)
#define RED_GB 5              // chunks per batch of peer reads (Humanoid: 1 391 chunks / 296 = one batch)
static_assert(RED_SY >= MRL_P2P_MAX_WORLD, "one thread row per rank in the exchange phase");
__global__ void __launch_bounds__(RED_PX * RED_SY) reduce_partials_kernel(
    NetGeom g, const float* __restrict__ part1, const float* __restrict__ partm, int n_slabs, double scale,
    const float* __restrict__ theta, double l2c2, const float* __restrict__ vlogstd_src, double vls,
    float* __restrict__ out32, double* __restrict__ out64, P2pPush push, P2pGather ga) {
  __shared__ double acc[RED_SY][RED_PX];
  const int px = threadIdx.x, sy = threadIdx.y;
  const int n_chunks = (g.P + RED_PX - 1) / RED_PX;
  for (int chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    const int i = chunk * RED_PX + px;
    double s0 = 0.0, s1 = 0.0;   // even / odd members of a batch of RED_UN slabs
    if (i < g.P) {
      const float* src = nullptr;
      size_t stride = 0;
      if (i < g.off_flat_b[1]) {
        const int k = i / g.d[1], n = i % g.d[1];
        src = part1 + (size_t)k * g.n1p + n;
        stride = (size_t)g.d[0] * g.n1p;
      } else if (g.off_flat_logstd >= 0 && i >= g.off_flat_logstd) {
        src = partm + g.off_pm_logstd + (i - g.off_flat_logstd);
        stride = g.pmid;
      } else {
        for (int l = g.L; l >= 1; --l) {
          if (i >= g.off_flat_b[l]) {
            src = partm + g.off_b[l] + (i - g.off_flat_b[l]);
            break;
          }
          if (i >= g.off_flat_W[l]) {
            const int q = i - g.off_flat_W[l];
            src = partm + g.off_W[l] + (q / g.d[l]) * g.ldw[l] + (q % g.d[l]);
            break;
          }
        }
        stride = g.pmid;
      }
      // this thread's slabs: sy, sy+8, ...; RED_UN loads in flight at a time, summed in slab order
      int sl = sy;
      for (; sl + (RED_UN - 1) * RED_SY < n_slabs; sl += RED_UN * RED_SY) {
        float a[RED_UN];
#pragma unroll
        for (int u = 0; u < RED_UN; ++u) a[u] = __ldcs(src + (size_t)(sl + u * RED_SY) * stride);
#pragma unroll
        for (int u = 0; u < RED_UN; u += 2) { s0 += (double)a[u]; s1 += (double)a[u + 1]; }
      }
      for (; sl < n_slabs; sl += RED_SY) s0 += (double)__ldcs(src + (size_t)sl * stride);
    }
    acc[sy][px] = s0 + s1;
    __syncthreads();
    if (sy == 0 && i < g.P) {
      double r = 0.0;
#pragma unroll
      for (int q = 0; q < RED_SY; ++q) r += acc[q][px];   // fixed order -> deterministic
      r *= scale;
      if (vlogstd_src != nullptr && g.off_flat_logstd >= 0 && i >= g.off_flat_logstd) r = vls * (double)vlogstd_src[i];
      if (theta != nullptr) r += l2c2 * (double)theta[i];
      if (push.world) {
        p2p_push_value(push, i, r);     // this rank's share; the totals are written in phase 2
      } else {
        if (out32) out32[i] = (float)r;
        if (out64) out64[i] = r;
      }
    }
    __syncthreads();                    // acc is reused
  }
  if (push.world == 0) return;
  const unsigned int ticket = p2p_push_done(push);
  // exchange phase: the last RED_GATHER_CTAS CTAs to finish phase 1 stay, everybody else leaves
  const int total = (int)gridDim.x, stay = total < RED_GATHER_CTAS ? total : RED_GATHER_CTAS;
  const int j = (int)ticket - (total - stay);
  if (j < 0) return;
  p2p_wait_flags(ga, sy * RED_PX + px);
  const double* peer = nullptr;          // rank sy's vector (selected without indexing the kernel parameter)
#pragma unroll
  for (int q = 0; q < MRL_P2P_MAX_WORLD; ++q)
    if (q == sy && q < ga.world) peer = ga.src[q];
  for (int c0 = j; c0 < n_chunks; c0 += stay * RED_GB) {
    double v[RED_GB];                    // RED_GB chunks per batch: all NVLink reads in flight before the first sum
#pragma unroll
    for (int u = 0; u < RED_GB; ++u) {
      const int i = (c0 + u * stay) * RED_PX + px;
      v[u] = (peer != nullptr && c0 + u * stay < n_chunks && i < g.P) ? p2p_load(peer + i) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < RED_GB; ++u) {
      const int i = (c0 + u * stay) * RED_PX + px;
      acc[sy][px] = v[u];
      __syncthreads();
      if (sy == 0 && c0 + u * stay < n_chunks && i < g.P) {
        double r = 0.0;
        for (int q = 0; q < ga.world; ++q) r += acc[q][px];   // rank order
        if (out32) out32[i] = (float)r;
        if (out64) out64[i] = r;
      }
      __syncthreads();
    }
  }
}

// loss partials [n_slabs][4] doubles -> out[4] = scale * sums (single block)
__global__ void reduce_losses_kernel(const double* __restrict__ parts, int n_slabs, double scale,
                                     double* __restrict__ out) {
  __shared__ double scratch[32];
  for (int q = 0; q < 4; ++q) {
    double s = 0.0;
    for (int i = threadIdx.x; i < n_slabs; i += blockDim.x) s += parts[(size_t)i * 4 + q];
    s = block_sum(s, scratch);
    if (threadIdx.x == 0) out[q] = s * scale;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------
// Batch repacking (once per bind).  src is the caller's row-major array [N x ncols] (float or
// double, leading dimension ld); dst is tile-major; feature rows [row_off, row_off+ncols_out)
// of each tile are written, columns >= ncols and timesteps >= N as zeros.
template <typename T>
__global__ void pack_tiles_kernel(const T* __restrict__ src, long long ld, int ncols, int ncols_out,
                                  long long N, float* __restrict__ dst, int rows_per_tile, int row_off) {
  __shared__ float tr[MRL_TILE][33];
  const int tile = blockIdx.x;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  for (int r = ty; r < MRL_TILE; r += 8) {
    const long long n = (long long)tile * MRL_TILE + r;
    const int c = c0 + tx;
    float v = 0.f;
    if (n < N && c < ncols) v = (float)src[n * ld + c];
    tr[r][tx] = v;
  }
  __syncthreads();
  for (int cc = ty; cc < 32; cc += 8) {
    const int c = c0 + cc;
    if (c < ncols_out) {
      float* d = dst + ((size_t)tile * rows_per_tile + row_off + c) * MRL_LDT;
      d[tx] = tr[tx][cc];
      d[tx + 32] = tr[tx + 32][cc];
    }
  }
}

// NnVf.preproc (core.py:659-660): feature `col` = (t - offsets[path(t)]) / timestep_limit, written into
// both tensor-core operand copies of the observations (mlp_l1_tc.cu layouts).  Also writes the
// within-path index (int32) for the bit-exact integer contract.
__global__ void time_feature_kernel(const long long* __restrict__ offsets, int n_paths, long long N,
                                    double timestep_limit, int col, int* __restrict__ tindex,
                                    float* __restrict__ XA, int xa_kgroups, float* __restrict__ XG,
                                    int xg_ftiles) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= N) return;
  int lo = 0, hi = n_paths;  // offsets[lo] <= t < offsets[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (offsets[mid] <= t) lo = mid; else hi = mid;
  }
  const long long k = t - offsets[lo];
  const float f = (float)((double)k / timestep_limit);
  if (tindex) tindex[t] = (int)k;
  {  // forward operand: [mtile][kg][khalf][mgroup][8 timesteps][4 features]  (raw fp32, mlp_l1_tc.cu)
    const long long mt = t / 128;
    const int m = (int)(t % 128);
    XA[((size_t)mt * xa_kgroups + (col >> 3)) * 1024 + ((col & 7) >> 2) * 512 + (m >> 3) * 32 + (m & 7) * 4 + (col & 3)] = f;
  }
  {  // gradient operand: [tg][ftile][khalf][fgroup][8 features][4 timesteps]
    const int fm = col % 128;
    XG[((size_t)(t >> 3) * xg_ftiles + col / 128) * 1024 + (int)((t & 7) >> 2) * 512 + (fm >> 3) * 32 + (fm & 7) * 4 + (int)(t & 3)] = f;
  }
}

// ------------------------------------------------------------------------------------ minibatch gather
// dst row i <- src row idx[i] for the three resident layouts of a batch (XA, XG, policy side inputs), on the device:
// a PpoSgd minibatch (ppo.py:194-199) is 128 rows of the batch that is already resident - no host round trip.
// Rows i >= n of the last destination tiles are written as zeros.
__global__ void gather_rows_kernel(const int* __restrict__ idx, int n, long long n_src,
                                   const float* __restrict__ sXA, float* __restrict__ dXA, int xa_kg, int rows_a,
                                   const float* __restrict__ sXG, float* __restrict__ dXG, int xg_ft, int rows_g,
                                   const float* __restrict__ sAux, float* __restrict__ dAux, int naux) {
  const int quads = xa_kg * 2, fpad = xg_ft * 128;
  const long long nA = (long long)rows_a * quads, nG = (long long)rows_g * fpad, nX = (long long)rows_g * naux;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nA) {                       // XA [mtile][kg][khalf][mgroup 16][8][4]: one float4 = 4 features of one timestep
    const int t = (int)(i / quads), q = (int)(i % quads);
    const int kg = q >> 1, kh = q & 1;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < n) {
      const long long ts = idx[t];
      if (ts >= 0 && ts < n_src)
        v = *reinterpret_cast<const float4*>(sXA + ((size_t)(ts / 128) * xa_kg + kg) * 1024 + kh * 512 + ((ts % 128) >> 3) * 32 + (ts & 7) * 4);
    }
    *reinterpret_cast<float4*>(dXA + ((size_t)(t / 128) * xa_kg + kg) * 1024 + kh * 512 + ((t % 128) >> 3) * 32 + (t & 7) * 4) = v;
    return;
  }
  long long j = i - nA;
  if (j < nG) {                       // XG [t/8][ftile][khalf][fgroup 16][8 features][4 timesteps]
    const int t = (int)(j / fpad), f = (int)(j % fpad);
    float v = 0.f;
    if (t < n) {
      const long long ts = idx[t];
      if (ts >= 0 && ts < n_src)
        v = sXG[((size_t)(ts >> 3) * xg_ft + f / 128) * 1024 + ((ts >> 2) & 1) * 512 + ((f % 128) >> 3) * 32 + (f & 7) * 4 + (ts & 3)];
    }
    dXG[((size_t)(t >> 3) * xg_ft + f / 128) * 1024 + ((t >> 2) & 1) * 512 + ((f % 128) >> 3) * 32 + (f & 7) * 4 + (t & 3)] = v;
    return;
  }
  j -= nG;
  if (j < nX && naux > 0) {           // side inputs, tile-major [tile][row][LDT]
    const int t = (int)(j / naux), r = (int)(j % naux);
    float v = 0.f;
    if (t < n) {
      const long long ts = idx[t];
      if (ts >= 0 && ts < n_src) v = sAux[((size_t)(ts / MRL_TILE) * naux + r) * MRL_LDT + ts % MRL_TILE];
    }
    dAux[((size_t)(t / MRL_TILE) * naux + r) * MRL_LDT + t % MRL_TILE] = v;
  }
}
cudaError_t launch_gather_rows(const int* idx, int n, long long n_src, const float* sXA, float* dXA, int xa_kg,
                               const float* sXG, float* dXG, int xg_ft, const float* sAux, float* dAux, int naux,
                               cudaStream_t st) {
  const int n_tiles = (n + MRL_TILE - 1) / MRL_TILE;
  const int rows_a = ((n_tiles + 1) / 2) * 128, rows_g = n_tiles * MRL_TILE;
  const long long total = (long long)rows_a * xa_kg * 2 + (long long)rows_g * xg_ft * 128 + (long long)rows_g * naux;
  gather_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(idx, n, n_src, sXA, dXA, xa_kg, rows_a, sXG, dXG, xg_ft,
                                                                     rows_g, sAux, dAux, naux);
  return cudaGetLastError();
}

// adam_updates (ppo.py:231-258) on the device, float32 like the host version it replaces: m, v, theta in place;
// a_t = lr sqrt(1 - b2^t) / (1 - b1^t) comes from the host (one float), epsilon is not bias-corrected.
__global__ void adam_step_kernel(int P, const double* __restrict__ g64, float* __restrict__ theta, float* __restrict__ m,
                                 float* __restrict__ v, float a_t, float b1, float b2, float eps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const float g = (float)g64[i];
  const float mi = __fadd_rn(__fmul_rn(b1, m[i]), __fmul_rn(1.f - b1, g));
  const float vi = __fadd_rn(__fmul_rn(b2, v[i]), __fmul_rn(__fmul_rn(1.f - b2, g), g));
  m[i] = mi;
  v[i] = vi;
  theta[i] = __fsub_rn(theta[i], __fdiv_rn(__fmul_rn(a_t, mi), __fadd_rn(__fsqrt_rn(vi), eps)));
}
cudaError_t launch_adam_step(int P, const double* g64, float* theta, float* m, float* v, float a_t, float b1, float b2,
                             float eps, cudaStream_t st) {
  adam_step_kernel<<<(P + 255) / 256, 256, 0, st>>>(P, g64, theta, m, v, a_t, b1, b2, eps);
  return cudaGetLastError();
}
__global__ void accum_losses_kernel(const double* __restrict__ scal, double* __restrict__ acc) {
  if (threadIdx.x < 3) acc[threadIdx.x] += scal[threadIdx.x];
  if (threadIdx.x == 3) acc[3] += 1.0;
}
cudaError_t launch_accum_losses(const double* scal, double* acc, cudaStream_t st) {
  accum_losses_kernel<<<1, 32, 0, st>>>(scal, acc);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ launchers
cudaError_t launch_pack_params(const NetGeom& g, const float* theta, float* img, float* WB, cudaStream_t st) {
  const int nu = l1tc_nu(g);
  const int n = g.d0p * nu + g.img_floats;
  pack_params_kernel<<<(n + 255) / 256, 256, 0, st>>>(g, theta, img, WB, nu);
  return cudaGetLastError();
}

cudaError_t launch_reduce_partials(const NetGeom& g, const float* part1, const float* partm, int n_slabs,
                                   double scale, const float* theta, double l2c2, const float* vflat, double vls,
                                   float* out32, double* out64, const P2pPush* push, const P2pGather* gather,
                                   cudaStream_t st) {
  P2pPush no_push;
  no_push.world = 0;
  P2pGather no_gather;
  no_gather.world = 0;
  const int n_chunks = (g.P + RED_PX - 1) / RED_PX;
  int grid = n_chunks;
  // the kernel that pushes this rank's share also gathers the sum over ranks
  if ((push == nullptr) != (gather == nullptr) || (push && gather->world != push->world)) return cudaErrorInvalidValue;
  reduce_partials_kernel<<<grid, dim3(RED_PX, RED_SY), 0, st>>>(g, part1, partm, n_slabs, scale, theta, l2c2, vflat, vls, out32,
                                                             out64, push ? *push : no_push, gather ? *gather : no_gather);
  return cudaGetLastError();
}

cudaError_t launch_reduce_losses(const double* parts, int n_slabs, double scale, double* out, cudaStream_t st) {
  reduce_losses_kernel<<<1, 256, 0, st>>>(parts, n_slabs, scale, out);
  return cudaGetLastError();
}

cudaError_t launch_pack_tiles(const void* src, int dtype, long long ld, int ncols, int ncols_out, long long N,
                              float* dst, int rows_per_tile, int row_off, int n_tiles, cudaStream_t st) {
  dim3 grid(n_tiles, (ncols_out + 31) / 32), block(32, 8);
#define PT(T) pack_tiles_kernel<T><<<grid, block, 0, st>>>((const T*)src, ld, ncols, ncols_out, N, dst, rows_per_tile, row_off)
  switch (dtype) {   // MRL_F32, MRL_F64, MRL_I32, MRL_I64
    case 0: PT(float); break;
    case 1: PT(double); break;
    case 2: PT(int); break;
    default: PT(long long); break;
  }
#undef PT
  return cudaGetLastError();
}

cudaError_t launch_time_feature(const long long* offsets, int n_paths, long long N, double limit, int col, int* tindex,
                                float* XA, int xa_kgroups, float* XG, int xg_ftiles, cudaStream_t st) {
  time_feature_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(offsets, n_paths, N, limit, col, tindex, XA,
                                                                   xa_kgroups, XG, xg_ftiles);
  return cudaGetLastError();
}
