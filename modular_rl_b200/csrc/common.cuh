// Shared declarations for the modular_rl_b200 CUDA kernels (sm_100a only).
//
// Data layout vocabulary (see DESIGN.md "Data layout in HBM"):
//   tile        = 64 consecutive timesteps of the flat batch.
//   tile-major  = [tile][feature][LDT] float, LDT = 68: the 64 timesteps of one feature are
//                 contiguous (+4 pad so that feature rows fall into distinct shared-memory
//                 banks); a tile is one contiguous block, i.e. exactly its shared-memory image.
//   row-major   = [timestep][feature padded] float, as the reference's numpy arrays.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "kernel_defs.cuh"    // MRL_MAX_LAYERS, the head and activation codes, act_fn

#define MRL_TILE 64           // timesteps per tile
#define MRL_LDT 68            // floats between consecutive features inside a tile
#define MRL_MID_THREADS 256
#define MRL_MAX_SLAB_TILES 16 // <=1024 timesteps accumulate in fp32 before the fp64 reduce

enum { MRL_MODE_GRAD = 0, MRL_MODE_FVP = 1, MRL_MODE_GRAD_CLIP = 2 };   // GRAD_CLIP: gradient of the PPO clipped objective

static inline __host__ __device__ int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Geometry of one MLP and of its packed parameter image.  Passed by value to kernels.
struct NetGeom {
  int L;                         // number of Dense layers
  int d[MRL_MAX_LAYERS + 1];     // d[0] = input dim, d[L] = output dim
  int head, act;
  int d0p;                       // d[0] rounded up to 8  (K of the layer-1 GEMM)
  int n1p;                       // d[1] rounded up to 8  (N of the layer-1 GEMM)
  int ldw[MRL_MAX_LAYERS + 1];   // row stride of W_l  [d[l-1] x ldw]   (l >= 2), round4(d[l])
  int ldt[MRL_MAX_LAYERS + 1];   // row stride of W_l^T [d[l] x ldt]    (l >= 2), round4(d[l-1])
  int off_b[MRL_MAX_LAYERS + 1]; // image offsets (floats): bias of layer l (l = 1..L)
  int off_W[MRL_MAX_LAYERS + 1]; // W_l  (l = 2..L)
  int off_WT[MRL_MAX_LAYERS + 1];// W_l^T (l = 2..L)
  int bias_floats;               // size of the bias block  (== off_W[2] or end)
  int bw_floats;                 // bias block + W block     (what forward / tangent images need)
  int img_floats;                // bias + W + WT blocks
  int act_rows;                  // sum_{l=1..L} d[l]  (features cached per timestep)
  int off_act[MRL_MAX_LAYERS + 1]; // feature-row offset of layer l's activations inside a cache tile
  int P;                         // flat parameter count (reference order, SURVEY A.1)
  int off_flat_W[MRL_MAX_LAYERS + 1]; // offsets in the flat vector
  int off_flat_b[MRL_MAX_LAYERS + 1];
  int off_flat_logstd;           // -1 if none
  int naux;                      // feature rows of the per-timestep side inputs (adv/act/oldprob | target)
  int pmid;                      // floats per slab partial written by the mid kernels
  int off_pm_logstd;             // offset of the logstd partial inside a mid partial
};

// B operands of the layer-1 tcgen05 GEMMs (mlp_l1_tc.cu) in HBM, in the UMMA K-major no-swizzle core-matrix order
// over N = nu layer-1 units (a multiple of 8) and K (timesteps for DG, input features for WB), in groups of 8 K:
//   DG  delta_1, raw fp32:            [t/8][khalf][n/8][8 n][4 t]
//   WB  W1 (or V1) split (hi, lo):    [k/8][hi | lo][khalf][n/8][8 n][4 k]   lo sits nu * 8 floats behind hi
// A core matrix is 8 rows of n x 4 consecutive K values (16 B): 32 floats.  Core matrices of consecutive 8-row groups
// are 128 B apart (SBO), the two K halves of a group nu * 16 B apart (LBO); a group of 8 K is one contiguous block of
// nu * 8 floats (WB: twice that, hi then lo), loaded as a whole by one bulk copy.  The offsets locate element n at
// K = 8 * group + 4 * khalf; the caller adds K % 4.
__host__ __device__ __forceinline__ size_t l1_dg_offset(size_t tgroup, int khalf, int n, int nu) {
  return tgroup * (nu * 8) + khalf * (nu * 4) + (n >> 3) * 32 + (n & 7) * 4;
}
__host__ __device__ __forceinline__ size_t l1_wb_offset(size_t kgroup, int khalf, int n, int nu) {
  return kgroup * (2 * nu * 8) + khalf * (nu * 4) + (n >> 3) * 32 + (n & 7) * 4;
}

// ----------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 1-D bulk async copy global -> shared (the TMA engine; SASS: UBLKCP).  bytes % 16 == 0,
// both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------- math helpers
template <int ACT>
__device__ __forceinline__ float dact_from_h(float h) {
  if (ACT == MRL_ACT_TANH) return 1.f - h * h;
  if (ACT == MRL_ACT_RELU) return h > 0.f ? 1.f : 0.f;
  return h * (1.f - h);
}

// g(u) = u - log1p(u) = u^2/2 - u^3/3 + ...  evaluated without the O(u) cancellation.  Both KL
// formulas reduce to sums of g(.) of a relative deviation, which is what keeps a float32 per-row KL
// accurate to 1e-7 RELATIVE even when kl ~ 1e-4 (mean KL is the quantity TRPO constrains).
__device__ __forceinline__ float u_minus_log1p(float u) {
  if (fabsf(u) < 0.2f) {
    float p = 1.f / 12.f;
    p = 1.f / 11.f - u * p; p = 1.f / 10.f - u * p; p = 1.f / 9.f - u * p; p = 1.f / 8.f - u * p;
    p = 1.f / 7.f - u * p;  p = 1.f / 6.f - u * p;  p = 1.f / 5.f - u * p; p = 1.f / 4.f - u * p;
    p = 1.f / 3.f - u * p;  p = 0.5f - u * p;
    return u * u * p;
  }
  return u - log1pf(u);
}

// round-to-nearest TF32 (10-bit mantissa) kept in an fp32 container
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// Sum over the whole block; result valid in thread 0.  `scratch` holds >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  double t = 0.0;
  if (w == 0) {
    t = lane < nw ? scratch[lane] : 0.0;
    t = warp_sum(t);
  }
  return t;
}

// host-side helpers implemented in geom.cu
void mrl_build_geom(NetGeom* g, int n_layers, const int* dims, int head, int act, int naux);
int mrl_sm_count();                                          // SMs of the current device (cached per device)
cudaError_t mrl_func_smem(const void* func, size_t bytes);   // opt in to `bytes` of dynamic shared memory (per device)
