// Fisher-vector product of layers >= 2 on the 5th-generation tensor cores (tcgen05 + TMEM), split-precision 3xTF32:
// R-forward (Pearlmutter), Fisher metric at the head, reverse sweep, hidden-layer weight / bias gradient partials and
// the delta_1 operand of the layer-1 gradient GEMM (trpo.py:45-58; SURVEY A.3).  On tcgen05 because a warp-level
// mma.sync chain (as in mlp_chain.cu) was issue-bound on the legacy tensor path for the Fvp.
//
// One CTA (16 warps) walks 128-timestep tiles (M = 128 = the TMEM lanes) of its slab.  Every GEMM of the chain runs in
// TS mode: the A operand (activations of the 128 timesteps) is written into tensor memory by the epilogue warps that
// produced it, as (hi, lo) TF32 pairs, the B operand (weights, pre-split on the host side of the launch into the UMMA
// K-major core-matrix order) is streamed from L2 through a shared-memory ring by bulk async copies:
//
//   stage 0         Rz_2  = [Rh_1 | h_1] . [W_2 ; V_2]         Rh_1 = act'(h_1) (x.V_1 + vb_1),  x.V_1 from l1_forward_tc
//   stage l-2       Rz_l  = [Rh_{l-1} | h_{l-1}] . [W_l ; V_l]  ... l = 3..L
//   stage L-1       d_{L-1}' = delta_L . W_L^T                  delta_L = M (Rz_L + vb_L)   (Fisher metric of the head)
//   ...             d_{l-1}' = delta_l . W_l^T                  delta_l = d_l' * act'(h_l)
//   final           delta_1 -> DG (HBM, operand of l1_grad_tc_kernel) + layer-1 bias partials
//
// An epilogue thread owns ONE timestep (its TMEM lane) and all features of it, so head metrics need no shuffles.
// The A operand of a stage is handed over in slots of 16 features through a two-slot TMEM ring (one slot per epilogue
// warp group), so the MMAs of a stage start while its A operand is still being produced.
//
// Hidden-layer weight gradients G_l = h_{l-1}^T delta_l (K = timesteps) need the transposed orientation.  delta_l is
// written by the epilogue threads into shared memory as the (hi, lo) K-major B operand [n][timestep]; h_{l-1}^T goes
// to tensor memory through four converter warps whose lanes are FEATURE rows (they read the tile-major activation
// cache, where a feature's timesteps are contiguous); a second MMA-issuing warp accumulates the (k) tiles over the whole
// slab in TMEM.  A row of ones in each (k) tile yields the bias gradients.  Several layers share one 128-row tile when
// their rows fit (Humanoid: h_2 and h_3 against [delta_3 | delta_4]).
//
// Warp roles (512 threads): 0 producer of the weight ring, 1 chain MMA
// issuer (+ TMEM allocation), 2 (k) MMA issuer, 3 idle, 4-7 / 8-11 epilogue groups 0 / 1 (TMEM lane quarter = warp % 4),
// 12-15 converters.  All hand-overs are mbarriers with a spin watchdog: a protocol bug traps, it never hangs the GPU.
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"
#include <string.h>

#define FT_THREADS 768        // 24 warps: 4 control, 8 R-phase epilogue, 8 delta-phase epilogue, 4 converters
#define FT_RSTAGES 3          // weight ring of the R-forward GEMMs (two k-groups of W_l and V_l per stage)
#define FT_DSTAGES 3          // weight ring of the delta GEMMs (two k-groups of a W_l^T column chunk per stage)
#define FT_KSLOTS 4           // (k) A-operand slots (8 timesteps x one tile = 16 TMEM columns each)
#define FT_MAX_R 3
#define FT_MAX_D 6
#define FT_MAX_PASS 3
#define FT_TMEM_COLS 512

struct FtRStage {   // Rz_l = [Rh_{l-1} | h_{l-1}] . [W_l ; V_l]
  int l, kgs, N, acc_col, w_off, v_off;
};
struct FtDStage {   // d_{l-1}'[:, col0 : col0 + N] = delta_l . W_l^T[:, chunk]
  int l, kgs, N, col0, acc_col, w_off;
};
struct FtPlan {
  int L, nR, nD;
  int Kg[MRL_MAX_LAYERS + 1], Np[MRL_MAX_LAYERS + 1];   // k-groups (round8 / 8) and MMA N (round16) of layers 1..L
  int vboff[MRL_MAX_LAYERS + 1];             // offset of layer l's tangent bias in the shared-memory copy
  FtRStage rs[FT_MAX_R];
  FtDStage ds[FT_MAX_D];
  int dstage_of[MRL_MAX_LAYERS + 1];         // first delta stage with A = delta_l
  int rz_wait_stage;                         // first R stage of a tile that writes the accumulator region of Rz_L
  int rring_col, dring_col, kslot_col;       // TMEM columns: R ring (2 x 32), delta ring (2 x 16), (k) A slots (FT_KSLOTS x 16)
  int rstage_floats, dstage_floats;          // floats per weight ring stage
  int n_pass;                                // (k) tiles
  int pass_N[FT_MAX_PASS], pass_acc[FT_MAX_PASS], pass_buf[FT_MAX_PASS];   // N, TMEM column, float offset of the B buffer
  int pass_first_l[FT_MAX_PASS], pass_last_l[FT_MAX_PASS];                 // first / last produced delta layer (max / min l)
  int lay_pass[MRL_MAX_LAYERS + 1], lay_col[MRL_MAX_LAYERS + 1];           // layer l >= 2: its pass and column in the B tile
  short row_cache[FT_MAX_PASS][128];         // cache feature row of (k) tile row m; -1 none; -2 ones
  short row_lay[FT_MAX_PASS][128];           // layer l whose W_l gradient the row feeds
  short row_f[FT_MAX_PASS][128];             // in-feature index
  int wc_floats, vc_floats, kbuf_floats, smem_bytes;
};

// hi = rna_tf32(x) (integer rounding), lo = x - hi pre-rounded for the tensor core's truncation (mma_tf32.cuh)
__device__ __forceinline__ void ft_split(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi)) + 0x1000u;
}
__device__ __forceinline__ void ft_rot8(uint32_t (&v)[8], int r) {   // v[i] <- v[(i + r) & 7]
  uint32_t a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = (r & 1) ? v[(i + 1) & 7] : v[i];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = (r & 2) ? a[(i + 2) & 7] : a[i];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = (r & 4) ? v[(i + 4) & 7] : v[i];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = a[i];
}
__device__ __forceinline__ void ft_dbar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 delta-phase warps
// one non-blocking try_wait issued EARLY: its result is consumed after the independent work that follows
__device__ __forceinline__ uint32_t mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n.reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done;
}
// in: a[i] = feature i at this lane's timestep (tq = lane & 3) -> out: a[i] = feature tq at timestep i of the quad
__device__ __forceinline__ void ft_quad_transpose(float (&a)[4], int lane) {
  const bool up = lane & 2;
  const float s0 = up ? a[0] : a[2], s1 = up ? a[1] : a[3];
  const float r0 = __shfl_xor_sync(0xffffffffu, s0, 2), r1 = __shfl_xor_sync(0xffffffffu, s1, 2);
  if (!up) { a[2] = r0; a[3] = r1; }   // [f0@t, f1@t, f0@t+2, f1@t+2]
  else { a[0] = r0; a[1] = r1; }       // [f2@t-2, f3@t-2, f2@t, f3@t]
  const bool odd = lane & 1;
  const float q0 = odd ? a[0] : a[1], q1 = odd ? a[2] : a[3];
  const float p0 = __shfl_xor_sync(0xffffffffu, q0, 1), p1 = __shfl_xor_sync(0xffffffffu, q1, 1);
  if (!odd) { a[1] = p0; a[3] = p1; }                          // [F@0, F@1, F@2, F@3]
  else { a[0] = p0; const float t = a[1]; a[1] = t; a[2] = p1; }   // [F@0 (recv), F@1 (own a[1]), F@2 (recv), F@3 (own a[3])]
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// Register redistribution between the warp roles (all four warps of a warpgroup execute the same instruction): the
// launch gives every thread 128 registers (512 threads = the whole register file); the control warps and the
// converters hand most of theirs back, the epilogue warps - which keep prefetched activations in registers to hide
// the L2 latency - take them.
#define FT_REGS_CTRL 32
#define FT_REGS_CONV 72
#define FT_REGS_EPI 88
template <int N> __device__ __forceinline__ void ft_reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void ft_reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
static_assert(4 * 32 * FT_REGS_CTRL + 4 * 32 * FT_REGS_CONV + 16 * 32 * FT_REGS_EPI <= FT_THREADS * 80, "register pool of the launch (80 registers per thread)");

struct FtArgs {
  const float* WC;      // chain weight images of theta
  const float* VC;      // tangent weight images
  const float* vflat;   // tangent, flat (biases are read from it)
  const float* logstd;  // theta image logstd block (DiagGauss) or nullptr
  const float* Zt;      // x . V_1, tile-major [tile][d1][LDT]
  const float* cache;   // activations of theta, tile-major [tile][act_rows][LDT]
  float* DG;            // delta_1 operand of the layer-1 gradient GEMM, K-major raw fp32: [t/8][khalf][n/8][8 n][4 t]
  float* partm;         // [n_slabs][pmid]
  long long N;
  int n_tiles, n_mtiles, slab_mt, n_slabs, nu;
};

template <int ACT>
__global__ void __launch_bounds__(FT_THREADS, 1) fvp_tc_kernel(NetGeom g, FtPlan P, FtArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* rw_full = bars;                       // [FT_RSTAGES] R weight stage landed
  uint64_t* rw_empty = rw_full + FT_RSTAGES;      // [FT_RSTAGES]
  uint64_t* dw_full = rw_empty + FT_RSTAGES;      // [FT_DSTAGES]
  uint64_t* dw_empty = dw_full + FT_DSTAGES;      // [FT_DSTAGES]
  uint64_t* ra_full = dw_empty + FT_DSTAGES;      // [2] R ring slot written (the 4 warps of its group)
  uint64_t* ra_empty = ra_full + 2;               // [2]
  uint64_t* da_full = ra_empty + 2;               // [2] delta ring slot
  uint64_t* da_empty = da_full + 2;               // [2]
  uint64_t* racc_full = da_empty + 2;             // [FT_MAX_R] accumulator of R stage complete (the last one = Rz_L)
  uint64_t* dacc_full = racc_full + FT_MAX_R;     // [FT_MAX_D]
  uint64_t* rz_free = dacc_full + FT_MAX_D;       // [1] the head has read Rz_L (8 warps)
  uint64_t* kconv = rz_free + 1;                  // [FT_KSLOTS]
  uint64_t* kempty = kconv + FT_KSLOTS;           // [FT_KSLOTS]
  uint64_t* d_full = kempty + FT_KSLOTS;          // [FT_MAX_PASS] delta blocks of a (k) pass in shared memory (8 warps)
  uint64_t* d_free = d_full + FT_MAX_PASS;        // [FT_MAX_PASS]
  uint64_t* gacc_full = d_free + FT_MAX_PASS;     // [1]
  uint64_t* gacc_empty = gacc_full + 1;           // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gacc_empty + 1);
  float* vb_s = reinterpret_cast<float*>(smem_raw + 512);       // tangent biases [vboff[l] + j], 512 floats
  float* ivar_s = vb_s + 512;                                   // 64 floats
  float* gb1s = ivar_s + 64;                                    // [8 delta-phase warps][128] layer-1 bias partials
  float* rring = reinterpret_cast<float*>(smem_raw + 8192);     // [FT_RSTAGES][rstage_floats]
  float* dring = rring + (size_t)FT_RSTAGES * P.rstage_floats;  // [FT_DSTAGES][dstage_floats]
  float* kbuf = dring + (size_t)FT_DSTAGES * P.dstage_floats;   // (k) B operands: per pass [hi | lo][ngroup][32 k-chunks][8][4]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = P.L, nR = P.nR, nD = P.nD;

  if (threadIdx.x == 0) {
    for (int i = 0; i < FT_RSTAGES; ++i) { mbar_init(&rw_full[i], 1); mbar_init(&rw_empty[i], 1); }
    for (int i = 0; i < FT_DSTAGES; ++i) { mbar_init(&dw_full[i], 1); mbar_init(&dw_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&ra_full[i], 4); mbar_init(&ra_empty[i], 1);
      mbar_init(&da_full[i], 4); mbar_init(&da_empty[i], 1);
    }
    for (int i = 0; i < FT_MAX_R; ++i) mbar_init(&racc_full[i], 1);
    for (int i = 0; i < FT_MAX_D; ++i) mbar_init(&dacc_full[i], 1);
    mbar_init(rz_free, 8);
    for (int i = 0; i < FT_KSLOTS; ++i) { mbar_init(&kconv[i], 4); mbar_init(&kempty[i], 1); }
    for (int i = 0; i < FT_MAX_PASS; ++i) { mbar_init(&d_full[i], 8); mbar_init(&d_free[i], 1); }
    mbar_init(gacc_full, 1);
    mbar_init(gacc_empty, 4);
    fence_barrier_init();
  }
  // tangent biases, 1/sigma^2, zeroed bias partials and (k) operand buffers (their padding columns stay zero)
  for (int i = threadIdx.x; i < 512; i += FT_THREADS) vb_s[i] = 0.f;
  for (int i = threadIdx.x; i < 8 * 128; i += FT_THREADS) gb1s[i] = 0.f;
  for (int i = threadIdx.x; i < P.kbuf_floats; i += FT_THREADS) kbuf[i] = 0.f;
  __syncthreads();
  for (int l = 1; l <= L; ++l)
    for (int j = threadIdx.x; j < g.d[l]; j += FT_THREADS) vb_s[P.vboff[l] + j] = a.vflat[g.off_flat_b[l] + j];
  for (int j = threadIdx.x; j < 64; j += FT_THREADS)
    ivar_s[j] = (g.head == MRL_HEAD_GAUSS && j < g.d[L]) ? expf(-2.f * a.logstd[j]) : 0.f;
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)FT_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  fence_proxy_async();     // the zeroed (k) buffers are read by the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const size_t tile_c = (size_t)g.act_rows * MRL_LDT;   // floats per 64-timestep cache tile
  const size_t tile_z = (size_t)g.d[1] * MRL_LDT;
  // tiles of this CTA, in order: slabs blockIdx.x, + gridDim.x, ...; every role walks the same sequence
#define FT_FOR_TILES(...)                                                                    \
  for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x) {                         \
    const int mt0 = slab * a.slab_mt, mt1 = min(mt0 + a.slab_mt, a.n_mtiles);                \
    for (int mt = mt0; mt < mt1; ++mt) { __VA_ARGS__ }                                       \
  }

  if (warp < 4) {
  ft_reg_dec<FT_REGS_CTRL>();
  if (warp == 0) {
    // ================================================================ producer: both weight rings
    // The two rings drain at unrelated rates (R phase of tile i + 1 next to the delta phase of tile i), so the one
    // producer thread never blocks on either: it probes both and refills whichever has a free stage.
    // No L2 prefetch of the next tile's activations: it competes with the demand loads (1 M Humanoid timesteps: none
    // 1.04 ms, one bulk prefetch per tile 1.07, 16 KB pieces 1.22).
    if (lane == 0) {
      long long total_tiles = 0;
      for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x)
        total_tiles += min(slab * a.slab_mt + a.slab_mt, a.n_mtiles) - slab * a.slab_mt;
      int r_per = 0, d_per = 0;                      // ring stages (pairs of k-groups) per tile
      for (int r = 0; r < nR; ++r) r_per += (P.rs[r].kgs + 1) >> 1;
      for (int k = 0; k < nD; ++k) d_per += (P.ds[k].kgs + 1) >> 1;
      long long r_left = total_tiles * r_per, d_left = total_tiles * d_per;
      uint32_t rc = 0, dc = 0;                       // stages issued so far
      int rst = 0, rkg = 0, dst_ = 0, dkg = 0;       // position inside the tile
      while (r_left > 0 || d_left > 0) {
        bool progressed = false;
        if (r_left > 0) {
          const int ws = rc % FT_RSTAGES;
          if (mbar_probe(&rw_empty[ws], ((rc / FT_RSTAGES) & 1) ^ 1)) {
            const FtRStage st = P.rs[rst];
            const int kgf = 2 * st.N * 8;                       // floats per k-group of one image (hi | lo)
            const int nk = min(2, st.kgs - rkg);
            float* dst = rring + (size_t)ws * P.rstage_floats;
            mbar_expect_tx(&rw_full[ws], 2u * nk * kgf * 4u);
            bulk_g2s(dst, a.WC + st.w_off + (size_t)rkg * kgf, nk * kgf * 4u, &rw_full[ws]);
            bulk_g2s(dst + 2 * kgf, a.VC + st.v_off + (size_t)rkg * kgf, nk * kgf * 4u, &rw_full[ws]);
            ++rc; --r_left; progressed = true;
            rkg += 2;
            if (rkg >= st.kgs) { rkg = 0; if (++rst == nR) rst = 0; }
          }
        }
        if (d_left > 0) {
          const int ws = dc % FT_DSTAGES;
          if (mbar_probe(&dw_empty[ws], ((dc / FT_DSTAGES) & 1) ^ 1)) {
            const FtDStage st = P.ds[dst_];
            const int kgf = 2 * st.N * 8;
            const int nk = min(2, st.kgs - dkg);
            mbar_expect_tx(&dw_full[ws], nk * kgf * 4u);
            bulk_g2s(dring + (size_t)ws * P.dstage_floats, a.WC + st.w_off + (size_t)dkg * kgf, nk * kgf * 4u, &dw_full[ws]);
            ++dc; --d_left; progressed = true;
            dkg += 2;
            if (dkg >= st.kgs) { dkg = 0; if (++dst_ == nD) dst_ = 0; }
          }
        }
        if (!progressed) __nanosleep(200);
      }
    }
  } else if (warp == 1) {
    // ================================================================ R-phase MMA issuer
    const uint32_t desc_hi = (uint32_t)(umma_desc(0, 0, 128) >> 32);
    const uint32_t ring_u32 = smem_u32(rring);
    uint32_t wc = 0, u = 0, tcount = 0;
    for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x) {
      const int mt0 = slab * a.slab_mt, mt1 = min(mt0 + a.slab_mt, a.n_mtiles);
      for (int mt = mt0; mt < mt1; ++mt) {
      for (int r = 0; r < nR; ++r) {
        const FtRStage st = P.rs[r];
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(st.N >> 3) << 17) | ((128u >> 4) << 24);
        const uint32_t lbo = (uint32_t)st.N * 16u;          // bytes between the two K halves of a B k-group
        const uint32_t kgb = (uint32_t)st.N * 64u;          // bytes per k-group of one image (hi | lo)
        const uint32_t d_tmem = tmem_base + st.acc_col;
        if (r == P.rz_wait_stage) {                         // the previous tile's Rz_L lives in this region until the head has read it
          mbar_wait_sleep(rz_free, (tcount & 1) ^ 1);
          tc_fence_after();
        }
        for (int kg0 = 0; kg0 < st.kgs; kg0 += 2, ++wc) {
          const int ws = wc % FT_RSTAGES, nk = min(2, st.kgs - kg0);
          mbar_wait_sleep(&rw_full[ws], (wc / FT_RSTAGES) & 1);
          const uint32_t bw = umma_desc_lo(ring_u32 + (uint32_t)ws * (uint32_t)P.rstage_floats * 4u, lbo);
          for (int c = 0; c < nk; ++c, ++u) {
            const int e = u & 1;
            mbar_wait_sleep(&ra_full[e], (u >> 1) & 1);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t bW = bw + ((c * kgb) >> 4), bV = bw + ((2 * kgb + c * kgb) >> 4);
              const uint32_t tr = tmem_base + P.rring_col + 32 * e, th = tr + 16;   // [Rh hi 8 | Rh lo 8 | h hi 8 | h lo 8]
              umma_tf32_ts(d_tmem, tr + 8, bW, desc_hi, idesc, (kg0 + c) ? 1u : 0u);   // Rh_lo . W_hi
              umma_tf32_ts(d_tmem, tr, bW + (kgb >> 5), desc_hi, idesc, 1u);           // Rh_hi . W_lo
              umma_tf32_ts(d_tmem, tr, bW, desc_hi, idesc, 1u);                        // Rh_hi . W_hi
              umma_tf32_ts(d_tmem, th + 8, bV, desc_hi, idesc, 1u);                    // h_lo . V_hi
              umma_tf32_ts(d_tmem, th, bV + (kgb >> 5), desc_hi, idesc, 1u);           // h_hi . V_lo
              umma_tf32_ts(d_tmem, th, bV, desc_hi, idesc, 1u);                        // h_hi . V_hi
              tc_commit(&ra_empty[e]);
              if (c + 1 == nk) tc_commit(&rw_empty[ws]);
              if (kg0 + c + 1 == st.kgs) tc_commit(&racc_full[r]);
            }
            __syncwarp();
          }
        }
      }
      ++tcount;
    }
    }
  } else if (warp == 2) {
    // ================================================================ delta-phase MMA issuer
    const uint32_t desc_hi = (uint32_t)(umma_desc(0, 0, 128) >> 32);
    const uint32_t ring_u32 = smem_u32(dring);
    uint32_t wc = 0, u = 0;
    for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x) {
      const int mt0 = slab * a.slab_mt, mt1 = min(mt0 + a.slab_mt, a.n_mtiles);
      for (int mt = mt0; mt < mt1; ++mt) {
      for (int k = 0; k < nD; ++k) {
        const FtDStage st = P.ds[k];
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(st.N >> 3) << 17) | ((128u >> 4) << 24);
        const uint32_t lbo = (uint32_t)st.N * 16u;
        const uint32_t kgb = (uint32_t)st.N * 64u;
        const uint32_t d_tmem = tmem_base + st.acc_col;
        for (int kg0 = 0; kg0 < st.kgs; kg0 += 2, ++wc) {
          const int ws = wc % FT_DSTAGES, nk = min(2, st.kgs - kg0);
          mbar_wait_sleep(&dw_full[ws], (wc / FT_DSTAGES) & 1);
          const uint32_t bw = umma_desc_lo(ring_u32 + (uint32_t)ws * (uint32_t)P.dstage_floats * 4u, lbo);
          for (int c = 0; c < nk; ++c, ++u) {
            const int e = u & 1;
            mbar_wait_sleep(&da_full[e], (u >> 1) & 1);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t bW = bw + ((c * kgb) >> 4);
              const uint32_t td = tmem_base + P.dring_col + 16 * e;                  // [delta hi 8 | delta lo 8]
              umma_tf32_ts(d_tmem, td + 8, bW, desc_hi, idesc, (kg0 + c) ? 1u : 0u);
              umma_tf32_ts(d_tmem, td, bW + (kgb >> 5), desc_hi, idesc, 1u);
              umma_tf32_ts(d_tmem, td, bW, desc_hi, idesc, 1u);
              tc_commit(&da_empty[e]);
              if (c + 1 == nk) tc_commit(&dw_empty[ws]);
              if (kg0 + c + 1 == st.kgs) tc_commit(&dacc_full[k]);
            }
            __syncwarp();
          }
        }
      }
    }
    }
  } else if (warp == 3) {
    // ================================================================ (k) MMA issuer: G tiles += h^T delta over the slab
    const uint32_t desc_hi = (uint32_t)(umma_desc(0, 0, 4096) >> 32);   // SBO = 32 k-chunks x 128 B between n-groups
    const uint32_t kbuf_u32 = smem_u32(kbuf);
    uint32_t kc = 0, tcount = 0, scount = 0;
    for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x, ++scount) {
      const int mt0 = slab * a.slab_mt, mt1 = min(mt0 + a.slab_mt, a.n_mtiles);
      mbar_wait_sleep(gacc_empty, (scount & 1) ^ 1);      // the previous slab's accumulators have been flushed
      tc_fence_after();
      for (int mt = mt0; mt < mt1; ++mt, ++tcount) {
        for (int p = 0; p < P.n_pass; ++p) {
          const int Np_ = P.pass_N[p];
          const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(Np_ >> 3) << 17) | ((128u >> 4) << 24);
          const uint32_t d_tmem = tmem_base + P.pass_acc[p];
          const uint32_t bbase = umma_desc_lo(kbuf_u32 + (uint32_t)P.pass_buf[p] * 4u, 128);   // LBO = 128 B: adjacent k-chunks
          const uint32_t lo_off = ((uint32_t)Np_ * 512u) >> 4;                                  // lo half of the buffer
          mbar_wait_sleep(&d_full[p], tcount & 1);          // this tile's delta blocks of the pass are in shared memory
          for (int ks = 0; ks < 16; ++ks, ++kc) {
            const int sl = kc % FT_KSLOTS;
            mbar_wait_sleep(&kconv[sl], (kc / FT_KSLOTS) & 1);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t ta = tmem_base + P.kslot_col + 16 * sl;     // [h^T hi 8 | lo 8]
              const uint32_t db = bbase + ((uint32_t)ks * 256u >> 4);
              const uint32_t first = (mt > mt0 || ks > 0) ? 1u : 0u;
              umma_tf32_ts(d_tmem, ta + 8, db, desc_hi, idesc, first);            // h_lo . d_hi
              umma_tf32_ts(d_tmem, ta, db + lo_off, desc_hi, idesc, 1u);          // h_hi . d_lo
              umma_tf32_ts(d_tmem, ta, db, desc_hi, idesc, 1u);                   // h_hi . d_hi
              tc_commit(&kempty[sl]);
              if (ks == 15) tc_commit(&d_free[p]);
              if (ks == 15 && p == P.n_pass - 1 && mt == mt1 - 1) tc_commit(gacc_full);
            }
            __syncwarp();
          }
        }
      }
    }
  }
  } else if (warp >= 20) {
    // ================================================================ converters: h^T -> tensor memory, slab flush
    ft_reg_dec<FT_REGS_CONV>();
    const int q = warp & 3, m = q * 32 + lane;
    const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t kc = 0, scount = 0;
    for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x, ++scount) {
      const int mt0 = slab * a.slab_mt, mt1 = min(mt0 + a.slab_mt, a.n_mtiles);
      for (int mt = mt0; mt < mt1; ++mt) {
        for (int p = 0; p < P.n_pass; ++p) {
          const int crow = P.row_cache[p][m];
          // the 16 k-steps (8 timesteps each) of the tile in groups of two; group g + 1 is requested before group g is
          // converted, so the L2 latency is covered by the conversion of two k-steps
          float4 xa[2][2], xb[2][2];
          auto request = [&](int g2, float4 (&x)[2][2]) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int ks = 2 * g2 + i, t64 = 2 * mt + (ks >> 3);
              if (crow >= 0 && t64 < a.n_tiles) {
                const float4* src = reinterpret_cast<const float4*>(a.cache + (size_t)t64 * tile_c + (size_t)crow * MRL_LDT + (ks & 7) * 8);
                x[i][0] = __ldg(src);
                x[i][1] = __ldg(src + 1);
              } else {
                const float c = crow == -2 ? 1.f : 0.f;
                x[i][0] = make_float4(c, c, c, c);
                x[i][1] = x[i][0];
              }
            }
          };
          auto convert = [&](const float4 (&xx)[2][2]) {
#pragma unroll
            for (int i = 0; i < 2; ++i, ++kc) {
              const int sl = kc % FT_KSLOTS;
              const uint32_t freeq = mbar_try(&kempty[sl], ((kc / FT_KSLOTS) & 1) ^ 1);
              const float x[8] = {xx[i][0].x, xx[i][0].y, xx[i][0].z, xx[i][0].w, xx[i][1].x, xx[i][1].y, xx[i][1].z, xx[i][1].w};
              uint32_t hi[8], lo[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) ft_split(x[k], hi[k], lo[k]);
              if (!freeq) mbar_wait_ns<200>(&kempty[sl], ((kc / FT_KSLOTS) & 1) ^ 1);
              tc_fence_after();
              const uint32_t ta = tlane + P.kslot_col + 16 * sl;
              tmem_st8(ta, hi);
              tmem_st8(ta + 8, lo);
              asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(&kconv[sl]);
            }
          };
          request(0, xa);
#pragma unroll 1
          for (int g2 = 0; g2 < 8; g2 += 2) {
            request(g2 + 1, xb);
            convert(xa);
            if (g2 + 2 < 8) request(g2 + 2, xa);
            convert(xb);
          }
        }
      }
      // ---- slab flush: accumulator rows -> fp32 slab partial (weights of layers >= 2, their biases from the ones row)
      mbar_wait_ns<500>(gacc_full, scount & 1);
      tc_fence_after();
      float* part = a.partm + (size_t)slab * g.pmid;
      for (int p = 0; p < P.n_pass; ++p) {
        const int crow = P.row_cache[p][m], rl = P.row_lay[p][m], rf = P.row_f[p][m];
        for (int c0 = 0; c0 < P.pass_N[p]; c0 += 8) {
          uint32_t v[8];
          tmem_ld8(tlane + P.pass_acc[p] + c0, v);
          if (crow == -1) continue;
          for (int l = P.pass_last_l[p]; l <= P.pass_first_l[p]; ++l) {
            if (crow >= 0 && l != rl) continue;
            const int col0 = P.lay_col[l];
            float* dst = crow >= 0 ? part + g.off_W[l] + (size_t)rf * g.ldw[l] : part + g.off_b[l];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int n = c0 + j - col0;
              if (n >= 0 && n < g.d[l]) dst[n] = __uint_as_float(v[j]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(gacc_empty);
    }
  } else {
    ft_reg_inc<FT_REGS_EPI>();
    const int q = warp & 3, m = q * 32 + lane;
    const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
    if (warp < 12) {
      // ============================================================== R-phase epilogue: one thread = one timestep
      // Two groups of four warps (one warp per TMEM lane quarter) take alternate k-groups: group e owns ring slot e.  A
      // slot is the A operand [Rh_ul | h_ul] of one k-group (8 features).  The cached activations (and x.V_1 for layer
      // 1) of a group's NEXT k-group are requested before its current one is processed, those of the first before the
      // wait for the previous stage's accumulator; the probe of the slot's empty barrier is issued before the arithmetic.
      const int e = (warp - 4) >> 2;
      const uint32_t ring = tlane + P.rring_col + 32 * e;
      uint32_t u = 0, ue = 0, tcount = 0;
      for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x) {
      const int mt0 = slab * a.slab_mt, mt1 = min(mt0 + a.slab_mt, a.n_mtiles);
      for (int mt = mt0; mt < mt1; ++mt) {
        const int t64c = min(2 * mt + (m >> 6), a.n_tiles - 1);      // a tile beyond the batch reads the last one (masked at the head)
        const float* cb = a.cache + (size_t)t64c * tile_c + (m & 63);
        const float* zb = a.Zt + (size_t)t64c * tile_z + (m & 63);
        for (int r = 0; r < nR; ++r) {
          const int ul = r + 1, kgs = P.rs[r].kgs;
          const float* hrow = cb + (size_t)g.off_act[ul] * MRL_LDT;
          const float* vbl = vb_s + P.vboff[ul];
          float hc[8], zc[8], hn[8], zn[8];                   // current and next k-group of this group
          auto request = [&](int kg, float (&hb)[8], float (&zz)[8]) {
            const float* ph = hrow + (size_t)(8 * kg) * MRL_LDT;
#pragma unroll
            for (int i = 0; i < 8; ++i) hb[i] = __ldg(ph + i * MRL_LDT);
            if (r == 0) {
              const float* pz = zb + (size_t)(8 * kg) * MRL_LDT;
#pragma unroll
              for (int i = 0; i < 8; ++i) zz[i] = __ldg(pz + i * MRL_LDT);
            }
          };
          int kg = (e - (int)(u & 1)) & 1;            // this group's first k-group of the stage
          u += kgs;
          if (kg < kgs) request(kg, hc, zc);
          uint32_t src_acc = 0;
          if (r > 0) {
            mbar_wait_sleep(&racc_full[r - 1], tcount & 1);
            tc_fence_after();
            src_acc = tlane + P.rs[r - 1].acc_col;
          }
          for (; kg < kgs; kg += 2, ++ue) {
            const uint32_t freeq = mbar_try(&ra_empty[e], (ue & 1) ^ 1);
            if (kg + 2 < kgs) request(kg + 2, hn, zn);
            float val[8];
            const float4 vb0 = *reinterpret_cast<const float4*>(vbl + 8 * kg), vb1 = *reinterpret_cast<const float4*>(vbl + 8 * kg + 4);
            const float vbk[8] = {vb0.x, vb0.y, vb0.z, vb0.w, vb1.x, vb1.y, vb1.z, vb1.w};
            if (r == 0) {
#pragma unroll
              for (int i = 0; i < 8; ++i) val[i] = dact_from_h<ACT>(hc[i]) * (zc[i] + vbk[i]);
            } else {
              uint32_t v[8];
              tmem_ld8(src_acc + 8 * kg, v);
#pragma unroll
              for (int i = 0; i < 8; ++i) val[i] = dact_from_h<ACT>(hc[i]) * (__uint_as_float(v[i]) + vbk[i]);
            }
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) ft_split(val[i], hi[i], lo[i]);
            if (!freeq) mbar_wait_sleep(&ra_empty[e], (ue & 1) ^ 1);
            tc_fence_after();
            tmem_st8(ring, hi);
            tmem_st8(ring + 8, lo);
#pragma unroll
            for (int i = 0; i < 8; ++i) ft_split(hc[i], hi[i], lo[i]);
            tmem_st8(ring + 16, hi);
            tmem_st8(ring + 24, lo);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ra_full[e]);
#pragma unroll
            for (int i = 0; i < 8; ++i) { hc[i] = hn[i]; zc[i] = zn[i]; }
          }
        }
        ++tcount;
      }
      }
    } else {
      // ============================================================== delta-phase epilogue: one thread = one timestep
      // head metric -> delta_L, delta_l = d_l' * act'(h_l) (l = L-1 .. 2), delta_1 -> DG + layer-1 bias partial sums.
      // Two groups of four warps take alternate k-groups (group e owns delta ring slot e) and alternate 8-column chunks
      // of delta_1.  delta_l (l >= 2) goes to the delta ring (A operand of the next GEMM) and, as the K-major B operand
      // of the (k) GEMM, to shared memory.  When the last GEMM is split into column chunks, delta_2 is produced once per chunk.
      const int e = (warp - 12) >> 2;
      const uint32_t ring = tlane + P.dring_col + 16 * e;
      float* gb1w = gb1s + (warp - 12) * 128;
      const int rot = (m >> 2) & 7;   // (k) operand stores are rotated against bank conflicts (see below)
      const bool cat = g.head == MRL_HEAD_CAT;
      const int nu = a.nu;
      uint32_t u = 0, ue = 0, tcount = 0;
      for (int slab = blockIdx.x; slab < a.n_slabs; slab += gridDim.x) {
        const int mt0 = slab * a.slab_mt, mt1 = min(mt0 + a.slab_mt, a.n_mtiles);
        for (int mt = mt0; mt < mt1; ++mt, ++tcount) {
          const int t64 = 2 * mt + (m >> 6);
          const bool ok = t64 < a.n_tiles;
          const int t64c = min(t64, a.n_tiles - 1);
          const long long T = (long long)mt * 128 + m;
          const bool valid = T < a.N;
          const float* cb = a.cache + (size_t)t64c * tile_c + (m & 63);
          int k = 0;                                           // delta stage index
          for (int l = L; l >= 2; --l) {
            // chunks of the GEMM that consumes delta_l: one stage, except for the last layer when N_1 > 64
            int nchunk = 0;
            while (k + nchunk < nD && P.ds[k + nchunk].l == l) ++nchunk;
            const int du = g.d[l], kgs = P.Kg[l];
            const float* hrow = cb + (size_t)g.off_act[l] * MRL_LDT;
            const float* vbl = vb_s + P.vboff[l];
            const bool is_head = l == L;
            const bool need_h = !(is_head && !cat);
            const int pass = P.lay_pass[l];
            float* kb = kbuf + P.pass_buf[pass] + (size_t)(P.lay_col[l] >> 3) * 1024 + (m >> 2) * 32 + (m & 3);
            const int lo_off = P.pass_N[pass] * 128;
            for (int c = 0; c < nchunk; ++c, ++k) {
              float hc[8], hn[8];
              auto request = [&](int kg, float (&hb)[8]) {
                if (need_h) {
                  const float* ph = hrow + (size_t)(8 * kg) * MRL_LDT;
#pragma unroll
                  for (int i = 0; i < 8; ++i) hb[i] = __ldg(ph + i * MRL_LDT);
                }
              };
              int kg = (e - (int)(u & 1)) & 1;        // this group's first k-group
              u += kgs;
              if (kg < kgs) request(kg, hc);
              uint32_t src_acc;
              if (c == 0) {
                if (is_head) {
                  mbar_wait_sleep(&racc_full[nR - 1], tcount & 1);
                  src_acc = tlane + P.rs[nR - 1].acc_col;
                } else {
                  mbar_wait_sleep(&dacc_full[k - 1], tcount & 1);
                  src_acc = tlane + P.ds[k - 1].acc_col;
                }
                tc_fence_after();
                if (l == P.pass_first_l[pass]) mbar_wait_sleep(&d_free[pass], (tcount & 1) ^ 1);   // previous tile's (k) MMAs are done
              } else {
                src_acc = tlane + (is_head ? P.rs[nR - 1].acc_col : P.ds[k - c - 1].acc_col);
              }
              float sdot = 0.f;     // Categorical: p . Rz over the whole row
              if (is_head && cat) {
                for (int c0 = 0; c0 < P.Np[L]; c0 += 8) {
                  uint32_t v[8];
                  tmem_ld8(src_acc + c0, v);
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const int f = c0 + i;
                    const float p = f < du ? __ldg(hrow + (size_t)f * MRL_LDT) : 0.f;
                    sdot += p * (__uint_as_float(v[i]) + vbl[f]);
                  }
                }
              }
              for (; kg < kgs; kg += 2, ++ue) {
                const uint32_t freeq = mbar_try(&da_empty[e], (ue & 1) ^ 1);
                if (kg + 2 < kgs) request(kg + 2, hn);
                uint32_t v[8];
                tmem_ld8(src_acc + 8 * kg, v);
                float val[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const int f = 8 * kg + i;
                  const float acc = __uint_as_float(v[i]);
                  float o;
                  if (is_head) {
                    const float rz = acc + vbl[f];
                    o = cat ? hc[i] * (rz - sdot) : rz * ivar_s[f < 64 ? f : 63];      // Fisher metric
                    if (!valid || f >= du) o = 0.f;
                  } else o = acc * dact_from_h<ACT>(hc[i]);                            // padding columns: zero accumulator
                  val[i] = o;
                }
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) ft_split(val[i], hi[i], lo[i]);
                if (!freeq) mbar_wait_sleep(&da_empty[e], (ue & 1) ^ 1);
                tc_fence_after();
                tmem_st8(ring, hi);
                tmem_st8(ring + 8, lo);
                if (c == 0) {
                  // the same block as the K-major B operand of the (k) GEMM: [n][timestep].  In the no-swizzle core-matrix
                  // order the 32 timesteps of a warp at one n hit 4 banks (8-way conflict), so the eight values are
                  // rotated per lane quad and one store instruction hits 32 banks.  The rotation costs 96 select
                  // instructions per k-group, but the plain order measured SLOWER: 1.095 vs 1.046 ms
                  float* kp = kb + (size_t)kg * 1024;
                  ft_rot8(hi, rot);
                  ft_rot8(lo, rot);
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const int nn = ((i + rot) & 7) * 4;
                    kp[nn] = __uint_as_float(hi[i]);
                    kp[nn + lo_off] = __uint_as_float(lo[i]);
                  }
                }
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&da_full[e]);
#pragma unroll
                for (int i = 0; i < 8; ++i) hc[i] = hn[i];
              }
              if (c == 0) {
                if (is_head) {                               // Rz_L has been read: the R phase may overwrite its region
                  tc_fence_before();
                  __syncwarp();
                  if (lane == 0) mbar_arrive(rz_free);
                }
                if (l == P.pass_last_l[pass]) {              // all delta blocks of the pass are written
                  fence_proxy_async();
                  __syncwarp();
                  if (lane == 0) mbar_arrive(&d_full[pass]);
                }
              }
              if (l == 2) {
                // ---- final, chunk c: delta_1 = d_1' * act'(h_1) -> DG (K-major tcgen05 B operand of the layer-1 gradient
                // GEMM as raw fp32, l1_dg_offset; l1_grad_tc_kernel splits it into (hi, lo)) + bias partial
                // sums.  The two groups take alternate 8-column blocks; a 4 x 4 transpose inside each lane quad turns
                // (4 features of my timestep) into (my feature at the quad's 4 timesteps) = one 16-byte store.
                const FtDStage st = P.ds[k];
                const float* h1row = cb + (size_t)g.off_act[1] * MRL_LDT;
                float h1c[8], h1n[8];
                auto request1 = [&](int c0, float (&hb)[8]) {
                  const float* ph = h1row + (size_t)c0 * MRL_LDT;
#pragma unroll
                  for (int i = 0; i < 8; ++i) hb[i] = __ldg(ph + i * MRL_LDT);
                };
                int j0 = 8 * e;
                if (j0 < st.N) request1(st.col0 + j0, h1c);
                mbar_wait_sleep(&dacc_full[k], tcount & 1);
                tc_fence_after();
                const uint32_t facc = tlane + st.acc_col;
                for (; j0 < st.N; j0 += 16) {
                  const int c0 = st.col0 + j0;
                  if (j0 + 16 < st.N) request1(c0 + 16, h1n);
                  uint32_t v[8];
                  tmem_ld8(facc + j0, v);
                  float val[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) val[i] = __uint_as_float(v[i]) * dact_from_h<ACT>(h1c[i]);   // padding columns are zero
#pragma unroll
                  for (int hq = 0; hq < 2; ++hq) {
                    float tq[4] = {val[4 * hq], val[4 * hq + 1], val[4 * hq + 2], val[4 * hq + 3]};
                    ft_quad_transpose(tq, lane);
                    if (ok) {
                      const int n = c0 + 4 * hq + (lane & 3);   // timesteps 4 (T / 4) .. + 3 of feature n
                      *reinterpret_cast<float4*>(a.DG + l1_dg_offset(T >> 3, (T >> 2) & 1, n, nu)) =
                          make_float4(tq[0], tq[1], tq[2], tq[3]);
                    }
                  }
                  // column sums over the warp's 32 timesteps: 8 -> 4 -> 2 -> 1 values per lane, then the quad
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    const float send = (lane & 16) ? val[i] : val[i + 4];
                    const float keep = (lane & 16) ? val[i + 4] : val[i];
                    val[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                  }
#pragma unroll
                  for (int i = 0; i < 2; ++i) {
                    const float send = (lane & 8) ? val[i] : val[i + 2];
                    const float keep = (lane & 8) ? val[i + 2] : val[i];
                    val[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                  }
                  {
                    const float send = (lane & 4) ? val[0] : val[1];
                    const float keep = (lane & 4) ? val[1] : val[0];
                    val[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                  }
                  val[0] += __shfl_xor_sync(0xffffffffu, val[0], 2);
                  val[0] += __shfl_xor_sync(0xffffffffu, val[0], 1);
                  // lane holds column c0 + 4 b4 + 2 b3 + b2 (b4 = bit 4 of the lane, ...)
                  if ((lane & 3) == 0) gb1w[c0 + ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1)] += val[0];
#pragma unroll
                  for (int i = 0; i < 8; ++i) h1c[i] = h1n[i];
                }
                tc_fence_before();
              }
            }
          }
        }
        // ---- slab end: layer-1 bias partial (fixed order over the 8 delta-phase warps), logstd block = 0 (set by the reduce)
        ft_dbar();
        float* part = a.partm + (size_t)slab * g.pmid;
        const int et = threadIdx.x - 384;              // 0..255 over the delta-phase warps
        for (int f = et; f < g.d[1]; f += 256) {
          float sum = 0.f;
#pragma unroll
          for (int w = 0; w < 8; ++w) sum += gb1s[w * 128 + f];
          part[g.off_b[1] + f] = sum;
        }
        for (int j = et; j < g.d[L]; j += 256) part[g.off_pm_logstd + j] = 0.f;
        ft_dbar();
        for (int f = et; f < 8 * 128; f += 256) gb1s[f] = 0.f;
        ft_dbar();
      }
    }
  }
#undef FT_FOR_TILES
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)FT_TMEM_COLS));
  }
}

// ------------------------------------------------------------------------------------ operand images
// src (flat parameter or tangent vector) -> the B images of the chain stages: per stage [k-group][hi | lo][khalf][n-group
// N/8][8 n][4 k]; R-forward stages hold W_l as B[n = out][k = in], delta stages a column chunk of W_l^T as
// B[n = in - col0][k = out].
struct FtPackJob { int off, N, kgs, l, transposed, col0, end; };
struct FtPackJobs { FtPackJob j[FT_MAX_R + FT_MAX_D]; int n; };
__global__ void ft_pack_kernel(NetGeom g, FtPackJobs jobs, const float* __restrict__ src, float* __restrict__ dst, int total,
                               float* __restrict__ WB1, int nu) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) {
    // the layer-1 operand of the same vector (WB of mlp_l1_tc.cu, l1_wb_offset) in the same launch
    const int j = i - total;
    if (WB1 == nullptr || j >= g.d0p * nu) return;
    const int k = j / nu, n = j % nu;
    const float x = (k < g.d[0] && n < g.d[1]) ? src[g.off_flat_W[1] + k * g.d[1] + n] : 0.f;
    const float h = tf32_rna(x);
    float* base = WB1 + l1_wb_offset(k >> 3, (k & 7) >> 2, n, nu) + (k & 3);
    base[0] = h;
    base[nu * 8] = tf32_rna(x - h);
    return;
  }
  int q = 0, base = 0;
  while (q < jobs.n - 1 && i >= jobs.j[q].end) { base = jobs.j[q].end; ++q; }
  const FtPackJob jb = jobs.j[q];
  const int e = i - base, K = jb.kgs * 8;
  const int n = e / K, k = e % K;
  const int l = jb.l;
  float x = 0.f;
  if (!jb.transposed) {          // n = out unit, k = in unit
    if (n < g.d[l] && k < g.d[l - 1]) x = src[g.off_flat_W[l] + k * g.d[l] + n];
  } else {                       // n + col0 = in unit, k = out unit
    if (n + jb.col0 < g.d[l - 1] && k < g.d[l]) x = src[g.off_flat_W[l] + (n + jb.col0) * g.d[l] + k];
  }
  const float h = tf32_rna(x);
  float* p = dst + jb.off + (size_t)(k >> 3) * (2 * jb.N * 8) + ((k & 7) >> 2) * (jb.N * 4) + (n >> 3) * 32 + (n & 7) * 4 + (k & 3);
  p[0] = h;
  p[jb.N * 8] = tf32_rna(x - h);
}

// ------------------------------------------------------------------------------------ host side
static bool ft_build_plan(const NetGeom& g, FtPlan* P) {
  memset(P, 0, sizeof(*P));
  const int L = g.L;
  if (L < 3 || L > 4) return false;
  if (g.head != MRL_HEAD_GAUSS && g.head != MRL_HEAD_CAT) return false;
  if (g.d[L] > 64) return false;
  P->L = L;
  int vb = 0;
  for (int l = 1; l <= L; ++l) {
    if (g.d[l] > 128) return false;
    if (l >= 2 && g.d[l] > 64) return false;      // accumulators of the inner GEMMs are at most 64 columns wide
    P->Kg[l] = (g.d[l] + 7) / 8;
    P->Np[l] = round_up(g.d[l], 16);
    P->vboff[l] = vb;
    vb += round_up(g.d[l], 16) + 16;      // the epilogue reads k-group-padded entries past d[l]
  }
  if (vb > 512) return false;
  if (P->Np[1] != l1tc_nu(g)) return false;
  // R-forward stages and delta stages (the last GEMM, N = N_1, in column chunks of at most 64) with their B images
  int wc = 0, vc = 0;
  P->nR = L - 1;
  for (int l = 2; l <= L; ++l) {
    FtRStage& st = P->rs[l - 2];
    st.l = l; st.kgs = P->Kg[l - 1]; st.N = P->Np[l];
    st.w_off = wc; st.v_off = vc;
    wc += st.kgs * 2 * st.N * 8;
    vc += st.kgs * 2 * st.N * 8;
    if (2 * 2 * 2 * st.N * 8 > P->rstage_floats) P->rstage_floats = 2 * 2 * 2 * st.N * 8;     // two k-groups x (W, V) x (hi, lo)
  }
  int nD = 0;
  for (int l = L; l >= 2; --l) {
    P->dstage_of[l] = nD;
    const int Nout = P->Np[l - 1];
    for (int col0 = 0; col0 < Nout; col0 += 64) {
      if (nD == FT_MAX_D) return false;
      if (col0 > 0 && l != 2) return false;
      FtDStage& st = P->ds[nD++];
      st.l = l; st.kgs = P->Kg[l]; st.N = Nout - col0 < 64 ? Nout - col0 : 64; st.col0 = col0;
      st.w_off = wc;
      wc += st.kgs * 2 * st.N * 8;
      if (2 * 2 * st.N * 8 > P->dstage_floats) P->dstage_floats = 2 * 2 * st.N * 8;
    }
  }
  P->nD = nD;
  P->wc_floats = wc;
  P->vc_floats = vc;
  // (k) tiles: layers are produced in the order delta_L, ..., delta_2; a tile takes consecutive layers while their input
  // rows plus one row of ones fit into 128 lanes
  int np = 0;
  for (int l = L; l >= 2;) {
    if (np == FT_MAX_PASS) return false;
    int rows = 0, cols = 0, lo_l = l;
    for (int k = l; k >= 2; --k) {
      if (rows + g.d[k - 1] + 1 > 128 || cols + P->Np[k] > 128) break;
      rows += g.d[k - 1];
      cols += P->Np[k];
      lo_l = k;
    }
    if (rows == 0) return false;
    P->pass_first_l[np] = l;
    P->pass_last_l[np] = lo_l;
    P->pass_N[np] = cols;
    for (int m = 0; m < 128; ++m) { P->row_cache[np][m] = -1; P->row_lay[np][m] = 0; P->row_f[np][m] = 0; }
    int m = 0, col = 0;
    for (int k = l; k >= lo_l; --k) {
      P->lay_pass[k] = np;
      P->lay_col[k] = col;
      col += P->Np[k];
      for (int f = 0; f < g.d[k - 1]; ++f, ++m) {
        P->row_cache[np][m] = (short)(g.off_act[k - 1] + f);
        P->row_lay[np][m] = (short)k;
        P->row_f[np][m] = (short)f;
      }
    }
    P->row_cache[np][m] = -2;   // ones
    ++np;
    l = lo_l - 1;
  }
  P->n_pass = np;
  // tensor memory: (k) accumulators | (k) A slots | R accumulators (two alternating regions) | delta accumulators
  // (alternating by layer; the chunks of the last GEMM reuse one region) | R ring | delta ring
  int col = 0;
  for (int p = 0; p < np; ++p) { P->pass_acc[p] = col; col += P->pass_N[p]; }
  P->kslot_col = col;
  col += 16 * FT_KSLOTS;
  int reg[2] = {0, 0};
  for (int r = 0; r < P->nR; ++r) if (P->rs[r].N > reg[r & 1]) reg[r & 1] = P->rs[r].N;
  for (int r = 0; r < P->nR; ++r) P->rs[r].acc_col = col + ((r & 1) ? reg[0] : 0);
  col += reg[0] + reg[1];
  P->rz_wait_stage = (P->nR - 1) & 1;      // first stage of a tile in the same region as the last one
  int dreg[2] = {0, 0};
  for (int k = 0; k < nD; ++k) { const int par = (L - P->ds[k].l) & 1; if (P->ds[k].N > dreg[par]) dreg[par] = P->ds[k].N; }
  for (int k = 0; k < nD; ++k) { const int par = (L - P->ds[k].l) & 1; P->ds[k].acc_col = col + (par ? dreg[0] : 0); }
  col += dreg[0] + dreg[1];
  P->rring_col = col;
  col += 64;
  P->dring_col = col;
  col += 32;
  if (col > FT_TMEM_COLS) return false;
  // shared memory: barriers + small (8 KB) | R weight ring | delta weight ring | (k) B buffers
  int kb = 0;
  for (int p = 0; p < np; ++p) { P->pass_buf[p] = kb; kb += 2 * P->pass_N[p] * 128; }
  P->kbuf_floats = kb;
  P->smem_bytes = 8192 + (FT_RSTAGES * P->rstage_floats + FT_DSTAGES * P->dstage_floats + kb) * 4;
  if (P->smem_bytes > 227 * 1024) return false;
  return true;
}

bool fvp_tc_supported(const NetGeom& g) {
  FtPlan P;
  return g.act == MRL_ACT_TANH && ft_build_plan(g, &P);
}
size_t fvp_tc_image_floats(const NetGeom& g, int tangent) {
  FtPlan P;
  if (!ft_build_plan(g, &P)) return 0;
  return tangent ? P.vc_floats : P.wc_floats;
}
cudaError_t launch_fvp_tc_pack(const NetGeom& g, const float* src_flat, float* dst, int tangent, cudaStream_t st, float* WB1) {
  FtPlan P;
  if (!ft_build_plan(g, &P)) return cudaErrorInvalidConfiguration;
  FtPackJobs jobs;
  memset(&jobs, 0, sizeof(jobs));
  int total = 0;
  for (int r = 0; r < P.nR; ++r) {
    const FtRStage& sg = P.rs[r];
    FtPackJob& jb = jobs.j[jobs.n++];
    jb.off = tangent ? sg.v_off : sg.w_off;
    jb.N = sg.N; jb.kgs = sg.kgs; jb.l = sg.l; jb.transposed = 0; jb.col0 = 0;
    total += sg.N * sg.kgs * 8;
    jb.end = total;
  }
  for (int k = 0; k < P.nD && !tangent; ++k) {
    const FtDStage& sg = P.ds[k];
    FtPackJob& jb = jobs.j[jobs.n++];
    jb.off = sg.w_off;
    jb.N = sg.N; jb.kgs = sg.kgs; jb.l = sg.l; jb.transposed = 1; jb.col0 = sg.col0;
    total += sg.N * sg.kgs * 8;
    jb.end = total;
  }
  const int nu = l1tc_nu(g);
  const int n_all = total + (WB1 ? g.d0p * nu : 0);
  ft_pack_kernel<<<(n_all + 255) / 256, 256, 0, st>>>(g, jobs, src_flat, dst, total, WB1, nu);
  return cudaGetLastError();
}

cudaError_t launch_fvp_tc(const NetGeom& g, const FvpTcArgs& x, cudaStream_t st) {
  FtPlan P;
  if (g.act != MRL_ACT_TANH || !ft_build_plan(g, &P)) return cudaErrorInvalidConfiguration;
  if (x.slab_tiles % 2) return cudaErrorInvalidValue;
  FtArgs a;
  a.WC = x.WC; a.VC = x.VC; a.vflat = x.vflat;
  a.logstd = g.head == MRL_HEAD_GAUSS ? x.img + g.off_pm_logstd : nullptr;
  a.Zt = x.Zt; a.cache = x.cache; a.DG = x.DG; a.partm = x.partm;
  a.N = x.N;
  a.n_tiles = x.n_tiles;
  a.n_mtiles = (x.n_tiles + 1) / 2;
  a.slab_mt = x.slab_tiles / 2;
  a.n_slabs = x.n_slabs;
  a.nu = l1tc_nu(g);
  cudaError_t e = mrl_func_smem((const void*)fvp_tc_kernel<MRL_ACT_TANH>, P.smem_bytes);
  if (e != cudaSuccess) return e;
  const int sms = mrl_sm_count();
  fvp_tc_kernel<MRL_ACT_TANH><<<x.n_slabs < sms ? x.n_slabs : sms, FT_THREADS, P.smem_bytes, st>>>(g, P, a);
  return cudaGetLastError();
}
