// Layer-1 GEMMs on the 5th-generation tensor cores (tcgen05 + TMEM), split-precision 3xTF32.
//
//   l1_forward_tc_kernel : Z1[128 timesteps x NU] = X[128 x d0p] . B[d0p x NU]        (B = W1 or V1)
//
// FP32 parity (1e-5 relative, north_star) rules out plain TF32 (10-bit mantissa).  Every operand is
// used as hi = rna_tf32(x) and lo = x - hi (the tensor core reads the top 19 bits of each) and
// each K=8 step issues three MMAs  D += A_lo.B_hi ; D += A_hi.B_lo ; D += A_hi.B_hi  with FP32
// accumulation in TMEM: per-product error ~2^-21, i.e. FP32-class results at 1/3 of the TF32 rate.
//
// Operands are pre-arranged in HBM in the UMMA canonical K-major / no-swizzle core-matrix order
// (8 rows x 16 bytes per core matrix, SBO = 128 B between row groups, LBO between the two K halves; the B
// operands WB and DG as l1_wb_offset / l1_dg_offset in common.cuh state it),
// so a pipeline stage is filled by 1-D bulk async copies (UBLKCP) with no tensor map.  The observations
// - the only operand that does not fit in L2 - are kept in HBM ONCE, as plain fp32 in that order.
//
// A (the observations) is fed to the tensor core from TENSOR MEMORY (TS-mode tcgen05.mma): four converter
// warps read each landed raw block from shared memory, split it into (hi, lo) in registers and write both with
// tcgen05.st into a ring of TMEM slots; B (weights: small, pre-split hi | lo; delta_1: raw, split in place by the
// same converter warps) stays in shared memory.
// With both operands in shared memory (round 1b/1c-early) the three MMAs of a k-group read 22.5 KB of it and the
// copies + converter another 23 KB: shared-memory bandwidth (128 B/cycle), not the tensor pipe, set the pace.
//   stage (forward):  [A raw fp32: 3 k-groups x 4 KB][B: 3 x (hi | lo) x [khalf 2][ngroup NU/8][8][4]]
//   stage (gradient): [A raw fp32: ftiles x 4 KB][B = delta_1 of 8 timesteps (hi | lo)]
// Warp roles (448 threads): warp 0 = bulk-copy producer (one thread), warp 1 = TMEM allocator + MMA issuer (the
// whole warp walks the loop, one elected lane issues: inside an `if (lane == 0)` region ptxas wraps every
// tcgen05.mma in an ELECT / BRA.U.ANY loop), warps 2..5 = epilogue (tcgen05.ld of their TMEM lane quarter ->
// HBM), warps 6..13 = converters (TC_CGROUPS groups of four, one TMEM lane quarter per warp; stage uses alternate between the groups).  The forward kernel double-
// buffers its accumulator so the epilogue of tile i overlaps the MMAs of tile i+1.  Persistent grid.
// The pipeline was tuned with a clock64 trace of every hand-over in CTA 0 (copy, conversion, mbarrier wake-up and MMA
// issue of each stage); DESIGN.md ("How the layer-1 kernels went from 36 % to 60 %") records what it measured.
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

#define TC_STAGES 12         // pipeline depth: ~4 KB of HBM data per stage must cover a ~4000-cycle round trip
#define TC_CGROUPS 2         // converter groups of four warps (one per TMEM lane quarter).  With `cgroups` = 2 group c
                             // converts the stage uses u = c (mod 2), so the tcgen05.st round trips of consecutive
                             // stages overlap; the rings then have even lengths, every stage / slot (and its 1-bit
                             // phase parity) belongs to ONE group, which visits it in pipeline order as before
#define TC_THREADS (192 + 128 * TC_CGROUPS)
#define TC_M 128

// Converter: `blocks` raw 4 KB operand blocks, contiguous at st -> hi in place, lo `lo_off` bytes behind.
// One warp per stage (converter warp c owns the stages s = c mod TC_CONV, so several stages convert
// concurrently).  The generic-proxy writes are fenced for the async proxy (UMMA).
__device__ __forceinline__ void convert_stage(unsigned char* st, int blocks, uint32_t lo_off, int lane) {
  for (int b = 0; b < blocks; ++b) {
    float4* p = reinterpret_cast<float4*>(st + (size_t)b * 4096) + lane;
    float4* pl = reinterpret_cast<float4*>(st + (size_t)b * 4096 + lo_off) + lane;
    float4 x[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = p[32 * j];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float4 h, l;
#define MRL_SPLIT(X, H, L_)                                                   \
      H = __uint_as_float((__float_as_uint(X) + 0x1000u) & 0xffffe000u);     \
      L_ = __uint_as_float(__float_as_uint(X - H) + 0x1000u);   /* the tensor core truncates: pre-round */
      MRL_SPLIT(x[j].x, h.x, l.x) MRL_SPLIT(x[j].y, h.y, l.y) MRL_SPLIT(x[j].z, h.z, l.z) MRL_SPLIT(x[j].w, h.w, l.w)
#undef MRL_SPLIT
      p[32 * j] = h;
      pl[32 * j] = l;
    }
  }
  fence_proxy_async();
}

// ------------------------------------------------------------------------------------
// XA: [mtile][kg][khalf][mgroup][8][4] raw fp32   WB: [kg][hi|lo][khalf][ngroup][8][4]
__global__ void __launch_bounds__(TC_THREADS, 1) l1_forward_tc_kernel(const float* __restrict__ XA,
                                                                      const float* __restrict__ WB,
                                                                      float* __restrict__ Zt, int kgroups,
                                                                      int xa_kgroups, int nu, int d1, int n_mtiles,
                                                                      int n_tiles, int acc_cols, int n_acc, int tmem_cols,
                                                                      int nstages, int kps, int cgroups) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);       // [TC_STAGES]
  uint64_t* empty = full + TC_STAGES;                           // [TC_STAGES]
  uint64_t* tfull = empty + TC_STAGES;                          // [2]
  uint64_t* tempty = tfull + 2;                                 // [2]
  uint64_t* conv = tempty + 2;                                  // [TC_STAGES]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(conv + TC_STAGES);
  unsigned char* stages = smem_raw + 512;
  // a stage holds kps k-groups (8 features each): [A raw fp32: kps x 4 KB][B: kps x (hi | lo)].  The converter
  // warps move A into tensor memory as (hi, lo): the MMAs then read only B from shared memory - with both
  // operands in shared memory the three MMAs of a k-group read 22.5 KB of it, the converter and the bulk copies
  // another 23 KB, and shared-memory bandwidth (128 B/cycle), not the tensor pipe, set the pace.
  const uint32_t blkA = TC_M * 8 * 4, bytesB = 2 * nu * 8 * 4;
  const uint32_t offB = kps * blkA;
  const uint32_t stage_bytes = offB + kps * bytesB;
  const int spt = (kgroups + kps - 1) / kps;                    // stages per tile
  const uint32_t a_col0 = n_acc * acc_cols;                     // TMEM: accumulators, then the A ring [stage][kg][hi 8 | lo 8]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < nstages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); mbar_init(&conv[s], 4); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 4); }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {   // ---------------- producer: one copy of the raw A blocks, one of the B blocks per stage
      int s = 0, ph = 0;
      for (int mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x) {
        const float* a_src = XA + (size_t)mt * xa_kgroups * (TC_M * 8);
        for (int q = 0; q < spt; ++q) {
          const int kg0 = q * kps, nk = min(kps, kgroups - kg0);
          mbar_wait_guard(&empty[s], ph ^ 1);
          unsigned char* st = stages + (size_t)s * stage_bytes;
          mbar_expect_tx(&full[s], nk * (blkA + bytesB));
          bulk_g2s(st, a_src + (size_t)kg0 * (TC_M * 8), nk * blkA, &full[s]);
          bulk_g2s(st + offB, WB + (size_t)kg0 * (2 * nu * 8), nk * bytesB, &full[s]);
          if (++s == nstages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {                  // ---------------- MMA issuer: the whole warp walks the loop, one elected lane issues
      // instruction descriptor (cute/arch/mma_sm100_desc.hpp InstrDescriptor): D=F32, A=B=TF32, K-major both
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(nu >> 3) << 17) | ((TC_M >> 4) << 24);
      const uint32_t lboB = nu * 4 * 4;   // bytes between the two K halves (l1_wb_offset)
      const uint32_t desc_hi = (uint32_t)(umma_desc(0, 0, 128) >> 32);
      const uint32_t dB0 = umma_desc_lo(smem_u32(stages) + offB, lboB);
      uint32_t tcount = 0;
      int s = 0, ph = 0;
      bool next_ready = false;
      for (int mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x, ++tcount) {
        const int acc = n_acc == 2 ? (tcount & 1) : 0;
        mbar_wait_guard(&tempty[acc], (n_acc == 2 ? ((tcount >> 1) & 1) : (tcount & 1)) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * acc_cols;
        for (int q = 0; q < spt; ++q) {
          const int nk = min(kps, kgroups - q * kps);
          // conv[s] is raised by the converter warps after THEY saw full[s] (A and B land in one transaction), so
          // this one wait covers both operands; every mbarrier wait costs this thread ~170 cycles during which
          // the tensor core idles (its instruction queue holds only ~2 MMAs)
          if (!next_ready) mbar_wait_guard(&conv[s], ph);    // A is in tensor memory as (hi, lo), B in shared memory
          tc_fence_after();
          uint32_t db = dB0 + s * (stage_bytes >> 4);
          uint32_t ta = tmem_base + a_col0 + (uint32_t)(s * kps) * 16;
          if (elect_one()) {
            for (int j = 0; j < nk; ++j) {
              umma_tf32_ts(d_tmem, ta + 8, db, desc_hi, idesc, (q | j) ? 1u : 0u);   // lo.hi: small terms first
              umma_tf32_ts(d_tmem, ta, db + (bytesB >> 5), desc_hi, idesc, 1u);      // hi.lo
              umma_tf32_ts(d_tmem, ta, db, desc_hi, idesc, 1u);                      // hi.hi
              ta += 16;
              db += bytesB >> 4;
            }
            tc_commit(&empty[s]);          // frees the stage (B in shared memory, A in tensor memory)
            if (q == spt - 1) tc_commit(&tfull[acc]);          // accumulator complete
          }
          __syncwarp();
          {   // with MMAs queued, look whether the next stage is converted already (usually it is)
            const int sn = s + 1 == nstages ? 0 : s + 1;
            next_ready = mbar_probe(&conv[sn], s + 1 == nstages ? ph ^ 1 : ph);
          }
          if (++s == nstages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp >= 6) {   // ---------------- converters: raw A rows -> tensor memory (hi, lo)
    const int quarter = warp & 3;          // TMEM lane quarter this warp may access
    const int m = quarter * 32 + lane;     // row of the 128-timestep tile
    const int cgroup = (warp - 6) >> 2;
    int s = cgroup, ph = 0, u = 0;
    for (int mt = blockIdx.x; cgroup < cgroups && mt < n_mtiles; mt += gridDim.x) {
      for (int q = 0; q < spt; ++q, ++u) {
        if ((u & (cgroups - 1)) != cgroup) continue;
        const int nk = min(kps, kgroups - q * kps);
        mbar_wait_guard(&full[s], ph);
        const unsigned char* st = stages + (size_t)s * stage_bytes;
        uint32_t ta = tmem_base + ((uint32_t)(quarter * 32) << 16) + a_col0 + (uint32_t)(s * kps) * 16;
        for (int j = 0; j < nk; ++j) {
          const float4 x0 = *reinterpret_cast<const float4*>(st + (size_t)j * blkA + (size_t)m * 16);          // k 0..3
          const float4 x1 = *reinterpret_cast<const float4*>(st + (size_t)j * blkA + 2048 + (size_t)m * 16);   // k 4..7
          const float x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            hi[k] = (__float_as_uint(x[k]) + 0x1000u) & 0xffffe000u;
            lo[k] = __float_as_uint(x[k] - __uint_as_float(hi[k])) + 0x1000u;   // the tensor core truncates: pre-round
          }
          tmem_st8(ta, hi);
          tmem_st8(ta + 8, lo);
          ta += 16;
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&conv[s]);
        s += cgroups;
        if (s >= nstages) { s -= nstages; ph ^= 1; }
      }
    }
  } else if (warp >= 2 && warp < 6) {   // ---------------- epilogue warps 2..5 -> TMEM lane quarter (warp % 4)
    const int q = warp & 3;
    uint32_t tcount = 0;
    for (int mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x, ++tcount) {
      const int acc = n_acc == 2 ? (tcount & 1) : 0;
      mbar_wait_guard(&tfull[acc], n_acc == 2 ? ((tcount >> 1) & 1) : (tcount & 1));
      tc_fence_after();
      const int r = q * 32 + lane;                 // timestep row inside the 128-row tile
      const int tile = 2 * mt + (r >> 6);
      float* zt = Zt + ((size_t)tile * d1) * MRL_LDT + (r & 63);
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * acc_cols;
      for (int c0 = 0; c0 < nu; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(taddr + c0, v);
        if (tile < n_tiles) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (c0 + j < d1) zt[(size_t)(c0 + j) * MRL_LDT] = __uint_as_float(v[j]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)tmem_cols));
  }
}

// ------------------------------------------------------------------------------------
// part1[slab][f][n] = sum_{t in slab} X[t][f] * delta1[t][n]  on the tensor cores:
// D[128 features x NU] += A[128 x 8 timesteps] . B[NU x 8 timesteps]^T, K = timesteps.
//   XG: [tg = t/8][ftile][khalf][fgroup 16][8 features][4 timesteps]  raw fp32 (split by the converter warps)
//   DG: [tg][khalf][ngroup NU/8][8][4 timesteps]  raw fp32 delta_1 (l1_dg_offset; written by the reverse sweep:
//       fvp_tc_kernel, chain_bwd_kernel, mid_backward_kernel or lw_dg_kernel; split into (hi, lo) in shared memory
//       by the converter warps)
// One CTA accumulates a whole slab (<= 1024 timesteps) for all feature tiles in TMEM (ftiles x
// acc_cols columns), then the epilogue warps store the fp32 partial that reduce_partials_kernel sums
// in fp64.  Same warp roles and stage ring as the forward kernel.
__global__ void __launch_bounds__(TC_THREADS, 1) l1_grad_tc_kernel(const float* __restrict__ XG,
                                                                   const float* __restrict__ DG,
                                                                   float* __restrict__ part1, int ftiles,
                                                                   int xg_ftiles, int nu, int d0, int n1p,
                                                                   int slab_tiles, int n_tiles, int n_slabs,
                                                                   int acc_stride, int tmem_cols, int nss, int nts,
                                                                   int cgroups) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // two rings: nss shared-memory stages (raw A blocks + B) cover the HBM latency; nts tensor-memory slots hold
  // the converted A operand (hi, lo) of the stages the MMA thread is working on - tensor memory is mostly taken
  // by the ftiles accumulators, and a slot only has to live from conversion to the end of its MMAs
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);   // [TC_STAGES] stage landed
  uint64_t* sempty = full + TC_STAGES;                      // [TC_STAGES] stage consumed by its MMAs
  uint64_t* conv = sempty + TC_STAGES;                      // [TC_STAGES] A slot converted
  uint64_t* aempty = conv + TC_STAGES;                      // [TC_STAGES] A slot consumed by its MMAs
  uint64_t* tfull = aempty + TC_STAGES;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 1);
  unsigned char* stages = smem_raw + 512;
  // a stage = one group of 8 timesteps: [A raw fp32: ftiles x 4 KB][B = delta_1 (hi | lo)]; HBM order = stage order.
  // DG holds delta_1 as raw fp32 (half the bytes of a pre-split copy): it lands in the hi block, the converter group
  // of the stage splits it in place and writes lo behind it
  const uint32_t blkA = TC_M * 8 * 4, bytesD = nu * 8 * 4, bytesB = 2 * bytesD;
  const uint32_t offB = ftiles * blkA;
  const uint32_t stage_bytes = offB + bytesB;
  const uint32_t a_col0 = ftiles * acc_stride;              // TMEM: accumulators, then the A ring [slot][ftile][hi 8 | lo 8]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < nss; ++s) { mbar_init(&full[s], 1); mbar_init(&sempty[s], 1); }
    for (int s = 0; s < nts; ++s) { mbar_init(&conv[s], 4); mbar_init(&aempty[s], 1); }
    mbar_init(&tfull[0], 1);
    mbar_init(&tempty[0], 4);
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {   // producer: the raw feature-tile blocks of the timestep group (contiguous), then DG
      int s = 0, ph = 0;
      for (int slab = blockIdx.x; slab < n_slabs; slab += gridDim.x) {
        const int t0 = slab * slab_tiles, t1 = min(t0 + slab_tiles, n_tiles);
        for (int tg = t0 * 8; tg < t1 * 8; ++tg) {
          mbar_wait_guard(&sempty[s], ph ^ 1);
          unsigned char* st = stages + (size_t)s * stage_bytes;
          mbar_expect_tx(&full[s], offB + bytesD);
          bulk_g2s(st, XG + (size_t)tg * xg_ftiles * (TC_M * 8), offB, &full[s]);
          bulk_g2s(st + offB, DG + (size_t)tg * (nu * 8), bytesD, &full[s]);
          if (++s == nss) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {   // MMA issuer: the whole warp walks the loop, one elected lane issues
    // delta_1, the B operand, is K-major: nu x 8 timesteps per stage, hi block then lo block, each
    // [khalf][ngroup nu/8][8 n][4 t] (l1_dg_offset: LBO = the K halves, SBO = 8-row groups)
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(nu >> 3) << 17) | ((TC_M >> 4) << 24);
    const uint32_t lboB = nu * 4 * 4;
    const uint32_t desc_hi = (uint32_t)(umma_desc(0, 0, 128) >> 32);
    const uint32_t dB0 = umma_desc_lo(smem_u32(stages) + offB, lboB);
    int s = 0, a = 0, aph = 0;
    uint32_t scount = 0;
    for (int slab = blockIdx.x; slab < n_slabs; slab += gridDim.x, ++scount) {
      const int t0 = slab * slab_tiles, t1 = min(t0 + slab_tiles, n_tiles);
      mbar_wait_guard(&tempty[0], (scount & 1) ^ 1);
      tc_fence_after();
      for (int tg = t0 * 8; tg < t1 * 8; ++tg) {
        mbar_wait_guard(&conv[a], aph);   // raised after the converters saw full[s]: covers A (tensor memory) and B (split)
        tc_fence_after();
        if (elect_one()) {
          const uint32_t db = dB0 + s * (stage_bytes >> 4);
          const uint32_t ta = tmem_base + a_col0 + (uint32_t)(a * ftiles) * 16;
          const uint32_t d_tmem = tmem_base;
          const uint32_t accf = tg > t0 * 8 ? 1u : 0u;
          // pass by pass over the feature tiles: consecutive MMAs then accumulate into DIFFERENT accumulators
          for (int ft = 0; ft < ftiles; ++ft) umma_tf32_ts(d_tmem + ft * acc_stride, ta + ft * 16 + 8, db, desc_hi, idesc, accf);   // lo.hi
          for (int ft = 0; ft < ftiles; ++ft) umma_tf32_ts(d_tmem + ft * acc_stride, ta + ft * 16, db + (bytesB >> 5), desc_hi, idesc, 1u);   // hi.lo
          for (int ft = 0; ft < ftiles; ++ft) umma_tf32_ts(d_tmem + ft * acc_stride, ta + ft * 16, db, desc_hi, idesc, 1u);   // hi.hi
          tc_commit(&sempty[s]);
          tc_commit(&aempty[a]);
          if (tg + 1 == t1 * 8) tc_commit(&tfull[0]);
        }
        __syncwarp();
        if (++s == nss) s = 0;
        if (++a == nts) { a = 0; aph ^= 1; }
      }
    }
  } else if (warp >= 6) {   // converters: raw A rows -> tensor memory (hi, lo); raw delta_1 -> (hi | lo) in place
    const int quarter = warp & 3;
    const int m = quarter * 32 + lane;
    const int cgroup = (warp - 6) >> 2;
    int s = cgroup, ph = 0, a = cgroup, aph = 0, u = 0;
    for (int slab = blockIdx.x; cgroup < cgroups && slab < n_slabs; slab += gridDim.x) {
      const int t0 = slab * slab_tiles, t1 = min(t0 + slab_tiles, n_tiles);
      for (int tg = t0 * 8; tg < t1 * 8; ++tg, ++u) {
        if ((u & (cgroups - 1)) != cgroup) continue;
        mbar_wait_guard(&full[s], ph);
        mbar_wait_guard(&aempty[a], aph ^ 1);
        tc_fence_after();
        const unsigned char* st = stages + (size_t)s * stage_bytes;
        uint32_t ta = tmem_base + ((uint32_t)(quarter * 32) << 16) + a_col0 + (uint32_t)(a * ftiles) * 16;
        for (int ft = 0; ft < ftiles; ++ft) {
          const float4 x0 = *reinterpret_cast<const float4*>(st + (size_t)ft * blkA + (size_t)m * 16);          // timesteps 0..3
          const float4 x1 = *reinterpret_cast<const float4*>(st + (size_t)ft * blkA + 2048 + (size_t)m * 16);   // timesteps 4..7
          const float x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            hi[k] = (__float_as_uint(x[k]) + 0x1000u) & 0xffffe000u;
            lo[k] = __float_as_uint(x[k] - __uint_as_float(hi[k])) + 0x1000u;   // the tensor core truncates: pre-round
          }
          tmem_st8(ta, hi);
          tmem_st8(ta + 8, lo);
          ta += 16;
        }
        {   // delta_1 (B) in shared memory, while the tensor-memory stores drain: raw -> hi in place, lo one block behind
          float4* pb = reinterpret_cast<float4*>(stages + (size_t)s * stage_bytes + offB);
          for (int i = m; i < 2 * nu; i += TC_M) {
            const float4 x = pb[i];
            uint32_t hi[4], lo[4];
            const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              hi[k] = (__float_as_uint(xs[k]) + 0x1000u) & 0xffffe000u;
              lo[k] = __float_as_uint(xs[k] - __uint_as_float(hi[k])) + 0x1000u;
            }
            pb[i] = make_float4(__uint_as_float(hi[0]), __uint_as_float(hi[1]), __uint_as_float(hi[2]), __uint_as_float(hi[3]));
            pb[i + 2 * nu] = make_float4(__uint_as_float(lo[0]), __uint_as_float(lo[1]), __uint_as_float(lo[2]), __uint_as_float(lo[3]));
          }
          fence_proxy_async();   // generic-proxy writes, read by tcgen05.mma through the async proxy
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&conv[a]);
        s += cgroups;
        if (s >= nss) { s -= nss; ph ^= 1; }
        a += cgroups;
        if (a >= nts) { a -= nts; aph ^= 1; }
      }
    }
  } else if (warp >= 2 && warp < 6) {   // epilogue warps 2..5
    const int q = warp & 3;
    uint32_t scount = 0;
    for (int slab = blockIdx.x; slab < n_slabs; slab += gridDim.x, ++scount) {
      mbar_wait_guard(&tfull[0], scount & 1);
      tc_fence_after();
      for (int ft = 0; ft < ftiles; ++ft) {
        const int f = ft * TC_M + q * 32 + lane;
        float* dst = part1 + ((size_t)slab * d0 + f) * n1p;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + ft * acc_stride;
        for (int c0 = 0; c0 < nu; c0 += 16) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          if (f < d0) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              if (c0 + j < n1p)
                *reinterpret_cast<float4*>(dst + c0 + j) =
                    make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                __uint_as_float(v[j + 3]));
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[0]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)tmem_cols));
  }
}

// ------------------------------------------------------------------------------------ operand packing
// src row-major [N x ld] (float/double) -> XA.  One thread per (timestep, 4 consecutive features).
template <typename T>
__global__ void pack_xa_kernel(const T* __restrict__ src, long long ld, int ncols, long long N, float* __restrict__ XA,
                               int xa_kgroups, long long rows_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int quads = xa_kgroups * 2;
  if (i >= rows_out * quads) return;
  const long long t = i / quads;
  const int kq4 = (int)(i % quads);             // quad index: features 4*kq4 .. +3
  const int kg = kq4 >> 1, khalf = kq4 & 1;
  const long long mt = t / TC_M;
  const int m = (int)(t % TC_M);
  float x[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = 4 * kq4 + j;
    x[j] = (t < N && c < ncols) ? (float)src[t * ld + c] : 0.f;
  }
  float* base = XA + ((size_t)mt * xa_kgroups + kg) * (TC_M * 8) + khalf * (TC_M * 4) + (m >> 3) * 32 + (m & 7) * 4;
  *reinterpret_cast<float4*>(base) = make_float4(x[0], x[1], x[2], x[3]);
}
// src row-major [N x ld] -> XG [tg][ftile][khalf][fgroup][8 features][4 timesteps] (raw fp32).
// One thread per (4 consecutive timesteps, feature).
template <typename T>
__global__ void pack_xg_kernel(const T* __restrict__ src, long long ld, int ncols, long long N, float* __restrict__ XG,
                               int xg_ftiles, long long n_tquads) {
  const int fpad = xg_ftiles * TC_M;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tquads * fpad) return;
  const long long tq = i / fpad;
  const int f = (int)(i % fpad);
  float x[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const long long t = tq * 4 + j;
    x[j] = (t < N && f < ncols) ? (float)src[t * ld + f] : 0.f;
  }
  const long long tg = tq >> 1;
  const int khalf = (int)(tq & 1), ft = f / TC_M, fm = f % TC_M;
  float* base = XG + ((size_t)tg * xg_ftiles + ft) * (TC_M * 8) + khalf * (TC_M * 4) + (fm >> 3) * 32 + (fm & 7) * 4;
  *reinterpret_cast<float4*>(base) = make_float4(x[0], x[1], x[2], x[3]);
}

// ------------------------------------------------------------------------------------ launchers
int l1tc_nu(const NetGeom& g) { return round_up(g.d[1], 16); }
size_t l1tc_wb_floats(const NetGeom& g) { return (size_t)g.d0p * l1tc_nu(g) * 2; }
size_t l1tc_xa_floats(int xa_kgroups, long long n_mtiles) { return (size_t)n_mtiles * xa_kgroups * TC_M * 8; }

cudaError_t launch_l1_forward_tc(const NetGeom& g, const float* XA, int xa_kgroups, const float* WB, float* Zt,
                                 int n_tiles, cudaStream_t st) {
  const int nu = l1tc_nu(g);
  const int acc_cols = nu <= 32 ? 32 : (nu <= 64 ? 64 : (nu <= 128 ? 128 : 256));
  const int n_acc = acc_cols <= 128 ? 2 : 1;     // double-buffered accumulator when tensor memory has room
  // k-groups per stage: one stage hand-over (bulk copies, mbarrier round trips between the producer, converter
  // and MMA threads) costs 500-1000 cycles whatever the copy size (tools/micro/bulk_rate*.cu), so a stage carries
  // several k-groups.  Stage count: shared memory (227 KB) and the tensor-memory A ring (16 columns per k-group
  // behind the accumulators, 512 columns in all).  Measured at 1M x 376 -> 100: one converter group, 5 stages of
  // 3 k-groups 0.447 ms (2: 0.47, 4: 0.42-0.44, 5: 0.44); two groups, 4 stages of 4: 0.437; two groups, 4 x 3: 0.470;
  // two groups, 8 x 2: 0.535.
  int kps = 0, nstages = 0, cgroups = 1;
  for (int pass = 0; pass < 2; ++pass) {
    // first choice: 4 k-groups per stage converted by two groups (needs an even ring of >= 4 stages, see TC_CGROUPS);
    // otherwise 3 per stage and one group
    kps = pass == 0 ? 4 : 3;
    const size_t sb = (size_t)kps * (TC_M * 8 * 4 + 2 * (size_t)nu * 8 * 4);
    nstages = (int)((227 * 1024 - 512) / sb);
    const int tmem_room = (512 - n_acc * acc_cols) / (kps * 16);
    if (nstages > tmem_room) nstages = tmem_room;
    if (nstages > TC_STAGES) nstages = TC_STAGES;
    cgroups = (pass == 0 && nstages >= 4) ? 2 : 1;
    if (cgroups == 2) {
      nstages &= ~1;
      break;
    }
  }
  if (nstages < 2) return cudaErrorInvalidConfiguration;
  const size_t stage_bytes = (size_t)kps * (TC_M * 8 * 4 + 2 * (size_t)nu * 8 * 4);
  int tmem_cols = 32;
  while (tmem_cols < n_acc * acc_cols + nstages * kps * 16) tmem_cols *= 2;
  const size_t smem = 512 + (size_t)nstages * stage_bytes;
  {
    cudaError_t e = mrl_func_smem((const void*)l1_forward_tc_kernel, smem);
    if (e != cudaSuccess) return e;
  }
  const int sms = mrl_sm_count();
  const int n_mtiles = (n_tiles + 1) / 2;
  const int grid = n_mtiles < sms ? n_mtiles : sms;
  l1_forward_tc_kernel<<<grid, TC_THREADS, smem, st>>>(XA, WB, Zt, g.d0p / 8, xa_kgroups, nu, g.d[1], n_mtiles, n_tiles,
                                                       acc_cols, n_acc, tmem_cols, nstages, kps, cgroups);
  return cudaGetLastError();
}

cudaError_t launch_pack_xa(const void* src, int dtype, long long ld, int ncols, long long N, float* XA, int xa_kgroups,
                           long long n_mtiles, cudaStream_t st) {
  const long long rows_out = n_mtiles * TC_M;
  const long long total = rows_out * xa_kgroups * 2;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  if (dtype == 1) pack_xa_kernel<double><<<blocks, 256, 0, st>>>((const double*)src, ld, ncols, N, XA, xa_kgroups, rows_out);
  else pack_xa_kernel<float><<<blocks, 256, 0, st>>>((const float*)src, ld, ncols, N, XA, xa_kgroups, rows_out);
  return cudaGetLastError();
}
size_t l1tc_xg_floats(int xg_ftiles, long long n_tiles) { return (size_t)n_tiles * 8 * xg_ftiles * TC_M * 8; }
size_t l1tc_dg_floats(const NetGeom& g, long long n_tiles) { return (size_t)n_tiles * 8 * l1tc_nu(g) * 8; }

cudaError_t launch_pack_xg(const void* src, int dtype, long long ld, int ncols, long long N, float* XG, int xg_ftiles,
                           long long n_tiles, cudaStream_t st) {
  const long long n_tquads = n_tiles * 16;
  const long long total = n_tquads * xg_ftiles * TC_M;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  if (dtype == 1) pack_xg_kernel<double><<<blocks, 256, 0, st>>>((const double*)src, ld, ncols, N, XG, xg_ftiles, n_tquads);
  else pack_xg_kernel<float><<<blocks, 256, 0, st>>>((const float*)src, ld, ncols, N, XG, xg_ftiles, n_tquads);
  return cudaGetLastError();
}

// tensor-memory plan of the gradient kernel: ftiles accumulators of nu columns, then the A ring
static bool l1g_plan(const NetGeom& g, int* acc_stride, int* nts, int* nss, int* tmem_cols, size_t* smem) {
  const int nu = l1tc_nu(g);
  const int ftiles = (g.d[0] + TC_M - 1) / TC_M;
  *acc_stride = nu;                                   // nu is a multiple of 16
  *nts = (512 - ftiles * nu) / (ftiles * 16);
  if (*nts > TC_STAGES) *nts = TC_STAGES;
  const size_t stage_bytes = (size_t)ftiles * TC_M * 8 * 4 + 2 * (size_t)nu * 8 * 4;
  *nss = (int)((227 * 1024 - 512) / stage_bytes);
  if (*nss > TC_STAGES) *nss = TC_STAGES;
  *tmem_cols = 32;
  while (*tmem_cols < ftiles * nu + *nts * ftiles * 16) *tmem_cols *= 2;
  *smem = 512 + (size_t)*nss * stage_bytes;
  return nu <= 256 && *nts >= 1 && *nss >= 2 && *tmem_cols <= 512;   // one A slot still works (serialised)
}

cudaError_t launch_l1_grad_tc(const NetGeom& g, const float* XG, int xg_ftiles, const float* DG, float* part1,
                              int slab_tiles, int n_tiles, int n_slabs, cudaStream_t st) {
  const int nu = l1tc_nu(g);
  const int ftiles = (g.d[0] + TC_M - 1) / TC_M;
  int acc_stride, nts, nss, tmem_cols;
  size_t smem;
  if (!l1g_plan(g, &acc_stride, &nts, &nss, &tmem_cols, &smem)) return cudaErrorInvalidConfiguration;
  {
    cudaError_t e = mrl_func_smem((const void*)l1_grad_tc_kernel, smem);
    if (e != cudaSuccess) return e;
  }
  const int cgroups = (nts >= 2 && nss >= 4) ? 2 : 1;   // two converter groups need even rings (see TC_CGROUPS)
  if (cgroups == 2) { nts &= ~1; nss &= ~1; }
  const int sms = mrl_sm_count();
  const int grid = n_slabs < sms ? n_slabs : sms;
  l1_grad_tc_kernel<<<grid, TC_THREADS, smem, st>>>(XG, DG, part1, ftiles, xg_ftiles, nu, g.d[0], g.n1p, slab_tiles,
                                                    n_tiles, n_slabs, acc_stride, tmem_cols, nss, nts, cgroups);
  return cudaGetLastError();
}

// nets the tensor-core layer-1 path can hold: TMEM (512 columns) and shared memory (>= 2 stages)
bool l1tc_supported(const NetGeom& g) {
  int acc_stride, nts, nss, tmem_cols;
  size_t smem;
  return l1g_plan(g, &acc_stride, &nts, &nss, &tmem_cols, &smem);
}
