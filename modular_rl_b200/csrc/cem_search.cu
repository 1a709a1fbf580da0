// Device search distribution of the noisy cross-entropy method (cem.py _DeviceGaussianSearch, run_cem.py
// --device_search): the draw of a generation's candidates and the refit of mean and variance to its elite, on the
// device, so that a generation of a built-in environment never leaves the GPU.  DESIGN.md 4b "Device search".
//
// State (api.cu mrl_cem_search): mean and var float64 [P], double-buffered; dev float64 [P]; the candidate rows
// float32 [M][ld], ld >= P a multiple of 4 (16-byte rows).
//
// Candidate m, parameter j: mean[j] + dev[j] * z[m][j] in float64, rounded to float32 for the rollout round.  The
// normals come from Philox4x32-10 keyed by the generation's round seed, counter (m, j / 2, CEM_PURPOSE_DRAW, 0): the
// block's words give u0, u1 and z[m][2p] = r cos(2 pi u1), z[m][2p + 1] = r sin(2 pi u1), r = sqrt(-2 log(1 - u0)).
// Nothing depends on the grid, so a draw is a pure function of (seed, mean, dev).
//
// The refit reads no stored row: it recomputes every elite row in float64 through cem_candidate, the function the draw
// rounded, so the elite statistics are those of the values the host search would hold.  Every product and sum below is
// an explicit _rn intrinsic: no FMA contraction, so the rounding is numpy's.
#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

#include <math.h>

#define CEM_DRAW_THREADS 128
#define CEM_RANK_THREADS 256
#define CEM_REFIT_PAIRS 32      // parameter pairs (64 columns) per refit CTA
#define CEM_REFIT_ROWS 8        // elite rows recomputed at once, one per warp

// The float64 values of candidate m at parameters 2p and 2p + 1 (the second only if 2p + 1 < P).
__device__ __forceinline__ void cem_candidate(int m, int p, uint32_t k0, uint32_t k1, double mean0, double dev0,
                                              double mean1, double dev1, double* x0, double* x1) {
  const uint4 w = philox4x32_10(make_uint4((uint32_t)m, (uint32_t)p, CEM_PURPOSE_DRAW, 0u), k0, k1);
  const double u0 = u53(w.x, w.y), u1 = u53(w.z, w.w);
  const double r = sqrt(__dmul_rn(-2.0, log(__dsub_rn(1.0, u0))));
  double s, c;
  sincospi(__dmul_rn(2.0, u1), &s, &c);           // cos(2 pi u1) with an exact argument: no reduction, no local memory
  *x0 = __dadd_rn(mean0, __dmul_rn(dev0, __dmul_rn(r, c)));
  *x1 = __dadd_rn(mean1, __dmul_rn(dev1, __dmul_rn(r, s)));
}

// dev[j] = sqrt(var[j] + extra_var * noise_left), as _GaussianSearch.draw computes it
__device__ __forceinline__ double cem_dev(double var, double extra_var, double noise_left) {
  return sqrt(__dadd_rn(var, __dmul_rn(extra_var, noise_left)));
}

// grid (pairs / CEM_DRAW_THREADS, M): thread (p, m) writes rows[m][2p], rows[m][2p + 1]; member 0 also writes dev
__global__ void __launch_bounds__(CEM_DRAW_THREADS) cem_draw_kernel(const double* __restrict__ mean,
                                                                    const double* __restrict__ var, double* dev,
                                                                    float* rows, int P, long long ld,
                                                                    double extra_var, double noise_left, uint32_t k0,
                                                                    uint32_t k1) {
  const int p = blockIdx.x * CEM_DRAW_THREADS + threadIdx.x, m = blockIdx.y;
  const int j = 2 * p;
  if (j >= P) return;
  const bool two = j + 1 < P;
  const double d0 = cem_dev(var[j], extra_var, noise_left);
  const double d1 = two ? cem_dev(var[j + 1], extra_var, noise_left) : 0.0;
  double x0, x1;
  cem_candidate(m, p, k0, k1, mean[j], d0, two ? mean[j + 1] : 0.0, d1, &x0, &x1);
  float* row = rows + (size_t)m * ld;
  if (two) {
    *reinterpret_cast<float2*>(row + j) = make_float2((float)x0, (float)x1);   // ld % 4 == 0: 8-byte aligned
  } else {
    row[j] = (float)x0;
  }
  if (m == 0) {
    dev[j] = d0;
    if (two) dev[j + 1] = d1;
  }
}

// Position in np.argsort(scores, kind="stable"): a before b when a < b, or a == b with the lower index; NaN after
// every number, NaNs in index order.
__device__ __forceinline__ bool cem_before(double a, int i, double b, int k) {
  const bool an = isnan(a), bn = isnan(b);
  if (an || bn) return an == bn ? i < k : bn;
  return a < b || (a == b && i < k);
}

// order[0..M - first) = the members of rank first.. in ascending (score, index) order: the elite of
// np.argsort(scores, kind="stable")[first:]
__global__ void __launch_bounds__(CEM_RANK_THREADS) cem_rank_kernel(const double* __restrict__ scores, int M,
                                                                    int first, int* order) {
  extern __shared__ double s_sc[];
  for (int i = threadIdx.x; i < M; i += CEM_RANK_THREADS) s_sc[i] = scores[i];
  __syncthreads();
  const int i = blockIdx.x * CEM_RANK_THREADS + threadIdx.x;
  if (i >= M) return;
  const double si = s_sc[i];
  int rank = 0;
  for (int k = 0; k < M; ++k) rank += cem_before(s_sc[k], k, si, i);
  if (rank >= first) order[rank - first] = i;
}

// grid P / 64 columns: warp w recomputes elite rows w, w + 8, ... for the CTA's 64 columns into shared memory; warp 0
// adds them in elite order.  Pass 1 sums the rows, pass 2 the squared deviations from the new mean (two-pass, ddof 0,
// as best.mean(axis=0) and best.var(axis=0)).
__global__ void __launch_bounds__(CEM_REFIT_PAIRS * CEM_REFIT_ROWS, 4) cem_refit_kernel(
    const double* __restrict__ mean, const double* __restrict__ dev, const int* __restrict__ order, int keep, int P,
    uint32_t k0, uint32_t k1, double* mean_out, double* var_out) {
  __shared__ double s_x[CEM_REFIT_ROWS][2 * CEM_REFIT_PAIRS];
  __shared__ double s_mean[2 * CEM_REFIT_PAIRS];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int p = blockIdx.x * CEM_REFIT_PAIRS + tx, j = 2 * p;
  const bool on = j < P, two = j + 1 < P;
  const double m0 = on ? mean[j] : 0.0, d0 = on ? dev[j] : 0.0;
  const double m1 = two ? mean[j + 1] : 0.0, d1 = two ? dev[j + 1] : 0.0;
  const double n_keep = (double)keep;
  double c0 = 0.0, c1 = 0.0;                       // pass 2: the new mean
  for (int pass = 0; pass < 2; ++pass) {
    double a0 = -0.0, a1 = -0.0;                  // -0.0 + x == x: the sum starts at the first row, as numpy's
    for (int base = 0; base < keep; base += CEM_REFIT_ROWS) {
      const int r = base + ty;
      if (on && r < keep) {
        double x0, x1;
        cem_candidate(order[r], p, k0, k1, m0, d0, m1, d1, &x0, &x1);
        if (pass) {
          x0 = __dsub_rn(x0, c0);
          x1 = __dsub_rn(x1, c1);
          x0 = __dmul_rn(x0, x0);
          x1 = __dmul_rn(x1, x1);
        }
        s_x[ty][2 * tx] = x0;
        s_x[ty][2 * tx + 1] = x1;
      }
      __syncthreads();
      if (ty == 0 && on) {
        const int n = min(CEM_REFIT_ROWS, keep - base);
        for (int q = 0; q < n; ++q) {
          a0 = __dadd_rn(a0, s_x[q][2 * tx]);
          a1 = __dadd_rn(a1, s_x[q][2 * tx + 1]);
        }
      }
      __syncthreads();
    }
    if (ty == 0 && on) {
      a0 = __ddiv_rn(a0, n_keep);
      a1 = __ddiv_rn(a1, n_keep);
      if (pass == 0) {
        s_mean[2 * tx] = a0;
        s_mean[2 * tx + 1] = a1;
      } else {
        var_out[j] = a0;
        if (two) var_out[j + 1] = a1;
      }
    }
    if (pass == 0) {
      __syncthreads();
      c0 = s_mean[2 * tx];
      c1 = s_mean[2 * tx + 1];
      if (ty == 0 && on) {
        mean_out[j] = c0;
        if (two) mean_out[j + 1] = c1;
      }
    }
  }
}

cudaError_t launch_cem_draw(const double* mean, const double* var, double* dev, float* rows, int P, int M,
                            long long ld, double extra_var, double noise_left, unsigned long long seed,
                            cudaStream_t st) {
  const int pairs = (P + 1) / 2;
  const dim3 grid((pairs + CEM_DRAW_THREADS - 1) / CEM_DRAW_THREADS, M);
  cem_draw_kernel<<<grid, CEM_DRAW_THREADS, 0, st>>>(mean, var, dev, rows, P, ld, extra_var, noise_left,
                                                     (uint32_t)seed, (uint32_t)(seed >> 32));
  return cudaGetLastError();
}

cudaError_t launch_cem_rank_refit(const double* scores, int M, int keep, int* order, const double* mean,
                                  const double* dev, int P, unsigned long long seed, double* mean_out, double* var_out,
                                  cudaStream_t st) {
  const size_t smem = (size_t)M * sizeof(double);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(cem_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  cem_rank_kernel<<<(M + CEM_RANK_THREADS - 1) / CEM_RANK_THREADS, CEM_RANK_THREADS, smem, st>>>(scores, M, M - keep,
                                                                                               order);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const int pairs = (P + 1) / 2;
  cem_refit_kernel<<<(pairs + CEM_REFIT_PAIRS - 1) / CEM_REFIT_PAIRS, dim3(CEM_REFIT_PAIRS, CEM_REFIT_ROWS), 0, st>>>(
      mean, dev, order, keep, P, (uint32_t)seed, (uint32_t)(seed >> 32), mean_out, var_out);
  return cudaGetLastError();
}
