// The rollout kernel: one launch runs one ROUND of lockstep episodes of one environment (rollout.cu has the whole
// description).  nvcc compiles it in rollout.cu for the built-in environments; the library embeds this text and NVRTC
// compiles it for a user environment (rollout_user.cu), with EnvT<id> (id >= RO_USER_ENV0) wrapped around the user's
// CUDA snippet.  So this header includes only NVRTC-clean headers and holds device code only.
#pragma once
#include "kernel_defs.cuh"
#include "philox.cuh"

#include <cooperative_groups.h>
#include <cuda/std/limits>
namespace cgr = cooperative_groups;

#define RO_KMAX (RO_KMAX_OBS + 1)   // observation features + the reward, scanned together (Acrobot: 6 + 1)
#define RO_PI 3.14159265358979323846   // math.h's M_PI, which NVRTC lacks
#define RO_INF (cuda::std::numeric_limits<float>::infinity())   // math.h's INFINITY, which NVRTC lacks

// ---------------------------------------------------------------------------------------------------- Welford
// ---------------------------------------------------------------------------------------------------- Welford
struct Wf { double n, m, s; };
__device__ __forceinline__ Wf wf_merge(const Wf& a, const Wf& b) {   // Chan merge, `a` holds the earlier samples
  if (b.n == 0.0) return a;
  if (a.n == 0.0) return b;
  Wf o;
  o.n = a.n + b.n;
  const double d = b.m - a.m;
  o.m = a.m + d * (b.n / o.n);
  o.s = a.s + b.s + d * d * (a.n * b.n / o.n);
  return o;
}
__device__ __forceinline__ Wf wf_shfl_up(const Wf& w, int o) {
  Wf r;
  r.n = __shfl_up_sync(0xffffffffu, w.n, o);
  r.m = __shfl_up_sync(0xffffffffu, w.m, o);
  r.s = __shfl_up_sync(0xffffffffu, w.s, o);
  return r;
}

// Inclusive scan of K Welford triples over the CTA's threads in index order; `tot` receives the CTA totals.
template <int K>
__device__ __forceinline__ void block_scan(Wf (&w)[K], Wf (*wtot)[RO_KMAX], Wf* tot) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const Wf u = wf_shfl_up(w[k], o);
      if (lane >= o) w[k] = wf_merge(u, w[k]);
    }
  }
  __syncthreads();                       // the previous readers of wtot are done
  if (lane == 31)
#pragma unroll
    for (int k = 0; k < K; ++k) wtot[warp][k] = w[k];
  __syncthreads();
  if (threadIdx.x < K) {                 // exclusive prefix of the warp totals, in warp order
    const int k = threadIdx.x;
    Wf acc = {0.0, 0.0, 0.0};
    for (int i = 0; i < nw; ++i) {
      const Wf t = wtot[i][k];
      wtot[i][k] = acc;
      acc = wf_merge(acc, t);
    }
    tot[k] = acc;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) w[k] = wf_merge(wtot[warp][k], w[k]);
}


// ---------------------------------------------------------------------------------------------------- environments
// EnvT<ENV>: D0 observation entries, SD state entries (float64), DOUT policy outputs, PD prob row width, HEAD; and
//   __device__ static void reset(double* s, int env, uint32_t k0, uint32_t k1)   start state of environment env
//   __device__ static void obs(const double* s, double* x)                        observation of a state
//   __device__ static bool step(double* s, int action, <action>, double* reward)  -> terminated
// <action>: float (the built-ins: the d = 1 DiagGauss action) or const float* a (user environments: the d entries).
// The built-in specialisations are in rollout.cu.
template <int ENV> struct EnvT;

__device__ __forceinline__ double py_mod(double a, double b) {   // Python's float %: the sign of the divisor
  double r = fmod(a, b);
  if (r != 0.0) {
    if ((b < 0.0) != (r < 0.0)) r += b;
  } else {
    r = copysign(0.0, b);
  }
  return r;
}

// The reset draw of a user environment: uniforms (u0, u1) of counter (env, 0, RO_PURPOSE_RESET, block), as the
// built-ins draw theirs
__device__ __forceinline__ void reset_uniforms(int env, int block, uint32_t k0, uint32_t k1, double* u0, double* u1) {
  const uint4 a = philox4x32_10(make_uint4((uint32_t)env, 0u, RO_PURPOSE_RESET, (uint32_t)block), k0, k1);
  *u0 = u53(a.x, a.y);
  *u1 = u53(a.z, a.w);
}

// ---------------------------------------------------------------------------------------------------- policy forward
// rows [0, nrows) of xin [nrows][d0] -> out [nrows][dout]: raw head output (softmax logits / Gauss mean).
// POP: row r uses the theta of environment rowe[r], W + rowe[r] * a.ld_theta.
template <int ACT, bool POP>
__device__ void mlp_rows(const RolloutArgs& a, const float* W, const float* xin, int nrows, float* h, float* out,
                         const int* rowe) {
  for (int c0 = 0; c0 < nrows; c0 += a.rows_chunk) {
    const int nr = min(a.rows_chunk, nrows - c0);
    const float* src = xin + (size_t)c0 * a.d[0];
    int lds = a.d[0], cur = 0;
    const float* th = W;
    for (int l = 1; l <= a.L; ++l) {
      const int din = a.d[l - 1], dout = a.d[l];
      const float* Wl = th;                        // [din][dout], C order (the reference's flat order)
      const float* bl = th + (size_t)din * dout;
      const bool last = l == a.L;
      float* dst = last ? out + (size_t)c0 * dout : h + (size_t)cur * a.rows_chunk * a.ldh;
      const int ldd = last ? dout : a.ldh;
      for (int o = threadIdx.x; o < nr * dout; o += blockDim.x) {
        const int r = o / dout, j = o - r * dout;
        const float* hr = src + (size_t)r * lds;
        const float* Wr = Wl;
        const float* br = bl;
        if constexpr (POP) {
          const size_t m = (size_t)rowe[c0 + r] * a.ld_theta;
          Wr += m;
          br += m;
        }
        float acc = 0.f;
        for (int k = 0; k < din; ++k) acc = fmaf(hr[k], Wr[(size_t)k * dout + j], acc);
        acc += br[j];
        dst[(size_t)r * ldd + j] = last ? acc : act_fn<ACT>(acc);
      }
      __syncthreads();
      src = dst;
      lds = ldd;
      cur ^= 1;
      th += (size_t)din * dout + dout;
    }
  }
}

// ---------------------------------------------------------------------------------------------------- the round
// POP (population round, the cross-entropy method): environment e acts deterministically with its own Dense theta
// (a.theta + e * a.ld_theta, no logstd block, read through L2), on the argmax of the raw outputs (Categorical heads)
// or the raw output (DiagGauss heads); a.returns[e] = the float64 sum of its raw rewards in step order; without a.want_rows no
// staging rows are written and nothing is compacted.
template <int ENV, int ACT, bool POP>
__global__ void __launch_bounds__(RO_MAX_THREADS, 1) rollout_kernel(const RolloutArgs a) {
  using E = EnvT<ENV>;
  constexpr int D0 = E::D0, SD = E::SD, DOUT = E::DOUT, PD = E::PD, K = D0 + 1;   // K - 1: the reward
  constexpr bool USER = ENV >= RO_USER_ENV0;   // DiagGauss heads of any d, step(s, action, a[d], &reward)
  static_assert(K <= RO_KMAX, "RO_KMAX must cover the observation features and the reward");
  static_assert(PD == (E::HEAD == MRL_HEAD_CAT ? DOUT : 2 * DOUT), "prob row: K probabilities / mean and std");
  cgr::cluster_group cluster = cgr::this_cluster();
  const int rank = (int)cluster.block_rank(), nc = (int)cluster.num_blocks();

  __shared__ Wf slot[2][RO_KMAX];          // this CTA's totals of the step (read by every CTA of the cluster)
  __shared__ Wf wtot[RO_MAX_THREADS / 32][RO_KMAX];
  __shared__ Wf ctatot[RO_KMAX];
  __shared__ Wf pre[RO_KMAX];              // filter state + totals of the lower-ranked CTAs (this step)
  __shared__ Wf run[RO_KMAX];              // running filter states: observation features, reward
  __shared__ Wf pushed[RO_KMAX];           // statistics of this round's samples alone
  __shared__ double live_total;
  __shared__ long long lslot, lbase, ltotal;
  __shared__ long long wlen[RO_MAX_THREADS / 32];
  extern __shared__ __align__(16) float dsm[];
  float* Ws = dsm;                                            // theta (a.w_floats; 0 when read through L2)
  float* H = Ws + a.w_floats;                                 // [2][rows_chunk][ldh]
  float* XIN = H + 2 * (size_t)a.rows_chunk * a.ldh;          // [per_cta][D0]
  float* OUT = XIN + (size_t)a.per_cta * D0;                  // [per_cta][DOUT]
  int* ROWE = (int*)(OUT + (size_t)a.per_cta * DOUT);         // POP: [per_cta] live row -> environment
  const bool rows = !POP || a.want_rows;

  for (int i = threadIdx.x; i < a.w_floats; i += blockDim.x) Ws[i] = a.theta[i];
  const float* W = a.w_floats ? Ws : a.theta;
  if (threadIdx.x < K) {
    const int k = threadIdx.x;
    const double* f = a.filt_in;
    run[k] = k < D0 ? Wf{f[0], f[1 + k], f[1 + D0 + k]} : Wf{f[1 + 2 * D0], f[2 + 2 * D0], f[3 + 2 * D0]};
    pushed[k] = Wf{0.0, 0.0, 0.0};
  }

  const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
  const int le = threadIdx.x, e = rank * a.per_cta + le;
  const bool mine = le < a.per_cta && e < a.N;
  double s[SD];
  if (mine) E::reset(s, e, k0, k1);
  else
#pragma unroll
    for (int i = 0; i < SD; ++i) s[i] = 0.0;
  bool live = mine, term = false, rlive = false;
  double rew = 0.0;
  int len = 0;
  double ret = 0.0;
  float logstd_exp[DOUT];
#pragma unroll
  for (int j = 0; j < DOUT; ++j) logstd_exp[j] = E::HEAD == MRL_HEAD_GAUSS && !POP ? expf(a.theta[a.P - DOUT + j]) : 0.f;

  for (int t = 0;; ++t) {
    const bool now = live && t < a.T;
    Wf w[K];
    {
      double x[D0];
      E::obs(s, x);
#pragma unroll
      for (int k = 0; k < D0; ++k) w[k] = now ? Wf{1.0, x[k], 0.0} : Wf{0.0, 0.0, 0.0};
    }
    w[D0] = rlive ? Wf{1.0, rew, 0.0} : Wf{0.0, 0.0, 0.0};   // the rewards of step t - 1
    block_scan<K>(w, wtot, ctatot);
    if (threadIdx.x < K) slot[t & 1][threadIdx.x] = ctatot[threadIdx.x];
    cluster.sync();
    if (threadIdx.x < K) {
      const int k = threadIdx.x;
      Wf tot = {0.0, 0.0, 0.0}, excl = {0.0, 0.0, 0.0};
      for (int r = 0; r < nc; ++r) {
        const Wf v = *cluster.map_shared_rank(&slot[t & 1][k], r);
        if (r < rank) excl = wf_merge(excl, v);
        tot = wf_merge(tot, v);
      }
      const bool on = k < D0 ? a.ob_on : a.rew_on;
      pre[k] = wf_merge(run[k], excl);
      if (on) {
        run[k] = wf_merge(run[k], tot);
        pushed[k] = wf_merge(pushed[k], tot);
      }
      if (k == 0) live_total = tot.n;
    }
    __syncthreads();
    if (live_total == 0.0) break;          // every episode has ended (or t == T): uniform over the cluster
    rlive = false;
    const int row = (int)w[0].n - 1;       // rank of this environment among the CTA's live ones
    const int nlive = (int)ctatot[0].n;
    const size_t st_row = (size_t)t * a.N + e;
    if (now) {
      double x[D0];
      E::obs(s, x);                        // recomputed, not kept live across the scan (Acrobot's 6 entries spill)
#pragma unroll
      for (int k = 0; k < D0; ++k) {
        double y = x[k];
        if (a.ob_on) {
          const Wf f = wf_merge(pre[k], w[k]);
          if (a.ob_demean) y = y - f.m;
          if (a.ob_destd) {
            const double var = f.n > 1.0 ? f.s / (f.n - 1.0) : f.m * f.m;   // running_stat.py:26-27
            y = y / (sqrt(var) + 1e-8);
          }
          if (a.ob_clip != 0.0) y = fmin(fmax(y, -a.ob_clip), a.ob_clip);
        }
        if (rows) a.s_obs[st_row * D0 + k] = y;
        XIN[row * D0 + k] = (float)y;
      }
      if (a.s_state)
#pragma unroll
        for (int i = 0; i < SD; ++i) a.s_state[st_row * SD + i] = s[i];
      if constexpr (POP) ROWE[row] = e;
    }
    __syncthreads();
    mlp_rows<ACT, POP>(a, W, XIN, nlive, H, OUT, ROWE);
    if (now) {
      const uint4 rnd = philox4x32_10(make_uint4((uint32_t)e, (uint32_t)t, RO_PURPOSE_ACTION, 0u), k0, k1);
      const double u0 = u53(rnd.x, rnd.y), u1 = u53(rnd.z, rnd.w);
      int ai = 0;
      float af = 0.f;
      float av[USER ? DOUT : 1];           // user environments: the action vector (DiagGauss)
      if constexpr (USER)
#pragma unroll
        for (int j = 0; j < DOUT; ++j) av[j] = 0.f;
      float* prob = a.s_prob + st_row * PD;
      if constexpr (POP) {                 // the raw outputs: argmax (first maximum) / the output itself
        if (E::HEAD == MRL_HEAD_CAT) {     // numpy's argmax: the first NaN wins, else the first maximum
          float best = OUT[row * DOUT];
#pragma unroll
          for (int j = 1; j < DOUT; ++j) {
            const float v = OUT[row * DOUT + j];
            if (!isnan(best) && (v > best || isnan(v))) { best = v; ai = j; }
          }
          if (rows) {
#pragma unroll
            for (int j = 0; j < DOUT; ++j) prob[j] = OUT[row * DOUT + j];
            ((int*)a.s_act)[st_row] = ai;
          }
        } else if constexpr (USER) {
#pragma unroll
          for (int j = 0; j < DOUT; ++j) {
            av[j] = OUT[row * DOUT + j];
            if (rows) {
              prob[j] = av[j];
              prob[DOUT + j] = 1.f;
              ((float*)a.s_act)[st_row * DOUT + j] = av[j];
            }
          }
        } else {
          af = OUT[row * DOUT];
          if (rows) {
            prob[0] = af;
            prob[1] = 1.f;
            ((float*)a.s_act)[st_row] = af;
          }
        }
      } else if (E::HEAD == MRL_HEAD_CAT) {
        float z[DOUT], p[DOUT], mx = -RO_INF, sum = 0.f;
#pragma unroll
        for (int j = 0; j < DOUT; ++j) { z[j] = OUT[row * DOUT + j]; mx = fmaxf(mx, z[j]); }
#pragma unroll
        for (int j = 0; j < DOUT; ++j) { p[j] = expf(z[j] - mx); sum += p[j]; }
#pragma unroll
        for (int j = 0; j < DOUT; ++j) { p[j] = p[j] / sum; prob[j] = p[j]; }
        if (a.stochastic) {                // argmax(cumsum(p) > u): float32 cumsum, compared in float64
          float c = 0.f;
          bool found = false;
#pragma unroll
          for (int j = 0; j < DOUT; ++j) {
            c += p[j];
            if (!found && (double)c > u0) { ai = j; found = true; }
          }
        } else {                           // argmax, first maximum
          float best = p[0];
#pragma unroll
          for (int j = 1; j < DOUT; ++j) if (p[j] > best) { best = p[j]; ai = j; }
        }
        ((int*)a.s_act)[st_row] = ai;
      } else if constexpr (USER) {         // entry j: the normal of block j (block 0: the draw of the d = 1 heads)
#pragma unroll
        for (int j = 0; j < DOUT; ++j) {
          const float mean = OUT[row * DOUT + j], sd = logstd_exp[j];
          prob[j] = mean;
          prob[DOUT + j] = sd;
          float aj = mean;
          if (a.stochastic) {
            const uint4 r = philox4x32_10(make_uint4((uint32_t)e, (uint32_t)t, RO_PURPOSE_ACTION, (uint32_t)j), k0, k1);
            const double v0 = u53(r.x, r.y), v1 = u53(r.z, r.w);
            const float z = (float)(sqrt(-2.0 * log(1.0 - v0)) * cos(2.0 * RO_PI * v1));
            aj = __fadd_rn(__fmul_rn(z, sd), mean);
          }
          av[j] = aj;
          ((float*)a.s_act)[st_row * DOUT + j] = aj;
        }
      } else {
        const float mean = OUT[row * DOUT], sd = logstd_exp[0];
        prob[0] = mean;
        prob[1] = sd;
        if (a.stochastic) {                // randn().astype(float32) * std + mean, in float32
          const float z = (float)(sqrt(-2.0 * log(1.0 - u0)) * cos(2.0 * RO_PI * u1));
          af = __fadd_rn(__fmul_rn(z, sd), mean);
        } else {
          af = mean;
        }
        ((float*)a.s_act)[st_row] = af;
      }
      bool done;
      if constexpr (USER) done = E::step(s, ai, av, &rew);
      else done = E::step(s, ai, af, &rew);
      if (rows) a.s_rew[st_row] = rew;
      if constexpr (POP) ret += rew;
      rlive = true;
      ++len;
      if (done) { term = true; live = false; }
    }
  }

  // ---- compaction: path-major rows at offsets from an exclusive scan of the lengths (CTA rank order, then index)
  if (mine) { a.lengths[e] = len; a.term[e] = term ? 1 : 0; }
  if (POP && mine) a.returns[e] = ret;
  long long incl = len;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) wlen[warp] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long acc = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { const long long v = wlen[i]; wlen[i] = acc; acc += v; }
    lslot = acc;
  }
  cluster.sync();
  if (threadIdx.x == 0) {
    long long base = 0, tot = 0;
    for (int r = 0; r < nc; ++r) {
      const long long v = *cluster.map_shared_rank(&lslot, r);
      if (r < rank) base += v;
      tot += v;
    }
    lbase = base;
    ltotal = tot;
  }
  __syncthreads();
  const long long off = lbase + wlen[warp] + incl - len, total = ltotal;
  const RolloutLayout lay = rollout_layout(total, D0, SD, PD, E::HEAD == MRL_HEAD_CAT ? 1 : DOUT, a.s_state != nullptr);
  double* b_obs = (double*)(a.body + lay.obs);
  double* b_rew = (double*)(a.body + lay.rew);
  double* b_st = (double*)(a.body + lay.state);
  float* b_prob = (float*)(a.body + lay.prob);
  for (int tt = 0; tt < (rows ? len : 0); ++tt) {
    const size_t src = (size_t)tt * a.N + e, dst = (size_t)(off + tt);
#pragma unroll
    for (int k = 0; k < D0; ++k) b_obs[dst * D0 + k] = a.s_obs[src * D0 + k];
    b_rew[dst] = a.s_rew[src];
    if (a.s_state)
#pragma unroll
      for (int i = 0; i < SD; ++i) b_st[dst * SD + i] = a.s_state[src * SD + i];
#pragma unroll
    for (int j = 0; j < PD; ++j) b_prob[dst * PD + j] = a.s_prob[src * PD + j];
    if (E::HEAD == MRL_HEAD_CAT) ((int*)(a.body + lay.act))[dst] = ((const int*)a.s_act)[src];
    else
#pragma unroll
      for (int j = 0; j < DOUT; ++j) ((float*)(a.body + lay.act))[dst * DOUT + j] = ((const float*)a.s_act)[src * DOUT + j];
  }
  if (rank == 0 && threadIdx.x == 0) {   // header: total, observation state, its pushed part, reward state, pushed
    double* h = a.head;
    h[0] = (double)total;
    h[1] = run[0].n;
    h[2 + 2 * D0] = pushed[0].n;
    for (int k = 0; k < D0; ++k) {
      h[2 + k] = run[k].m; h[2 + D0 + k] = run[k].s;
      h[3 + 2 * D0 + k] = pushed[k].m; h[3 + 3 * D0 + k] = pushed[k].s;
    }
    double* r = h + 3 + 4 * D0;
    r[0] = run[D0].n; r[1] = run[D0].m; r[2] = run[D0].s;
    r[3] = pushed[D0].n; r[4] = pushed[D0].m; r[5] = pushed[D0].s;
  }
  cluster.sync();                        // no CTA leaves while another may still read its slots
}
