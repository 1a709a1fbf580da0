// Device-resident rollouts of the built-in environments (envs.py: CartPole-v0, Pendulum-v0, Acrobot-v1,
// MountainCar-v0, MountainCarContinuous-v0).
//
// One launch runs one ROUND: N environments from reset until every episode has ended or reached the timestep limit,
// in the lockstep order of core.rollouts_vectorized (core.py:182-221 run per environment).  Per step t, over the
// environments still live, in index order:
//   observation ZFilter (filters.py:30-38): sample j is normalised with Welford statistics that include the incoming
//     state and every live sample of this step with a smaller index, itself included;
//   policy forward (FP32) on the float32 cast of the filtered observation, reading the net's flat theta;
//   action: Categorical inverse-CDF sample / DiagGauss mean + std * z, or maxprob when not stochastic;
//   dynamics in float64 with the equations and evaluation order of envs.py;
//   reward ZFilter: the raw rewards of the step advance its statistics (only they matter, SURVEY A.5).
//
// Layout: ONE thread-block cluster (<= RO_MAX_CTAS CTAs) per round; CTA c owns environments [c * per_cta, ...), one
// environment per thread.  The ZFilter prefix crosses every environment at every step: each CTA scans its own
// environments (Kogge-Stone Chan merges inside a warp, then the warp totals in order), publishes its total in its
// shared memory, and after the cluster barrier every CTA folds the totals of the lower-ranked CTAs from distributed
// shared memory in rank order.  One cluster barrier per step; the slots are double-buffered by step parity so that a
// slot is never rewritten before every CTA has read it.  The merge tree depends on N only (not on timing), so a round
// is deterministic.  The reward statistics of step t travel with the exchange of step t + 1.
//
// Forward: the live environments of a CTA are compacted (their rank in the scan) and pushed through the MLP in chunks
// of rows; thread o computes output unit o % dout of row o / dout with an in-order FP32 FMA chain, activations of
// the chunk in shared memory, theta staged in shared memory when it fits (4-64-64-2 is 18 KB), else read through L2.
//
// Random numbers: Philox4x32-10 keyed by the round seed, counter (environment, step, purpose, block), so no draw
// depends on the thread / CTA mapping.  DESIGN.md "Device rollouts" gives the mapping to uniforms and normals.
//
// After the round the rows, staged as [step][environment], are compacted into path-major order (offsets from a scan of
// the episode lengths) in the same launch, so the host copies only the collected timesteps.
#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"
#include "../../include/mrl_b200.h"

#include <cooperative_groups.h>
namespace cgr = cooperative_groups;

#define RO_KMAX 7   // observation features + the reward, scanned together (Acrobot: 6 + 1)

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
template <int ENV> struct EnvT;
template <> struct EnvT<MRL_ENV_CARTPOLE> {
  static constexpr int D0 = 4, SD = 4, DOUT = 2, PD = 2, HEAD = MRL_HEAD_CAT;   // prob row: 2 probabilities
  __device__ static void reset(double* s, int e, uint32_t k0, uint32_t k1) {   // uniform(-0.05, 0.05, size=4)
    const uint4 a = philox4x32_10(make_uint4((uint32_t)e, 0u, RO_PURPOSE_RESET, 0u), k0, k1);
    const uint4 b = philox4x32_10(make_uint4((uint32_t)e, 0u, RO_PURPOSE_RESET, 1u), k0, k1);
    const double u[4] = {u53(a.x, a.y), u53(a.z, a.w), u53(b.x, b.y), u53(b.z, b.w)};
#pragma unroll
    for (int i = 0; i < 4; ++i) s[i] = -0.05 + (0.05 - -0.05) * u[i];
  }
  __device__ static void obs(const double* s, double* x) {
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = s[i];
  }
  // envs.py CartPoleEnv.step; reward 1.0 on every step, the terminating one included
  __device__ static bool step(double* s, int action, float, double* reward) {
    const double gravity = 9.8, masscart = 1.0, masspole = 0.1, length = 0.5, force_mag = 10.0, tau = 0.02;
    const double theta_threshold = 12 * 2 * M_PI / 360, x_threshold = 2.4;
    const double x = s[0], x_dot = s[1], th = s[2], th_dot = s[3];
    const double force = action == 1 ? force_mag : -force_mag;
    const double total_mass = masspole + masscart;
    const double pml = masspole * length;
    const double c = cos(th), sn = sin(th);
    const double temp = (force + pml * th_dot * th_dot * sn) / total_mass;
    const double thacc = (gravity * sn - c * temp) / (length * (4.0 / 3.0 - masspole * c * c / total_mass));
    const double xacc = temp - pml * thacc * c / total_mass;
    s[0] = x + tau * x_dot;
    s[1] = x_dot + tau * xacc;
    s[2] = th + tau * th_dot;
    s[3] = th_dot + tau * thacc;
    *reward = 1.0;
    return s[0] < -x_threshold || s[0] > x_threshold || s[2] < -theta_threshold || s[2] > theta_threshold;
  }
};
__device__ __forceinline__ double py_mod(double a, double b) {   // Python's float %: the sign of the divisor
  double r = fmod(a, b);
  if (r != 0.0) {
    if ((b < 0.0) != (r < 0.0)) r += b;
  } else {
    r = copysign(0.0, b);
  }
  return r;
}
template <> struct EnvT<MRL_ENV_PENDULUM> {
  static constexpr int D0 = 3, SD = 2, DOUT = 1, PD = 2, HEAD = MRL_HEAD_GAUSS;  // prob row: mean, std
  __device__ static void reset(double* s, int e, uint32_t k0, uint32_t k1) {   // uniform([-pi, -1], [pi, 1])
    const uint4 a = philox4x32_10(make_uint4((uint32_t)e, 0u, RO_PURPOSE_RESET, 0u), k0, k1);
    s[0] = -M_PI + (M_PI - -M_PI) * u53(a.x, a.y);
    s[1] = -1.0 + (1.0 - -1.0) * u53(a.z, a.w);
  }
  __device__ static void obs(const double* s, double* x) {
    x[0] = cos(s[0]);
    x[1] = sin(s[0]);
    x[2] = s[1];
  }
  // envs.py PendulumEnv.step: u clipped for the dynamics and the cost only; the new angle uses the unclipped velocity
  __device__ static bool step(double* s, int, float action, double* reward) {
    const double max_speed = 8.0, max_torque = 2.0, dt = 0.05, g = 10.0, m = 1.0, l = 1.0;
    const double th = s[0], thdot = s[1];
    const double u = fmin(fmax((double)action, -max_torque), max_torque);
    const double angle = py_mod(th + M_PI, 2 * M_PI) - M_PI;
    const double cost = angle * angle + .1 * thdot * thdot + .001 * (u * u);
    double newthdot = thdot + (-3 * g / (2 * l) * sin(th + M_PI) + 3. / (m * l * l) * u) * dt;
    const double newth = th + newthdot * dt;
    newthdot = fmin(fmax(newthdot, -max_speed), max_speed);
    s[0] = newth;
    s[1] = newthdot;
    *reward = -cost;
    return false;
  }
};

// The dynamics below are written with __dmul_rn for every product so that no product is contracted with a sum into an
// FMA: each operation rounds as the float64 arithmetic of envs.py does, and only cos / sin may differ in the last bits.
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }

template <> struct EnvT<MRL_ENV_ACROBOT> {
  static constexpr int D0 = 6, SD = 4, DOUT = 3, PD = 3, HEAD = MRL_HEAD_CAT;   // prob row: 3 probabilities
  __device__ static void reset(double* s, int e, uint32_t k0, uint32_t k1) {   // uniform(-0.1, 0.1, size=4)
    const uint4 a = philox4x32_10(make_uint4((uint32_t)e, 0u, RO_PURPOSE_RESET, 0u), k0, k1);
    const uint4 b = philox4x32_10(make_uint4((uint32_t)e, 0u, RO_PURPOSE_RESET, 1u), k0, k1);
    const double u[4] = {u53(a.x, a.y), u53(a.z, a.w), u53(b.x, b.y), u53(b.z, b.w)};
#pragma unroll
    for (int i = 0; i < 4; ++i) s[i] = -0.1 + mul(0.1 - -0.1, u[i]);
  }
  __device__ static void obs(const double* s, double* x) {
    x[0] = cos(s[0]);
    x[1] = sin(s[0]);
    x[2] = cos(s[1]);
    x[3] = sin(s[1]);
    x[4] = s[2];
    x[5] = s[3];
  }
  // envs.py AcrobotEnv._dsdt: y = (theta1, theta2, dtheta1, dtheta2), torque a -> k = d/dt of y
  __device__ static void dsdt(const double* y, double a, double* k) {
    const double m1 = 1.0, m2 = 1.0, l1 = 1.0, lc1 = 0.5, lc2 = 0.5, I1 = 1.0, I2 = 1.0, g = 9.8;
    const double th1 = y[0], th2 = y[1], dth1 = y[2], dth2 = y[3];
    double s2, c2;
    sincos(th2, &s2, &c2);                         // one argument reduction: keeps the kernel at 128 registers, no spills
    const double d1 = mul(m1, mul(lc1, lc1)) + mul(m2, mul(l1, l1) + mul(lc2, lc2) + mul(mul(mul(2.0, l1), lc2), c2)) + I1 + I2;
    const double d2 = mul(m2, mul(lc2, lc2) + mul(mul(l1, lc2), c2)) + I2;
    const double phi2 = mul(mul(mul(m2, lc2), g), cos(th1 + th2 - M_PI / 2.0));
    const double phi1 = mul(mul(mul(mul(-m2, l1), lc2), mul(dth2, dth2)), s2)
                        - mul(mul(mul(mul(mul(mul(2.0, m2), l1), lc2), dth2), dth1), s2)
                        + mul(mul(mul(m1, lc1) + mul(m2, l1), g), cos(th1 - M_PI / 2.0)) + phi2;
    const double dd2 = (a + mul(d2 / d1, phi1) - mul(mul(mul(mul(m2, l1), lc2), mul(dth1, dth1)), s2) - phi2)
                       / (mul(m2, mul(lc2, lc2)) + I2 - mul(d2, d2) / d1);
    k[0] = dth1;
    k[1] = dth2;
    k[2] = -(mul(d2, dd2) + phi1) / d1;
    k[3] = dd2;
  }
  // envs.py AcrobotEnv.step: one RK4 step of the torque-augmented state (the torque's derivative is 0, so it stays a
  // constant), the sum (k1 + 2 k2) + 2 k3 + k4 accumulated stage by stage in that order, then wrap, bound, terminal
  __device__ static bool step(double* s, int action, float, double* reward) {
    const double dt = 0.2, dt2 = dt / 2.0, max_vel_1 = 4 * M_PI, max_vel_2 = 9 * M_PI;
    const double a = action == 0 ? -1.0 : (action == 1 ? 0.0 : 1.0);
    double k[4], y[4], acc[4];
    dsdt(s, a, k);
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc[i] = k[i]; y[i] = s[i] + mul(dt2, k[i]); }
    dsdt(y, a, k);
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc[i] = acc[i] + mul(2.0, k[i]); y[i] = s[i] + mul(dt2, k[i]); }
    dsdt(y, a, k);
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc[i] = acc[i] + mul(2.0, k[i]); y[i] = s[i] + mul(dt, k[i]); }
    dsdt(y, a, k);
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = s[i] + mul(dt / 6.0, acc[i] + k[i]);
#pragma unroll
    for (int i = 0; i < 2; ++i) {                  // wrap into [-pi, pi] with envs.py's loops (not fmod)
      double x = y[i];
      const double diff = M_PI - -M_PI;
      while (x > M_PI) x = x - diff;
      while (x < -M_PI) x = x + diff;
      s[i] = x;
    }
    s[2] = fmin(fmax(y[2], -max_vel_1), max_vel_1);
    s[3] = fmin(fmax(y[3], -max_vel_2), max_vel_2);
    const bool terminal = -cos(s[0]) - cos(s[1] + s[0]) > 1.0;
    *reward = terminal ? 0.0 : -1.0;
    return terminal;
  }
};

// envs.py MountainCarEnv._move: velocity += dv and the clips, the left wall, the goal test; state (position, velocity)
__device__ __forceinline__ bool mountain_car_move(double* s, double dv, double goal) {
  const double min_position = -1.2, max_position = 0.6, max_speed = 0.07;
  const double velocity = fmin(fmax(s[1] + dv, -max_speed), max_speed);
  const double position = fmin(fmax(s[0] + velocity, min_position), max_position);
  s[0] = position;
  s[1] = position == min_position && velocity < 0.0 ? 0.0 : velocity;
  return position >= goal && s[1] >= 0.0;
}
__device__ __forceinline__ void mountain_car_reset(double* s, int e, uint32_t k0, uint32_t k1) {   // [uniform(-0.6, -0.4), 0]
  const uint4 a = philox4x32_10(make_uint4((uint32_t)e, 0u, RO_PURPOSE_RESET, 0u), k0, k1);
  s[0] = -0.6 + mul(-0.4 - -0.6, u53(a.x, a.y));
  s[1] = 0.0;
}
template <> struct EnvT<MRL_ENV_MOUNTAIN_CAR> {
  static constexpr int D0 = 2, SD = 2, DOUT = 3, PD = 3, HEAD = MRL_HEAD_CAT;   // prob row: 3 probabilities
  __device__ static void reset(double* s, int e, uint32_t k0, uint32_t k1) { mountain_car_reset(s, e, k0, k1); }
  __device__ static void obs(const double* s, double* x) { x[0] = s[0]; x[1] = s[1]; }
  // envs.py MountainCarEnv.step; reward -1 on every step, the terminating one included
  __device__ static bool step(double* s, int action, float, double* reward) {
    const double dv = mul((double)(action - 1), 0.001) + mul(cos(mul(3.0, s[0])), -0.0025);
    *reward = -1.0;
    return mountain_car_move(s, dv, 0.5);
  }
};
template <> struct EnvT<MRL_ENV_MOUNTAIN_CAR_CONTINUOUS> {
  static constexpr int D0 = 2, SD = 2, DOUT = 1, PD = 2, HEAD = MRL_HEAD_GAUSS;  // prob row: mean, std
  __device__ static void reset(double* s, int e, uint32_t k0, uint32_t k1) { mountain_car_reset(s, e, k0, k1); }
  __device__ static void obs(const double* s, double* x) { x[0] = s[0]; x[1] = s[1]; }
  // envs.py MountainCarContinuousEnv.step: the force is the clipped action, the penalty takes the unclipped one
  __device__ static bool step(double* s, int, float action, double* reward) {
    const double a = (double)action;
    const double force = fmin(fmax(a, -1.0), 1.0);
    const bool done = mountain_car_move(s, mul(force, 0.0015) - mul(0.0025, cos(mul(3.0, s[0]))), 0.45);
    *reward = (done ? 100.0 : 0.0) - mul(0.1, mul(a, a));
    return done;
  }
};

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
        } else {
          af = OUT[row * DOUT];
          if (rows) {
            prob[0] = af;
            prob[1] = 1.f;
            ((float*)a.s_act)[st_row] = af;
          }
        }
      } else if (E::HEAD == MRL_HEAD_CAT) {
        float z[DOUT], p[DOUT], mx = -INFINITY, sum = 0.f;
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
      } else {
        const float mean = OUT[row * DOUT], sd = logstd_exp[0];
        prob[0] = mean;
        prob[1] = sd;
        if (a.stochastic) {                // randn().astype(float32) * std + mean, in float32
          const float z = (float)(sqrt(-2.0 * log(1.0 - u0)) * cos(2.0 * M_PI * u1));
          af = __fadd_rn(__fmul_rn(z, sd), mean);
        } else {
          af = mean;
        }
        ((float*)a.s_act)[st_row] = af;
      }
      const bool done = E::step(s, ai, af, &rew);
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

// ---------------------------------------------------------------------------------------------------- launcher
template <int ENV>
static int env_dims(int* d0, int* sd, int* dout, int* pd) {
  using E = EnvT<ENV>;
  *d0 = E::D0; *sd = E::SD; *dout = E::DOUT; *pd = E::PD;
  return E::HEAD;
}
int rollout_env_dims(int env, int* d0, int* sd, int* dout, int* pd) {
  switch (env) {
    case MRL_ENV_CARTPOLE: return env_dims<MRL_ENV_CARTPOLE>(d0, sd, dout, pd);
    case MRL_ENV_PENDULUM: return env_dims<MRL_ENV_PENDULUM>(d0, sd, dout, pd);
    case MRL_ENV_ACROBOT: return env_dims<MRL_ENV_ACROBOT>(d0, sd, dout, pd);
    case MRL_ENV_MOUNTAIN_CAR: return env_dims<MRL_ENV_MOUNTAIN_CAR>(d0, sd, dout, pd);
    case MRL_ENV_MOUNTAIN_CAR_CONTINUOUS: return env_dims<MRL_ENV_MOUNTAIN_CAR_CONTINUOUS>(d0, sd, dout, pd);
    default: return -1;
  }
}

void rollout_shape(int N, int* n_ctas, int* per_cta, int* threads) {
  int nc = (N + RO_MIN_PER_CTA - 1) / RO_MIN_PER_CTA;
  nc = nc < 1 ? 1 : (nc > RO_MAX_CTAS ? RO_MAX_CTAS : nc);
  const int pc = (N + nc - 1) / nc;
  int th = round_up(pc, 32);
  *n_ctas = nc;
  *per_cta = pc;
  *threads = th < 128 ? 128 : th;
}

size_t rollout_smem_bytes(const RolloutArgs& a, int d0, int dout, bool pop) {
  return ((size_t)a.w_floats + 2 * (size_t)a.rows_chunk * a.ldh + (size_t)a.per_cta * (d0 + dout + (pop ? 1 : 0))) * 4;
}

template <int ENV, int ACT, bool POP>
static cudaError_t launch_t(const RolloutArgs& a, int n_ctas, int threads, size_t smem, cudaStream_t st) {
  const void* f = (const void*)rollout_kernel<ENV, ACT, POP>;
  cudaError_t e = mrl_func_smem(f, smem);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(n_ctas);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = n_ctas;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, rollout_kernel<ENV, ACT, POP>, a);
}

template <bool POP>
static cudaError_t launch_pop(const RolloutArgs& a, int env, int act, int n_ctas, int threads, size_t smem, cudaStream_t st) {
#define RO_ACTS(ENV)                                                          \
  switch (act) {                                                              \
    case MRL_ACT_TANH: return launch_t<ENV, MRL_ACT_TANH, POP>(a, n_ctas, threads, smem, st); \
    case MRL_ACT_RELU: return launch_t<ENV, MRL_ACT_RELU, POP>(a, n_ctas, threads, smem, st); \
    default: return launch_t<ENV, MRL_ACT_SIGMOID, POP>(a, n_ctas, threads, smem, st);        \
  }
  switch (env) {   // mrl_rollout_create accepts only these
    case MRL_ENV_CARTPOLE: RO_ACTS(MRL_ENV_CARTPOLE)
    case MRL_ENV_ACROBOT: RO_ACTS(MRL_ENV_ACROBOT)
    case MRL_ENV_MOUNTAIN_CAR: RO_ACTS(MRL_ENV_MOUNTAIN_CAR)
    case MRL_ENV_MOUNTAIN_CAR_CONTINUOUS: RO_ACTS(MRL_ENV_MOUNTAIN_CAR_CONTINUOUS)
    default: RO_ACTS(MRL_ENV_PENDULUM)
  }
#undef RO_ACTS
}

cudaError_t launch_rollout(const RolloutArgs& a, int env, int act, bool pop, int n_ctas, int threads, size_t smem,
                           cudaStream_t st) {
  return pop ? launch_pop<true>(a, env, act, n_ctas, threads, smem, st)
             : launch_pop<false>(a, env, act, n_ctas, threads, smem, st);
}
