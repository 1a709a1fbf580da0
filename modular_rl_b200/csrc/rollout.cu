// Device-resident rollouts of the built-in environments (envs.py: CartPole-v0, Pendulum-v0, Acrobot-v1,
// MountainCar-v0, MountainCarContinuous-v0).  The kernel is in rollout_kernel.cuh, which rollout_user.cu also compiles
// at run time for user environments; this file holds the built-in EnvT specialisations and the launchers.
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
#include "rollout_kernel.cuh"
#include "../../include/mrl_b200.h"

// ---------------------------------------------------------------------------------------------------- built-in environments
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
    default: return rollout_user_dims(env, d0, sd, dout, pd);
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

// One round's launch of rollout_kernel instance f (built in, or loaded by rollout_user.cu): one cluster of n_ctas CTAs
cudaError_t launch_rollout_kernel(const void* f, const RolloutArgs& a, int n_ctas, int threads, size_t smem,
                                  cudaStream_t st) {
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
  void* args[] = {(void*)&a};
  return cudaLaunchKernelExC(&cfg, f, args);
}

template <int ENV, int ACT, bool POP>
static cudaError_t launch_t(const RolloutArgs& a, int n_ctas, int threads, size_t smem, cudaStream_t st) {
  return launch_rollout_kernel((const void*)rollout_kernel<ENV, ACT, POP>, a, n_ctas, threads, smem, st);
}

template <bool POP>
static cudaError_t launch_pop(const RolloutArgs& a, int env, int act, int n_ctas, int threads, size_t smem, cudaStream_t st) {
#define RO_ACTS(ENV)                                                          \
  switch (act) {                                                              \
    case MRL_ACT_TANH: return launch_t<ENV, MRL_ACT_TANH, POP>(a, n_ctas, threads, smem, st); \
    case MRL_ACT_RELU: return launch_t<ENV, MRL_ACT_RELU, POP>(a, n_ctas, threads, smem, st); \
    default: return launch_t<ENV, MRL_ACT_SIGMOID, POP>(a, n_ctas, threads, smem, st);        \
  }
  switch (env) {   // the built-in environments
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
  if (env >= RO_USER_ENV0) return launch_rollout_user(a, env, act, pop, n_ctas, threads, smem, st);
  return pop ? launch_pop<true>(a, env, act, n_ctas, threads, smem, st)
             : launch_pop<false>(a, env, act, n_ctas, threads, smem, st);
}
