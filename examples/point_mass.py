"""PointMass-v0: a user environment that also runs in device rollouts, and the template for writing one.

A point mass in the plane, state (x, y, vx, vy), observation = state.  The action is a 2-D force, each entry clipped
to [-1, 1]; one step of dt = 0.1 is semi-implicit Euler:
    v += dt * f;  p += dt * v
    reward = -(x^2 + y^2) - 0.01 |f|^2   (after the move, with the clipped force)
    terminated when x^2 + y^2 < 0.05^2 and vx^2 + vy^2 < 0.05^2
Reset: x, y uniform in [-1, 1), at rest.  Episodes end after 200 steps.

The host class is the reference: run_pg.py / run_cem.py run it without --device_envs.  `device_kind` gives the same
reset / obs / step as CUDA, in float64 and in the same order of operations, so that a device round replays through
this class exactly.  The products are written __dmul_rn and the sums __dadd_rn: otherwise the compiler may contract
a product and a sum into one fused multiply-add, which rounds once where Python rounds twice.  The reset draws its
uniforms with reset_uniforms (include/mrl_b200.h, mrl_rollout_env_compile); it does not follow numpy's stream, so a
device round starts from other states than a host rollout with the same seed.

    python run_pg.py --env examples.point_mass:PointMass-v0 --agent modular_rl_b200.agentzoo.TrpoAgent \\
        --device_envs 256
"""
import numpy as np

from modular_rl_b200 import envs
from modular_rl_b200.spaces import Box

DEVICE_SOURCE = r"""
__device__ static void reset(double* s, int env, uint32_t k0, uint32_t k1) {
  double u0, u1;
  reset_uniforms(env, 0, k0, k1, &u0, &u1);
  s[0] = __dadd_rn(-1.0, __dmul_rn(2.0, u0));
  s[1] = __dadd_rn(-1.0, __dmul_rn(2.0, u1));
  s[2] = 0.0;
  s[3] = 0.0;
}
__device__ static void obs(const double* s, double* x) {
  for (int i = 0; i < 4; ++i) x[i] = s[i];
}
__device__ static bool step(double* s, int, const float* a, double* reward) {
  const double dt = 0.1;
  const double fx = fmin(fmax((double)a[0], -1.0), 1.0), fy = fmin(fmax((double)a[1], -1.0), 1.0);
  const double vx = __dadd_rn(s[2], __dmul_rn(dt, fx)), vy = __dadd_rn(s[3], __dmul_rn(dt, fy));
  const double x = __dadd_rn(s[0], __dmul_rn(dt, vx)), y = __dadd_rn(s[1], __dmul_rn(dt, vy));
  s[0] = x;
  s[1] = y;
  s[2] = vx;
  s[3] = vy;
  const double d2 = __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y));
  const double v2 = __dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy));
  const double f2 = __dadd_rn(__dmul_rn(fx, fx), __dmul_rn(fy, fy));
  *reward = __dadd_rn(-d2, -__dmul_rn(0.01, f2));
  return d2 < 0.0025 && v2 < 0.0025;
}
"""


class _Spec(object):
    def __init__(self, id_, max_episode_steps):
        self.id = id_
        self.max_episode_steps = self.timestep_limit = max_episode_steps


class PointMassEnv(object):
    device_kind = envs.DeviceEnv(DEVICE_SOURCE, state_dim=4)
    dt = 0.1

    def __init__(self):
        self.observation_space = Box(np.full(4, -np.inf), np.full(4, np.inf))
        self.action_space = Box(-np.ones(2), np.ones(2))
        self.spec = _Spec("PointMass-v0", 200)
        self.state = None

    def reset(self):
        x, y = np.random.uniform(-1.0, 1.0, size=2)
        self.state = np.array([x, y, 0.0, 0.0])
        return np.array(self.state)

    def step(self, action):
        a = np.asarray(action).reshape(-1)
        x, y, vx, vy = (float(v) for v in self.state)
        fx, fy = min(max(float(a[0]), -1.0), 1.0), min(max(float(a[1]), -1.0), 1.0)
        vx, vy = vx + self.dt * fx, vy + self.dt * fy
        x, y = x + self.dt * vx, y + self.dt * vy
        self.state = np.array([x, y, vx, vy])
        d2 = x * x + y * y
        v2 = vx * vx + vy * vy
        reward = -d2 - 0.01 * (fx * fx + fy * fy)
        return np.array(self.state), reward, bool(d2 < 0.0025 and v2 < 0.0025), {}

    def render(self):
        pass

    def close(self):
        pass


envs.register("PointMass-v0", PointMassEnv)
