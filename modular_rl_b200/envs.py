"""The classic-control environments with the old gym API (reset() -> ob, step(a) -> ob, rew, done,
info) so that BASELINE config 1 (CartPole-v0 TrpoAgent via run_pg.py) and the reference's coverage
smoke (run_cem.py on Acrobot, run_pg.py on Pendulum, coverage.sh:6-7) run without gym, which is not installed here.
Dynamics follow the published classic-control equations (Barto-Sutton-Anderson cart-pole; torque-limited pendulum;
Sutton-Barto acrobot; Moore's mountain car, discrete and continuous).  Every one of them also runs on the device
(rollout.cu), which replays the float64 arithmetic of these classes.

A user environment runs on the device too when its class sets `device_kind = DeviceEnv(source, state_dim)`: the same
reset / obs / step as a CUDA snippet, which the library compiles into the rollout kernel at run time
(examples/point_mass.py is the template).  register(id, cls) adds a class to make(), and make("pkg.module:Id")
imports pkg.module first, as gym's make does."""
import importlib
import math

import numpy as np

from .spaces import Box, Discrete


class _Spec(object):
    def __init__(self, id_, max_episode_steps):
        self.id = id_
        self.max_episode_steps = max_episode_steps
        self.timestep_limit = max_episode_steps


class CartPoleEnv(object):
    device_kind = "cartpole"        # rollout.cu implements these dynamics (core.do_rollouts_device)
    gravity, masscart, masspole, length, force_mag, tau = 9.8, 1.0, 0.1, 0.5, 10.0, 0.02
    theta_threshold = 12 * 2 * math.pi / 360
    x_threshold = 2.4

    def __init__(self):
        high = np.array([self.x_threshold * 2, np.finfo(np.float32).max, self.theta_threshold * 2,
                         np.finfo(np.float32).max])
        self.observation_space = Box(-high, high)
        self.action_space = Discrete(2)
        self.spec = _Spec("CartPole-v0", 200)
        self.state = None

    def reset(self):
        self.state = np.random.uniform(-0.05, 0.05, size=(4,))
        return np.array(self.state)

    def step(self, action):
        x, x_dot, th, th_dot = self.state
        force = self.force_mag if int(action) == 1 else -self.force_mag
        total_mass = self.masspole + self.masscart
        pml = self.masspole * self.length
        c, s = math.cos(th), math.sin(th)
        temp = (force + pml * th_dot * th_dot * s) / total_mass
        thacc = (self.gravity * s - c * temp) / (self.length * (4.0 / 3.0 - self.masspole * c * c / total_mass))
        xacc = temp - pml * thacc * c / total_mass
        self.state = np.array([x + self.tau * x_dot, x_dot + self.tau * xacc, th + self.tau * th_dot,
                               th_dot + self.tau * thacc])
        x, _, th, _ = self.state
        done = bool(x < -self.x_threshold or x > self.x_threshold or th < -self.theta_threshold
                    or th > self.theta_threshold)
        return np.array(self.state), 1.0, done, {}

    def render(self):
        pass

    def close(self):
        pass


class PendulumEnv(object):
    device_kind = "pendulum"
    max_speed, max_torque, dt, g, m, l = 8.0, 2.0, 0.05, 10.0, 1.0, 1.0

    def __init__(self):
        high = np.array([1.0, 1.0, self.max_speed])
        self.observation_space = Box(-high, high)
        self.action_space = Box(np.array([-self.max_torque]), np.array([self.max_torque]))
        self.spec = _Spec("Pendulum-v0", 200)
        self.state = None

    def _ob(self):
        th, thdot = self.state
        return np.array([math.cos(th), math.sin(th), thdot])

    def reset(self):
        self.state = np.random.uniform([-math.pi, -1.0], [math.pi, 1.0])
        return self._ob()

    def step(self, u):
        th, thdot = self.state
        u = float(np.clip(np.asarray(u).reshape(-1)[0], -self.max_torque, self.max_torque))
        angle = ((th + math.pi) % (2 * math.pi)) - math.pi
        cost = angle ** 2 + .1 * thdot ** 2 + .001 * u ** 2
        newthdot = thdot + (-3 * self.g / (2 * self.l) * math.sin(th + math.pi) + 3. / (self.m * self.l ** 2) * u) * self.dt
        newth = th + newthdot * self.dt
        newthdot = float(np.clip(newthdot, -self.max_speed, self.max_speed))
        self.state = np.array([newth, newthdot])
        return self._ob(), -cost, False, {}

    def render(self):
        pass

    def close(self):
        pass


class AcrobotEnv(object):
    """Acrobot-v1, the "book" dynamics of Sutton & Barto: two links hanging from a fixed pivot, torque on the joint
    between them.  Limit 500 steps.  Constants dt = 0.2, m1 = m2 = l1 = 1, lc1 = lc2 = 0.5, I1 = I2 = 1, g = 9.8;
    velocity bounds 4 pi and 9 pi; torques [-1, 0, +1] indexed by the action.

    State (theta1, theta2, dtheta1, dtheta2), reset uniform(-0.1, 0.1, size=4).  Observation [cos theta1, sin theta1,
    cos theta2, sin theta2, dtheta1, dtheta2].  A step takes one classical RK4 step over [0, dt] of the state augmented
    with the torque (k1..k4, y0 + dt / 6 * (k1 + 2 k2 + 2 k3 + k4)), wraps both angles into [-pi, pi] with `while`
    loops, clips both velocities to their bounds, and ends the episode when -cos theta1 - cos(theta2 + theta1) > 1;
    reward -1 on every other step, 0 on the terminal one.  The derivative (_dsdt):
        d1 = m1 lc1^2 + m2 (l1^2 + lc2^2 + 2 l1 lc2 cos theta2) + I1 + I2
        d2 = m2 (lc2^2 + l1 lc2 cos theta2) + I2
        phi2 = m2 lc2 g cos(theta1 + theta2 - pi/2)
        phi1 = -m2 l1 lc2 dtheta2^2 sin theta2 - 2 m2 l1 lc2 dtheta2 dtheta1 sin theta2
               + (m1 lc1 + m2 l1) g cos(theta1 - pi/2) + phi2
        ddtheta2 = (a + d2 / d1 phi1 - m2 l1 lc2 dtheta1^2 sin theta2 - phi2) / (m2 lc2^2 + I2 - d2^2 / d1)
        ddtheta1 = -(d2 ddtheta2 + phi1) / d1
    The device rollouts (rollout.cu) replay this code operation by operation, so its evaluation order is the spec."""
    device_kind = "acrobot"
    dt = 0.2
    m1, m2, l1, lc1, lc2, I1, I2, g = 1.0, 1.0, 1.0, 0.5, 0.5, 1.0, 1.0, 9.8
    MAX_VEL_1, MAX_VEL_2 = 4 * math.pi, 9 * math.pi
    AVAIL_TORQUE = (-1.0, 0.0, 1.0)

    def __init__(self):
        high = np.array([1.0, 1.0, 1.0, 1.0, self.MAX_VEL_1, self.MAX_VEL_2])
        self.observation_space = Box(-high, high)
        self.action_space = Discrete(3)
        self.spec = _Spec("Acrobot-v1", 500)
        self.state = None

    def _ob(self):
        s = self.state
        return np.array([math.cos(s[0]), math.sin(s[0]), math.cos(s[1]), math.sin(s[1]), s[2], s[3]])

    def reset(self):
        self.state = np.random.uniform(-0.1, 0.1, size=(4,))
        return self._ob()

    def _dsdt(self, y):
        """d/dt of the augmented state y = (theta1, theta2, dtheta1, dtheta2, a)."""
        m1, m2, l1, lc1, lc2, I1, I2, g = self.m1, self.m2, self.l1, self.lc1, self.lc2, self.I1, self.I2, self.g
        theta1, theta2, dtheta1, dtheta2, a = y
        d1 = m1 * (lc1 * lc1) + m2 * (l1 * l1 + lc2 * lc2 + 2 * l1 * lc2 * math.cos(theta2)) + I1 + I2
        d2 = m2 * (lc2 * lc2 + l1 * lc2 * math.cos(theta2)) + I2
        phi2 = m2 * lc2 * g * math.cos(theta1 + theta2 - math.pi / 2.0)
        phi1 = (-m2 * l1 * lc2 * (dtheta2 * dtheta2) * math.sin(theta2)
                - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * math.sin(theta2)
                + (m1 * lc1 + m2 * l1) * g * math.cos(theta1 - math.pi / 2.0) + phi2)
        ddtheta2 = ((a + d2 / d1 * phi1 - m2 * l1 * lc2 * (dtheta1 * dtheta1) * math.sin(theta2) - phi2)
                    / (m2 * (lc2 * lc2) + I2 - d2 * d2 / d1))
        ddtheta1 = -(d2 * ddtheta2 + phi1) / d1
        return (dtheta1, dtheta2, ddtheta1, ddtheta2, 0.0)

    def _rk4(self, y0):
        dt = self.dt
        dt2 = dt / 2.0
        k1 = self._dsdt(y0)
        k2 = self._dsdt([y + dt2 * k for y, k in zip(y0, k1)])
        k3 = self._dsdt([y + dt2 * k for y, k in zip(y0, k2)])
        k4 = self._dsdt([y + dt * k for y, k in zip(y0, k3)])
        return [y + dt / 6.0 * (a + 2 * b + 2 * c + d) for y, a, b, c, d in zip(y0, k1, k2, k3, k4)]

    @staticmethod
    def _wrap(x, m, M):
        diff = M - m
        while x > M:
            x = x - diff
        while x < m:
            x = x + diff
        return x

    def step(self, action):
        s = [float(v) for v in self.state]
        ns = self._rk4(s + [self.AVAIL_TORQUE[int(action)]])
        th1 = self._wrap(ns[0], -math.pi, math.pi)
        th2 = self._wrap(ns[1], -math.pi, math.pi)
        dth1 = min(max(ns[2], -self.MAX_VEL_1), self.MAX_VEL_1)
        dth2 = min(max(ns[3], -self.MAX_VEL_2), self.MAX_VEL_2)
        self.state = np.array([th1, th2, dth1, dth2])
        terminal = bool(-math.cos(th1) - math.cos(th2 + th1) > 1.0)
        return self._ob(), (0.0 if terminal else -1.0), terminal, {}

    def render(self):
        pass

    def close(self):
        pass


class MountainCarEnv(object):
    """MountainCar-v0: an underpowered car in a valley must reach the hill top at position 0.5.  Limit 200 steps,
    Discrete(3) actions (push left, none, right).  State and observation (position, velocity), a Box from
    [-1.2, -0.07] to [0.6, 0.07]; reset [uniform(-0.6, -0.4), 0].  A step:
        velocity += (a - 1) * 0.001 + cos(3 position) * (-0.0025), clipped to [-0.07, 0.07]
        position += velocity, clipped to [-1.2, 0.6]
        velocity = 0 if position == -1.2 and velocity < 0 (the left wall)
        done = position >= 0.5 and velocity >= 0; reward -1 on every step.
    The device rollouts (rollout.cu) replay this code operation by operation, so its evaluation order is the spec."""
    device_kind = "mountaincar"
    min_position, max_position, max_speed, goal_position = -1.2, 0.6, 0.07, 0.5
    force, gravity = 0.001, 0.0025

    def __init__(self):
        self.observation_space = Box(np.array([self.min_position, -self.max_speed]),
                                     np.array([self.max_position, self.max_speed]))
        self.action_space = Discrete(3)
        self.spec = _Spec("MountainCar-v0", 200)
        self.state = None

    def reset(self):
        self.state = np.array([np.random.uniform(-0.6, -0.4), 0.0])
        return np.array(self.state)

    def _move(self, position, velocity, dv, goal):
        """The shared tail of both MountainCars: velocity += dv, the clips, the left wall, the goal test."""
        velocity = min(max(velocity + dv, -self.max_speed), self.max_speed)
        position = min(max(position + velocity, self.min_position), self.max_position)
        if position == self.min_position and velocity < 0:
            velocity = 0.0
        self.state = np.array([position, velocity])
        return bool(position >= goal and velocity >= 0)

    def step(self, action):
        position, velocity = float(self.state[0]), float(self.state[1])
        dv = (int(action) - 1) * self.force + math.cos(3 * position) * (-self.gravity)
        done = self._move(position, velocity, dv, self.goal_position)
        return np.array(self.state), -1.0, done, {}

    def render(self):
        pass

    def close(self):
        pass


class MountainCarContinuousEnv(MountainCarEnv):
    """MountainCarContinuous-v0: MountainCar with a force a in Box([-1], [1]).  Limit 999 steps, goal position 0.45;
    reset, observation, clips and the left wall as MountainCar.  A step:
        force = clip(a[0], -1, 1); velocity += force * 0.0015 - 0.0025 cos(3 position)
        done = position >= 0.45 and velocity >= 0
        reward = (100 if done else 0) - 0.1 * a[0]^2, with the UNCLIPPED action.
    The device rollouts (rollout.cu) replay this code operation by operation, so its evaluation order is the spec."""
    device_kind = "mountaincar_continuous"
    goal_position, power = 0.45, 0.0015

    def __init__(self):
        super(MountainCarContinuousEnv, self).__init__()
        self.action_space = Box(np.array([-1.0]), np.array([1.0]))
        self.spec = _Spec("MountainCarContinuous-v0", 999)

    def step(self, action):
        position, velocity = float(self.state[0]), float(self.state[1])
        a = float(np.asarray(action).reshape(-1)[0])
        force = min(max(a, -1.0), 1.0)
        done = self._move(position, velocity, force * self.power - 0.0025 * math.cos(3 * position), self.goal_position)
        reward = (100.0 if done else 0.0) - 0.1 * (a * a)
        return np.array(self.state), reward, done, {}


class DeviceEnv(object):
    """The device implementation of a user environment: `source` defines, as CUDA in float64,
        __device__ static void reset(double* s, int env, uint32_t k0, uint32_t k1)
        __device__ static void obs(const double* s, double* x)
        __device__ static bool step(double* s, int action, const float* a, double* reward)
    over a state of `state_dim` entries (include/mrl_b200.h, mrl_rollout_env_compile).  Set it as the class's
    `device_kind`; the observation, head and action shapes come from the class's spaces (envs.device_kind)."""

    def __init__(self, source, state_dim, name=None, ob_dim=None, categorical=None, n_out=None):
        self.source, self.state_dim, self.name = str(source), int(state_dim), name
        self.ob_dim, self.categorical, self.n_out = ob_dim, categorical, n_out

    def _key(self):
        return (self.source, self.state_dim, self.ob_dim, self.categorical, self.n_out)

    def __eq__(self, other):
        return isinstance(other, DeviceEnv) and self._key() == other._key()

    def __hash__(self):
        return hash(self._key())

    def __repr__(self):
        return "DeviceEnv(%s, ob_dim=%s, %s %s)" % (self.name, self.ob_dim,
                                                    "Categorical" if self.categorical else "DiagGauss", self.n_out)

    def bind(self, env):
        """This snippet with the shapes of `env` (an instance): Box observation (k,); Discrete(K) -> Categorical K,
        Box action (d,) -> DiagGauss d.  Raises ValueError for any other space."""
        name = getattr(getattr(env, "spec", None), "id", None) or type(env).__name__
        ob, ac = getattr(env, "observation_space", None), getattr(env, "action_space", None)
        if not isinstance(ob, Box) or len(ob.shape) != 1:
            raise ValueError("environment %s: device rollouts need a Box observation space of shape (k,), not %r"
                             % (name, ob))
        if isinstance(ac, Discrete):
            categorical, n_out = True, int(ac.n)
        elif isinstance(ac, Box) and len(ac.shape) == 1:
            categorical, n_out = False, int(ac.shape[0])
        else:
            raise ValueError("environment %s: device rollouts need a Discrete or a Box action space of shape (d,), "
                             "not %r" % (name, ac))
        return DeviceEnv(self.source, self.state_dim, name, int(ob.shape[0]), categorical, n_out)


_REGISTRY = {"CartPole-v0": CartPoleEnv, "CartPole": CartPoleEnv, "Pendulum-v0": PendulumEnv,
             "Pendulum": PendulumEnv, "Acrobot-v1": AcrobotEnv, "Acrobot": AcrobotEnv,
             "MountainCar-v0": MountainCarEnv, "MountainCar": MountainCarEnv,
             "MountainCarContinuous-v0": MountainCarContinuousEnv, "MountainCarContinuous": MountainCarContinuousEnv}


def register(id_, cls):
    """Make `cls` (called without arguments) available as make(id_)."""
    _REGISTRY[str(id_)] = cls


def _registered(name):
    """The class registered as `name`; "pkg.module:Id" imports pkg.module first.  None when unknown."""
    if ":" in name:
        module, _, id_ = name.partition(":")
        try:
            importlib.import_module(module)
        except ImportError as e:
            raise KeyError("environment %r: cannot import module %r (%s)" % (name, module, e))
        if id_ not in _REGISTRY:
            raise KeyError("environment %r: module %r registers no environment %r (registered: %s)"
                           % (name, module, id_, ", ".join(sorted(_REGISTRY))))
        return _REGISTRY[id_]
    return _REGISTRY.get(name)


def make(name):
    """gym.envs.make stand-in: a registered id, or "pkg.module:Id" (imports pkg.module, which registers Id); falls
    through to gym when it is installed and the id is unknown."""
    cls = _registered(name)
    if cls is not None:
        return cls()
    try:
        from gym.envs import make as gym_make
    except ImportError:
        raise KeyError("unknown environment %r (registered: %s; gym is not installed)" % (name, sorted(_REGISTRY)))
    return gym_make(name)


def device_kind(env):
    """The device implementation of an environment (an instance or an id): 'cartpole', 'pendulum', 'acrobot',
    'mountaincar' or 'mountaincar_continuous' for the built-ins, the class's DeviceEnv bound to its shapes for a user
    environment.  Raises ValueError for any other environment."""
    cls = _registered(env) if isinstance(env, str) else type(env)
    kind = getattr(cls, "device_kind", None)
    if kind is None:
        name = env if isinstance(env, str) else getattr(getattr(env, "spec", None), "id", type(env).__name__)
        raise ValueError("environment %s has no device implementation; device rollouts run the built-in environments "
                         "only: %s" % (name, ", ".join(sorted(_REGISTRY))))
    if isinstance(kind, DeviceEnv):
        return kind.bind(cls() if isinstance(env, str) else env)
    return kind
