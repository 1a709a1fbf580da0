"""Two classic-control environments with the old gym API (reset() -> ob, step(a) -> ob, rew, done,
info) so that BASELINE config 1 (CartPole-v0 TrpoAgent via run_pg.py) and the reference's coverage
smoke (Pendulum, coverage.sh:7) run without gym, which is not installed here.  Dynamics follow the
published classic-control equations (Barto-Sutton-Anderson cart-pole; torque-limited pendulum)."""
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


_REGISTRY = {"CartPole-v0": CartPoleEnv, "CartPole": CartPoleEnv, "Pendulum-v0": PendulumEnv,
             "Pendulum": PendulumEnv}


def make(name):
    """gym.envs.make stand-in; falls through to gym when it is installed and the id is unknown."""
    if name in _REGISTRY:
        return _REGISTRY[name]()
    try:
        from gym.envs import make as gym_make
    except ImportError:
        raise KeyError("unknown environment %r (built in: %s; gym is not installed)" % (name, sorted(_REGISTRY)))
    return gym_make(name)


def device_kind(env):
    """The device implementation of a built-in environment (an instance or an id): 'cartpole' or 'pendulum'.
    Raises ValueError for any other environment."""
    cls = _REGISTRY.get(env) if isinstance(env, str) else type(env)
    kind = getattr(cls, "device_kind", None)
    if kind is None:
        name = env if isinstance(env, str) else getattr(getattr(env, "spec", None), "id", type(env).__name__)
        raise ValueError("environment %s has no device implementation; device rollouts run the built-in environments "
                         "only: %s" % (name, ", ".join(sorted(_REGISTRY))))
    return kind
