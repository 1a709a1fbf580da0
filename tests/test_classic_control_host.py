"""Acrobot-v1, MountainCar-v0 and MountainCarContinuous-v0 (envs.py) on the host: the dynamics against independent
statements of the same physics, the boundary rules, the spaces and ids, the shapes the C ABI reports for every device
environment, and the Philox reset mapping of the device rollouts for the three environments.  No GPU is needed."""
import ctypes as C
import math
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reset_states(kind, seed, envs):
    """Start states of environments `envs` of a device round of a new environment (rollout.cu, DESIGN.md 4b), on the
    Philox stream of oracle/rollout.py: Acrobot takes u0, u1 of blocks 0 and 1 as -0.1 + 0.2 u (CartPole's order);
    both MountainCars take block 0's u0 as position = -0.6 + (-0.4 - -0.6) u0, velocity 0."""
    from oracle import rollout as orc
    envs = np.asarray(envs)
    if kind == "acrobot":
        a0, a1 = orc.uniforms(seed, envs, 0, orc.PURPOSE_RESET, 0)
        b0, b1 = orc.uniforms(seed, envs, 0, orc.PURPOSE_RESET, 1)
        return -0.1 + (0.1 - -0.1) * np.stack([a0, a1, b0, b1], axis=-1)
    assert kind in ("mountaincar", "mountaincar_continuous"), kind
    u0, _ = orc.uniforms(seed, envs, 0, orc.PURPOSE_RESET, 0)
    return np.stack([-0.6 + (-0.4 - -0.6) * u0, np.zeros_like(u0)], axis=-1)


def _lagrangian_qdd(s, tau):
    """Acrobot accelerations from M(q) qdd = [0, tau] - C(q, qd) - G(q), angles from the hanging position (Spong's
    manipulator form), independent of the derivative's closed form in envs.py."""
    m1 = m2 = l1 = 1.0
    lc1 = lc2 = 0.5
    I1 = I2 = 1.0
    g = 9.8
    t1, t2, w1, w2 = s
    M = np.array([[m1 * lc1 ** 2 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * np.cos(t2)) + I1 + I2,
                   m2 * (lc2 ** 2 + l1 * lc2 * np.cos(t2)) + I2],
                  [m2 * (lc2 ** 2 + l1 * lc2 * np.cos(t2)) + I2, m2 * lc2 ** 2 + I2]])
    h = m2 * l1 * lc2 * np.sin(t2)
    Cv = np.array([-h * (w2 ** 2 + 2 * w1 * w2), h * w1 ** 2])
    G = np.array([(m1 * lc1 + m2 * l1) * g * np.sin(t1) + m2 * lc2 * g * np.sin(t1 + t2), m2 * lc2 * g * np.sin(t1 + t2)])
    return np.linalg.solve(M, np.array([0.0, tau]) - Cv - G)


def _acrobot():
    from modular_rl_b200 import envs
    return envs.AcrobotEnv()


def test_acrobot_derivative_matches_lagrangian_form():
    env = _acrobot()
    rng = np.random.default_rng(0)
    for _ in range(1000):
        s = [rng.uniform(-np.pi, np.pi), rng.uniform(-np.pi, np.pi), rng.uniform(-4 * np.pi, 4 * np.pi),
             rng.uniform(-9 * np.pi, 9 * np.pi)]
        tau = float(rng.choice([-1.0, 0.0, 1.0]))
        d = env._dsdt(s + [tau])
        assert d[0] == s[2] and d[1] == s[3] and d[4] == 0.0
        want = _lagrangian_qdd(s, tau)
        assert np.linalg.norm(np.array(d[2:4]) - want) <= 1e-12 * np.linalg.norm(want), (s, tau, d, want)


def _rk4(f, y, h):
    k1 = f(y)
    k2 = f(y + h / 2 * k1)
    k3 = f(y + h / 2 * k2)
    k4 = f(y + h * k3)
    return y + h / 6 * (k1 + 2 * k2 + 2 * k3 + k4)


def test_acrobot_step_is_one_rk4_step():
    """One step from small velocities (no wrap, no clip) against scipy's solve_ivp (DOP853, rtol 1e-12) on the
    Lagrangian form.  The step is one classical RK4 step of dt = 0.2: it equals an independent RK4 step to 1e-12, its
    distance to the exact solution is RK4's local error (about 3e-4 here, where gravity alone gives accelerations near
    10; one explicit Euler step misses by about 1e-2), and two half steps shrink that error at least tenfold, as a
    fourth-order method must (2^5 = 32 in the limit)."""
    from scipy.integrate import solve_ivp
    env = _acrobot()
    rng = np.random.default_rng(1)
    for _ in range(20):
        s0 = rng.uniform(-0.1, 0.1, size=4)
        a = int(rng.integers(3))
        tau = env.AVAIL_TORQUE[a]

        def f(y):
            return np.concatenate([y[2:], _lagrangian_qdd(y, tau)])
        ref = solve_ivp(lambda _, y: f(y), (0.0, env.dt), s0, method="DOP853", rtol=1e-12, atol=1e-14).y[:, -1]
        env.state = s0.copy()
        env.step(a)
        err = np.abs(env.state - ref).max()
        assert np.abs(env.state - _rk4(f, s0, env.dt)).max() <= 1e-12 * np.abs(ref).max()
        assert err < 1e-3, (env.state, ref)
        half = _rk4(f, _rk4(f, s0, env.dt / 2), env.dt / 2)
        assert np.abs(half - ref).max() < err / 10
        assert np.abs(s0 + env.dt * f(s0) - ref).max() > 10 * err


def test_acrobot_wrap_bound_terminal_and_rewards():
    env = _acrobot()
    # wrap: an angle carried past pi comes back by exactly 2 pi, with the while loop's subtraction
    env.state = np.array([np.pi - 0.01, -np.pi + 0.01, 2.0, -2.0])
    ns = env._rk4(list(env.state) + [0.0])
    assert ns[0] > np.pi and ns[1] < -np.pi
    env.step(1)
    assert env.state[0] == ns[0] - 2 * np.pi and env.state[1] == ns[1] + 2 * np.pi
    assert -np.pi <= env.state[0] <= np.pi and -np.pi <= env.state[1] <= np.pi
    assert env._wrap(3 * np.pi + 0.5, -np.pi, np.pi) == (3 * np.pi + 0.5) - 2 * np.pi - 2 * np.pi
    # bound: velocities at their limits are clipped to exactly the bound
    rng = np.random.default_rng(2)
    clipped = 0
    for _ in range(200):
        s = np.array([rng.uniform(-np.pi, np.pi), rng.uniform(-np.pi, np.pi), rng.choice([-1, 1]) * 4 * np.pi,
                      rng.choice([-1, 1]) * 9 * np.pi])
        a = int(rng.integers(3))
        ns = env._rk4(list(s) + [env.AVAIL_TORQUE[a]])
        env.state = s.copy()
        env.step(a)
        assert env.state[2] == min(max(ns[2], -4 * np.pi), 4 * np.pi)
        assert env.state[3] == min(max(ns[3], -9 * np.pi), 9 * np.pi)
        clipped += abs(env.state[2]) == 4 * np.pi or abs(env.state[3]) == 9 * np.pi
    assert clipped > 0
    # terminal: the tip above the bar ends the episode with reward 0; hanging gives -1 and goes on
    env.state = np.array([np.pi, 0.0, 0.0, 0.0])
    ob, r, done, _ = env.step(1)
    assert done and r == 0.0
    assert -math.cos(env.state[0]) - math.cos(env.state[1] + env.state[0]) > 1.0
    env.state = np.zeros(4)
    ob, r, done, _ = env.step(1)
    assert not done and r == -1.0 and np.abs(env.state).max() < 1e-15    # cos(-pi / 2) is not exactly 0
    assert ob.shape == (6,) and ob[0] == 1.0 and ob[2] == 1.0


def test_mountain_car_step_wall_and_goal():
    from modular_rl_b200 import envs
    env = envs.MountainCarEnv()
    env.state = np.array([-0.5, 0.01])
    ob, r, done, _ = env.step(2)
    v = 0.01 + (1 * 0.001 + math.cos(3 * -0.5) * -0.0025)
    assert r == -1.0 and not done and np.array_equal(ob, [-0.5 + v, v]) and np.array_equal(env.state, ob)
    # the velocity clip, then the position clip at the left wall zeroes a negative velocity
    env.state = np.array([-1.19, -0.069])
    ob, r, done, _ = env.step(0)
    assert ob[0] == -1.2 and ob[1] == 0.0 and not done
    env.state = np.array([-0.5, -0.2])
    env.step(1)
    assert env.state[1] == -0.07
    # goal: position >= 0.5 with a velocity >= 0 ends the episode, reward -1 still
    env.state = np.array([0.49, 0.05])
    ob, r, done, _ = env.step(2)
    assert done and r == -1.0 and ob[0] >= 0.5
    env.state = np.array([0.59, 0.07])
    ob, r, done, _ = env.step(2)
    assert ob[0] == 0.6 and done


def test_mountain_car_continuous_force_penalty_and_goal():
    from modular_rl_b200 import envs
    env = envs.MountainCarContinuousEnv()
    env.state = np.array([-0.5, 0.0])
    ob, r, done, _ = env.step(np.array([5.0], np.float32))
    v = 0.0 + (1.0 * 0.0015 - 0.0025 * math.cos(3 * -0.5))
    assert np.array_equal(ob, [-0.5 + v, v]) and not done
    assert r == 0.0 - 0.1 * 25.0                        # the penalty takes the unclipped action
    env.state = np.array([-0.5, 0.0])
    _, r, _, _ = env.step(np.array([-0.25], np.float32))
    a = float(np.float32(-0.25))
    assert r == -0.1 * (a * a)
    env.state = np.array([0.44, 0.02])
    ob, r, done, _ = env.step([0.5])
    assert done and ob[0] >= 0.45 and r == 100.0 - 0.1 * 0.25
    env.state = np.array([-1.19, -0.07])
    ob, _, _, _ = env.step([-1.0])
    assert ob[0] == -1.2 and ob[1] == 0.0


def test_spaces_ids_limits_make_and_device_kind():
    from modular_rl_b200 import envs
    from modular_rl_b200.spaces import Box, Discrete
    cases = [("Acrobot-v1", "Acrobot", envs.AcrobotEnv, 500, "acrobot", 6, 3),
             ("MountainCar-v0", "MountainCar", envs.MountainCarEnv, 200, "mountaincar", 2, 3),
             ("MountainCarContinuous-v0", "MountainCarContinuous", envs.MountainCarContinuousEnv, 999,
              "mountaincar_continuous", 2, None)]
    for id_, short, cls, limit, kind, ob_dim, n in cases:
        for name in (id_, short):
            env = envs.make(name)
            assert type(env) is cls and envs.device_kind(name) == kind and envs.device_kind(env) == kind
        assert env.spec.id == id_ and env.spec.max_episode_steps == limit == env.spec.timestep_limit
        assert isinstance(env.observation_space, Box) and env.observation_space.shape == (ob_dim,)
        if n is None:
            assert isinstance(env.action_space, Box) and env.action_space.shape == (1,)
            assert np.array_equal(env.action_space.low, [-1.0]) and np.array_equal(env.action_space.high, [1.0])
        else:
            assert isinstance(env.action_space, Discrete) and env.action_space.n == n
        ob = env.reset()
        assert ob.shape == (ob_dim,)
    hi = envs.AcrobotEnv().observation_space.high
    assert np.array_equal(hi, [1, 1, 1, 1, 4 * np.pi, 9 * np.pi])
    mc = envs.MountainCarEnv().observation_space
    assert np.array_equal(mc.low, [-1.2, -0.07]) and np.array_equal(mc.high, [0.6, 0.07])
    np.random.seed(3)
    for _ in range(50):
        s = envs.MountainCarEnv().reset()
        assert -0.6 <= s[0] <= -0.4 and s[1] == 0.0
        a = envs.AcrobotEnv()
        a.reset()
        assert np.all(np.abs(a.state) <= 0.1)
    with pytest.raises(KeyError):
        envs.make("Acrobot-v0")


@pytest.fixture(scope="module")
def lib():
    from modular_rl_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.lib()


def test_rollout_env_info(lib):
    from modular_rl_b200 import _lib
    from modular_rl_b200.device import rollout_env_info
    want = {"cartpole": (4, 4, _lib.CATEGORICAL, 2), "pendulum": (3, 2, _lib.GAUSS, 1),
            "acrobot": (6, 4, _lib.CATEGORICAL, 3), "mountaincar": (2, 2, _lib.CATEGORICAL, 3),
            "mountaincar_continuous": (2, 2, _lib.GAUSS, 1)}
    assert set(want) == set(_lib.DEVICE_ENVS)
    for kind, w in want.items():
        v = [C.c_int(-1) for _ in range(4)]
        assert lib.mrl_rollout_env_info(_lib.DEVICE_ENVS[kind], *[C.byref(x) for x in v]) == 0
        assert tuple(x.value for x in v) == w, kind
    info = rollout_env_info("acrobot")
    assert info == dict(ob_dim=6, state_dim=4, categorical=True, n_out=3, act_dim=1, prob_dim=3)
    info = rollout_env_info("mountaincar_continuous")
    assert info == dict(ob_dim=2, state_dim=2, categorical=False, n_out=1, act_dim=1, prob_dim=2)
    v = C.c_int()
    assert lib.mrl_rollout_env_info(5, C.byref(v), C.byref(v), C.byref(v), C.byref(v)) != 0
    msg = lib.mrl_last_error()
    assert b"unknown env 5" in msg and b"MRL_ENV_ACROBOT" in msg and b"MRL_ENV_MOUNTAIN_CAR_CONTINUOUS" in msg


def test_reset_mapping_in_range():
    a = reset_states("acrobot", 7, np.arange(200))
    assert a.shape == (200, 4) and np.all(np.abs(a) <= 0.1) and a.std() > 0.03
    for kind in ("mountaincar", "mountaincar_continuous"):
        m = reset_states(kind, 7, np.arange(200))
        assert m.shape == (200, 2) and np.all((m[:, 0] >= -0.6) & (m[:, 0] <= -0.4)) and np.all(m[:, 1] == 0.0)
    assert np.array_equal(reset_states("mountaincar", 7, [3]), reset_states("mountaincar_continuous", 7, [3]))
    assert not np.array_equal(reset_states("acrobot", 8, [0]), a[:1])
