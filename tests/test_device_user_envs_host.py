"""Host side of user environments in device rollouts (envs.DeviceEnv, mrl_rollout_env_compile): NVRTC compiles the
rollout kernel around a CUDA snippet without a device, compiles a snippet once per process, reports compile errors
at the snippet's own line numbers, rejects shapes and spaces the kernel cannot run, and envs.make imports
"module:Id".  No GPU is needed."""
import ctypes as C
import os
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# CartPole-v0 restated as a user environment: rollout.cu's EnvT<MRL_ENV_CARTPOLE> with the reset drawn through
# reset_uniforms.  Its rounds must equal those of the built-in CartPole bit for bit.
CARTPOLE_SOURCE = r"""
__device__ static void reset(double* s, int env, uint32_t k0, uint32_t k1) {
  double u[4];
  reset_uniforms(env, 0, k0, k1, &u[0], &u[1]);
  reset_uniforms(env, 1, k0, k1, &u[2], &u[3]);
  for (int i = 0; i < 4; ++i) s[i] = -0.05 + (0.05 - -0.05) * u[i];
}
__device__ static void obs(const double* s, double* x) {
  for (int i = 0; i < 4; ++i) x[i] = s[i];
}
__device__ static bool step(double* s, int action, const float*, double* reward) {
  const double gravity = 9.8, masscart = 1.0, masspole = 0.1, length = 0.5, force_mag = 10.0, tau = 0.02;
  const double theta_threshold = 12 * 2 * RO_PI / 360, x_threshold = 2.4;
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
"""


def cartpole_user_env():
    """CartPoleEnv with the restated snippet as its device implementation."""
    from modular_rl_b200 import envs

    class UserCartPole(envs.CartPoleEnv):
        device_kind = envs.DeviceEnv(CARTPOLE_SOURCE, state_dim=4)
    return UserCartPole


def action_normals(seed, env, step, d):
    """The d normals of a DiagGauss action at (environment, step): entry j from Philox block j of the action purpose,
    z = sqrt(-2 log(1 - u0)) cos(2 pi u1) in float64.  -> [..., d]; column 0 is oracle.rollout.action_normal."""
    from oracle import rollout as orc
    cols = []
    for j in range(d):
        u0, u1 = orc.uniforms(seed, env, step, orc.PURPOSE_ACTION, j)
        cols.append(np.sqrt(-2.0 * np.log(1.0 - u0)) * np.cos(2.0 * np.pi * u1))
    return np.stack(cols, axis=-1)


@pytest.fixture(scope="module")
def lib():
    from modular_rl_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.lib()


def _compile(lib, source, ob_dim=4, state_dim=4, head=1, n_out=2, name=b"test_env"):
    env = C.c_int(-1)
    rc = lib.mrl_rollout_env_compile(name, source.encode() if isinstance(source, str) else source, ob_dim, state_dim,
                                     head, n_out, C.byref(env))
    return rc, env.value, lib.mrl_last_error().decode()


def test_compiles_without_a_device_and_once_per_source(lib):
    from modular_rl_b200 import device, envs
    cp = envs.device_kind(cartpole_user_env()())
    assert (cp.ob_dim, cp.state_dim, cp.categorical, cp.n_out) == (4, 4, True, 2)
    pm = envs.device_kind("examples.point_mass:PointMass-v0")
    assert (pm.ob_dim, pm.state_dim, pm.categorical, pm.n_out) == (4, 4, False, 2)
    assert cp != pm and len({cp, pm}) == 2          # the rollout cache tells the two apart
    ids = {device.rollout_env_id(cp), device.rollout_env_id(pm)}
    assert len(ids) == 2 and min(ids) >= 64
    assert device.rollout_env_info(pm) == dict(ob_dim=4, state_dim=4, categorical=False, n_out=2, act_dim=2, prob_dim=4)
    assert device.rollout_env_info(cp) == device.rollout_env_info("cartpole")
    t = time.perf_counter()
    rc, again, err = _compile(lib, CARTPOLE_SOURCE, 4, 4, 1, 2, name=b"another name")
    assert rc == 0, err
    assert again == device.rollout_env_id(cp) and time.perf_counter() - t < 0.5    # found, not compiled again
    rc, other, err = _compile(lib, CARTPOLE_SOURCE, 4, 4, 1, 3)                    # other shapes: another kernel
    assert rc == 0 and other not in ids, err
    log = device.rollout_env_log(pm)
    assert log.count("registers") == 6 and "spill" in log, log


def test_compile_error_reports_the_snippets_lines(lib):
    src = ("__device__ static void reset(double* s, int env, uint32_t k0, uint32_t k1) { s[0] = 0.0; }\n"
           "__device__ static void obs(const double* s, double* x) { x[0] = s[0]; }\n"
           "__device__ static bool step(double* s, int action, const float* a, double* reward) {\n"
           "  *reward = undefined_name;\n"
           "  return false;\n"
           "}\n")
    rc, _, err = _compile(lib, src, 1, 1, 1, 2, name=b"broken_env.cu")
    assert rc != 0
    assert "broken_env.cu(4)" in err and "undefined_name" in err, err
    rc, _, err = _compile(lib, "int x = ;", 1, 1, 1, 2, name=b"other.cu")
    assert rc != 0 and "other.cu(1)" in err, err


@pytest.mark.parametrize("args,words", [
    ((7, 4, 1, 2), "ob_dim = 7"),                 # the per-step scan carries 6 observation entries + the reward
    ((0, 4, 1, 2), "ob_dim = 0"),
    ((4, 17, 1, 2), "state_dim = 17"),
    ((4, 0, 1, 2), "state_dim = 0"),
    ((4, 4, 1, 17), "1..16 classes"),
    ((4, 4, 0, 9), "1..8 entries"),
    ((4, 4, 0, 0), "1..8 entries"),
    ((4, 4, 2, 1), "Categorical"),                # a value head does not act
])
def test_shape_limits_are_rejected(lib, args, words):
    rc, _, err = _compile(lib, CARTPOLE_SOURCE, *args)
    assert rc != 0 and words in err, err


def test_unknown_ids_fail(lib):
    ob, st, head, n_out = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    for env in (5, 63, 4095):
        assert lib.mrl_rollout_env_info(env, C.byref(ob), C.byref(st), C.byref(head), C.byref(n_out)) != 0
        assert b"unknown env" in lib.mrl_last_error()
    buf = C.create_string_buffer(64)
    assert lib.mrl_rollout_env_log(4095, buf, 64) != 0
    h = C.c_void_p()
    assert lib.mrl_rollout_create(C.byref(h), 0, 4095, 16, 10) != 0


def test_unsupported_spaces_are_rejected():
    from modular_rl_b200 import envs
    from modular_rl_b200.spaces import Box, Discrete

    class Env(object):
        device_kind = envs.DeviceEnv(CARTPOLE_SOURCE, state_dim=4)

        def __init__(self, ob, ac):
            self.observation_space, self.action_space = ob, ac

    box4 = Box(-np.ones(4), np.ones(4))
    assert envs.device_kind(Env(box4, Discrete(3))).n_out == 3
    with pytest.raises(ValueError, match="observation space"):
        envs.device_kind(Env(Discrete(4), Discrete(2)))
    with pytest.raises(ValueError, match="observation space"):
        envs.device_kind(Env(Box(-np.ones((2, 2)), np.ones((2, 2))), Discrete(2)))
    with pytest.raises(ValueError, match="action space"):
        envs.device_kind(Env(box4, Box(-np.ones((2, 3)), np.ones((2, 3)))))
    with pytest.raises(ValueError, match="action space"):
        envs.device_kind(Env(box4, None))
    with pytest.raises(ValueError, match="no device implementation"):
        envs.device_kind(object())


def test_make_module_id():
    from modular_rl_b200 import envs
    env = envs.make("examples.point_mass:PointMass-v0")
    assert type(env).__name__ == "PointMassEnv" and env.spec.id == "PointMass-v0"
    assert env.spec.max_episode_steps == 200
    assert type(envs.make("PointMass-v0")) is type(env)          # registered by the import
    with pytest.raises(KeyError, match="cannot import module"):
        envs.make("examples.no_such_module:PointMass-v0")
    with pytest.raises(KeyError, match="registers no environment"):
        envs.make("examples.point_mass:NoSuchEnv-v0")


def test_point_mass_host_dynamics():
    from modular_rl_b200 import envs
    env = envs.make("examples.point_mass:PointMass-v0")
    np.random.seed(0)
    ob = env.reset()
    assert ob.shape == (4,) and np.all(np.abs(ob[:2]) <= 1.0) and np.all(ob[2:] == 0.0)
    x, y = ob[:2]
    ob, rew, done, _ = env.step(np.array([3.0, -0.5], np.float32))           # the force is clipped to [-1, 1]
    vx, vy = 0.0 + 0.1 * 1.0, 0.0 + 0.1 * -0.5
    np.testing.assert_array_equal(ob, [x + 0.1 * vx, y + 0.1 * vy, vx, vy])
    assert rew == -(ob[0] ** 2 + ob[1] ** 2) - 0.01 * (1.0 + 0.25) and not done
    env.state = np.array([0.01, 0.0, 0.0, 0.0])
    assert env.step(np.zeros(2, np.float32))[2]                              # near the origin and at rest


def test_action_normals_extend_action_normal():
    from oracle import rollout as orc
    envs_, steps = np.arange(50), np.arange(50) * 3
    z = action_normals(11, envs_, steps, 6)
    assert z.shape == (50, 6)
    np.testing.assert_array_equal(z[:, 0], orc.action_normal(11, envs_, steps))
    assert np.all(z[:, 1] != z[:, 0]) and abs(z.mean()) < 0.3 and 0.7 < z.std() < 1.3
