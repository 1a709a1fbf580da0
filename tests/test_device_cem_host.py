"""Host side of the cross-entropy method's device population path (cem.evaluate_population_device,
cem.DEVICE_ENVS, run_cem.py --device_envs): the command-line rejections, the checks that run before any library call,
and the per-generation seed sequence with numpy's stream left to the search.  No device is used."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run_cem(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "run_cem.py"), "--agent",
                           "modular_rl.agentzoo.DeterministicAgent"] + list(args),
                          capture_output=True, text=True, timeout=300, cwd=ROOT)


def test_run_cem_device_envs_flag(tmp_path):
    out = _run_cem("--env", "CartPole-v0", "--help")
    assert out.returncode == 0 and "--device_envs" in out.stdout
    out = _run_cem("--env", "CartPole-v0", "--device_envs", "--parallel", "1", "--outfile", str(tmp_path / "a.h5"))
    assert out.returncode == 2 and "--device_envs and --parallel 1" in out.stderr
    out = _run_cem("--env", "CartPole-v0", "--device_envs", "--batch_size", "5000", "--outfile", str(tmp_path / "a.h5"))
    assert out.returncode == 2 and "at most 4096 environments; --batch_size is 5000" in out.stderr
    out = _run_cem("--env", "Hopper-v1", "--device_envs", "--outfile", str(tmp_path / "a.h5"))
    assert out.returncode == 2 and "Hopper-v1 has no device implementation" in out.stderr
    assert "CartPole-v0" in out.stderr and "Pendulum-v0" in out.stderr
    assert not os.path.exists(str(tmp_path / "a.h5.dir"))


class _GymLikeEnv(object):
    class spec:
        id = "Hopper-v1"


def test_evaluate_population_device_checks_before_any_library_call(monkeypatch):
    from modular_rl_b200 import _lib, cem, envs
    from modular_rl_b200.filters import Flatten, ZFilter
    from modular_rl_b200.misc_utils import IDENTITY

    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "lib", no_library)

    class Agent(object):
        pass
    ths = np.zeros((4, 10), np.float32)
    a = Agent()
    a.obfilter, a.rewfilter, a.policy = ZFilter((4,), clip=5), IDENTITY, object()
    with pytest.raises(ValueError, match="Hopper-v1 has no device implementation.*CartPole-v0.*Pendulum-v0"):
        cem.evaluate_population_device(_GymLikeEnv(), a, ths, 10, 0)
    with pytest.raises(TypeError, match="need a policy with a DeviceNet"):
        cem.evaluate_population_device(envs.CartPoleEnv(), a, ths, 10, 0)
    a.obfilter = Flatten()
    with pytest.raises(TypeError, match="ZFilter or IDENTITY as the observation filter"):
        cem.evaluate_population_device(envs.CartPoleEnv(), a, ths, 10, 0)
    a.obfilter, a.rewfilter = IDENTITY, (lambda r: r)
    with pytest.raises(TypeError, match="ZFilter or IDENTITY as the reward filter"):
        cem.evaluate_population_device(envs.PendulumEnv(), a, ths, 10, 0)


class _FlatAgent(object):
    def __init__(self, dim):
        self.th = np.zeros(dim)

    def get_flat(self):
        return self.th

    def set_from_flat(self, th):
        self.th = np.array(th)


def test_generation_seeds_and_numpy_stream(monkeypatch):
    """One round seed per generation, counting from cfg["seed"]; the search's randn calls are numpy's only draws."""
    from modular_rl_b200 import cem
    seeds, shapes = [], []

    def fake(env, agent, ths, timestep_limit, seed):
        seeds.append(seed)
        shapes.append((np.shape(ths), timestep_limit))
        return -np.square(np.asarray(ths) - 1.0).sum(axis=1)
    monkeypatch.setattr(cem, "DEVICE_ENVS", True)
    monkeypatch.setattr(cem, "evaluate_population_device", fake)
    np.random.seed(123)
    agent = _FlatAgent(6)
    infos = []
    cem.run_cem_algorithm("env", agent, dict(batch_size=20, n_iter=4, timestep_limit=30, seed=7), callback=infos.append)
    assert seeds == [7, 8, 9, 10]
    assert shapes == [((20, 6), 30)] * 4
    after = np.random.get_state()[1].copy()
    np.random.seed(123)
    for _ in range(4):
        np.random.randn(20, 6)
    assert np.array_equal(after, np.random.get_state()[1])
    assert infos[-1]["ymean"] > infos[0]["ymean"]
    np.testing.assert_array_equal(agent.get_flat(), infos[-1]["th"])


def test_device_envs_and_parallel_are_rejected(monkeypatch):
    from modular_rl_b200 import cem
    monkeypatch.setattr(cem, "DEVICE_ENVS", True)
    with pytest.raises(ValueError, match="choose one"):
        cem.run_cem_algorithm("env", _FlatAgent(3), dict(batch_size=4, n_iter=1, parallel=1))
