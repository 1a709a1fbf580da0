"""Host side of the device-resident rollouts (core.do_rollouts_device, run_pg.py --device_envs): the Philox stream the
oracle restates, path assembly from the compacted arrays, the flag and every configuration rejected before anything
runs.  No GPU is needed."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_philox_known_answers():
    """Random123's kat_vectors for philox4x32-10 (same constants and round as curand_philox4x32_x.h)."""
    from oracle import rollout as orc
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        got = orc.philox4x32_10(np.array(ctr, np.uint32), key)
        assert tuple(int(v) for v in got) == want


def test_oracle_uniform_mapping_and_resets():
    from oracle import rollout as orc
    assert orc.u53(0, 0) == 0.0 and orc.u53(0xFFFFFFFF, 0xFFFFFFFF) == 1.0 - 2.0 ** -53
    s = orc.reset_states("cartpole", 7, np.arange(100))
    assert s.shape == (100, 4) and np.all(np.abs(s) <= 0.05)
    p = orc.reset_states("pendulum", 7, np.arange(100))
    assert np.all(np.abs(p[:, 0]) <= np.pi) and np.all(np.abs(p[:, 1]) <= 1.0)
    assert not np.array_equal(orc.reset_states("cartpole", 8, [0]), s[:1])      # the seed is the key


def test_device_paths_assembly():
    from modular_rl_b200 import core
    lengths = np.array([3, 1, 2], np.int32)
    T = int(lengths.sum())
    out = dict(lengths=lengths, terminated=np.array([1, 0, 1], np.uint8),
               observation=np.arange(T * 4, dtype=np.float64).reshape(T, 4), action=np.array([0, 1, 1, 0, 1, 0], np.int32),
               prob=np.full((T, 2), 0.5, np.float32), reward=np.ones(T))
    paths = core.device_paths(out, categorical=True)
    assert [core.pathlength(p) for p in paths] == [3, 1, 2]
    assert [p["terminated"] for p in paths] == [True, False, True]
    assert list(paths[0]) == ["observation", "action", "prob", "reward", "terminated"]
    for p in paths:
        assert p["observation"].dtype == np.float64 and p["observation"].shape[1] == 4
        assert p["action"].dtype == np.int64 and p["prob"].dtype == np.float32 and p["reward"].dtype == np.float64
    np.testing.assert_array_equal(paths[2]["observation"], out["observation"][4:6])
    gauss = dict(out, action=np.arange(T, dtype=np.float32).reshape(T, 1))
    gp = core.device_paths(gauss, categorical=False)
    assert gp[1]["action"].dtype == np.float32 and gp[1]["action"].shape == (1, 1) and gp[1]["action"][0, 0] == 3.0


class _GymLikeEnv(object):
    class spec:
        id = "Hopper-v1"


def test_rejects_env_without_device_implementation():
    from modular_rl_b200 import core, envs
    with pytest.raises(ValueError, match="Hopper-v1 has no device implementation.*CartPole-v0.*Pendulum-v0"):
        envs.device_kind(_GymLikeEnv())
    with pytest.raises(ValueError, match="built-in environments only"):
        core.check_device_rollouts(_GymLikeEnv(), None)
    with pytest.raises(ValueError, match="Walker2d-v1 has no device implementation"):
        envs.device_kind("Walker2d-v1")


def _cpu_agent():
    """An agent whose parts are host objects: the checks run before any device call."""
    from modular_rl_b200.filters import ZFilter
    from modular_rl_b200.misc_utils import IDENTITY

    class Agent(object):
        pass
    a = Agent()
    a.obfilter, a.rewfilter = ZFilter((4,), clip=5), IDENTITY
    a.policy = object()
    return a


def test_rejects_other_filters_and_policies():
    from modular_rl_b200 import core, envs
    from modular_rl_b200.filters import Flatten
    env = envs.CartPoleEnv()
    a = _cpu_agent()
    a.obfilter = Flatten()
    with pytest.raises(TypeError, match="ZFilter or IDENTITY as the observation filter"):
        core.check_device_rollouts(env, a)
    a = _cpu_agent()
    a.rewfilter = lambda r: r
    with pytest.raises(TypeError, match="ZFilter or IDENTITY as the reward filter"):
        core.check_device_rollouts(env, a)
    a = _cpu_agent()
    with pytest.raises(TypeError, match="need a policy with a DeviceNet"):
        core.check_device_rollouts(env, a)


def test_device_and_vec_envs_together_are_rejected(monkeypatch):
    from modular_rl_b200 import core
    monkeypatch.setattr(core, "DEVICE_ENVS", 8)
    monkeypatch.setattr(core, "VEC_ENVS", 4)
    cfg = dict(parallel=0, timesteps_per_batch=10, timestep_limit=5)
    with pytest.raises(ValueError, match="both set; choose one"):
        core.get_paths(None, None, cfg, iter([0]))


def _run_pg(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "run_pg.py")] + list(args), capture_output=True,
                          text=True, timeout=300, cwd=ROOT)


def test_run_pg_device_envs_flag():
    out = _run_pg("--help")
    assert out.returncode == 0 and "--device_envs" in out.stdout
    out = _run_pg("--device_envs", "64", "--vec_envs", "16", "--env", "CartPole-v0")
    assert out.returncode == 2 and "--device_envs and --vec_envs" in out.stderr
    out = _run_pg("--device_envs", "-1")
    assert out.returncode == 2 and "--device_envs must be >= 0" in out.stderr


def test_do_rollouts_device_round_structure(monkeypatch):
    """do_rollouts_device around a stand-in for the device handle: it is built from the environment, each round takes
    one seed, rounds stop strictly above the quota, the filters take the returned states and a data-parallel
    `pushed` state takes the Chan merge of the rounds' own samples."""
    from modular_rl_b200 import core, envs
    from modular_rl_b200.device import DeviceNet
    from modular_rl_b200.filters import ZFilter
    from modular_rl_b200.running_stat import RunningStat
    made, seeds, pushed_samples = [], [], []

    class FakeRollouts(object):
        categorical = True

        def __init__(self, env, n_envs, timestep_limit, device=None):
            made.append((envs.device_kind(env), n_envs, timestep_limit, device))
            self.n = n_envs

        def run(self, net, seed, stochastic, obfilter, rewfilter):
            seeds.append(seed)
            lengths = np.full(self.n, 10, np.int32)
            T = int(lengths.sum())
            x = np.random.default_rng(seed).standard_normal((T, 4))
            pushed_samples.append(x)
            own = RunningStat((4,))
            for row in x:
                own.push(row)
            (n, M, S), _, _, _ = obfilter
            return dict(lengths=lengths, terminated=np.zeros(self.n, np.uint8), observation=x,
                        action=np.zeros(T, np.int32), prob=np.full((T, 2), 0.5, np.float32), reward=np.ones(T),
                        ob_state=(n + T, M + 1.0, S + 1.0), ob_pushed=own.state(), rew_state=None, rew_pushed=None)

    class Agent(object):
        pass
    from modular_rl_b200.misc_utils import IDENTITY
    agent = Agent()
    agent.obfilter, agent.rewfilter = ZFilter((4,), clip=5), IDENTITY
    agent.obfilter.start_round()
    net = DeviceNet.__new__(DeviceNet)
    net.device = 0
    agent.policy = Agent()
    agent.policy.net = net
    monkeypatch.setattr(core, "DeviceRollouts", FakeRollouts)
    monkeypatch.setattr(core, "_device_rollouts", {})
    from itertools import count
    it = count(5, 2)
    paths = core.do_rollouts_device(envs.CartPoleEnv(), agent, 40, 100, it, 4)
    assert made == [("cartpole", 4, 40, 0)]
    assert seeds == [5, 7, 9] and next(it) == 11                   # 40 + 40 <= 100 < 120: three rounds, one seed each
    assert len(paths) == 12 and all(core.pathlength(p) == 10 for p in paths)
    assert agent.obfilter.rs.n == 120 and np.all(agent.obfilter.rs.mean == 3.0)
    ref = RunningStat((4,))
    for row in np.concatenate(pushed_samples):
        ref.push(row)
    assert agent.obfilter.pushed.n == 120
    np.testing.assert_allclose(agent.obfilter.pushed.mean, ref.mean, rtol=1e-12)
    np.testing.assert_allclose(agent.obfilter.pushed.state()[2], ref.state()[2], rtol=1e-12)
