"""User environments in device rollouts on the GPU (envs.DeviceEnv, the rollout kernel compiled by NVRTC): CartPole
restated as a user environment gives the built-in CartPole's rounds bit for bit, and PointMass-v0 (examples/, a
DiagGauss head with d = 2) replays through its host class, draws its actions from the oracle's normals, filters as
the lockstep oracle and scores populations as cem.evaluate_population.  Then whole runs of run_pg.py and run_cem.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import test_device_user_envs_host as uh
import test_gpu_device_envs as de

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
PM = "examples.point_mass:PointMass-v0"


def _filters(d, on):
    if not on:
        return None, None
    return (((de.OB_STATE[0], de.OB_STATE[1][:d], de.OB_STATE[2][:d]), True, True, 5.0),
            (de.REW_STATE, False, True, 10.0))


def _equal(a, b, keys):
    for k in keys:
        if a[k] is None:
            assert b[k] is None, k
        elif isinstance(a[k], tuple):
            assert a[k][0] == b[k][0] and np.array_equal(a[k][1], b[k][1]) and np.array_equal(a[k][2], b[k][2]), k
        else:
            assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k


ROW_KEYS = ("lengths", "terminated", "observation", "action", "prob", "reward", "states", "ob_state", "ob_pushed",
            "rew_state", "rew_pushed")


@pytest.mark.parametrize("N,stochastic,filters", [(1, True, True), (33, True, False), (33, False, True),
                                                  (4096, True, True)])
def test_restated_cartpole_equals_builtin(N, stochastic, filters):
    from modular_rl_b200.device import DeviceRollouts
    pol = de._policy("cartpole", scale=0.3, seed=3)
    ob, rew = _filters(4, filters)
    got = DeviceRollouts(uh.cartpole_user_env()(), N, 200).run(pol.net, 77, stochastic, ob, rew, want_states=True)
    want = DeviceRollouts("CartPole-v0", N, 200).run(pol.net, 77, stochastic, ob, rew, want_states=True)
    _equal(got, want, ROW_KEYS)
    assert got["lengths"].sum() > N


@pytest.mark.parametrize("want_rows", [True, False])
def test_restated_cartpole_population_equals_builtin(want_rows):
    import test_gpu_device_cem as dc
    from modular_rl_b200.device import DeviceRollouts
    dims = [4, 32, 2]
    th = dc._thetas(dims, 300, 0.5, seed=5)
    ob, rew = _filters(4, True)
    kw = dict(want_rows=want_rows, want_states=want_rows)
    got = DeviceRollouts(uh.cartpole_user_env()(), 300, 200).run_population(dims, "relu", th, 9, ob, rew, **kw)
    want = DeviceRollouts("CartPole-v0", 300, 200).run_population(dims, "relu", th, 9, ob, rew, **kw)
    _equal(got, want, ("returns", "lengths", "terminated", "ob_state", "rew_state")
           + (("observation", "action", "prob", "reward", "states") if want_rows else ()))


def _pm_policy(seed=0, scale=0.3):
    from modular_rl_b200 import core
    np.random.seed(seed)
    pol = core.StochPolicyMLP(4, [32, 32], core.DiagGauss(2), "tanh")
    th = pol.get_flat()
    th = np.random.default_rng(seed).standard_normal(th.size).astype(np.float32) * scale
    th[-2:] = [-0.5, 0.3]                           # two different standard deviations
    pol.set_from_flat(th)
    return pol


def test_point_mass_replays_through_host_class():
    from modular_rl_b200 import envs
    from modular_rl_b200.device import DeviceRollouts
    from oracle import rollout as orc
    pol = _pm_policy()
    N, seed = 300, 123
    ob, rew = _filters(4, True)
    out = DeviceRollouts(PM, N, 200).run(pol.net, seed, True, ob, rew, want_states=True)
    off, sl = de._split(out)
    lengths = out["lengths"]
    assert out["action"].shape == (off[-1], 2) and out["prob"].shape == (off[-1], 4)
    assert (lengths == 200).any()
    env = envs.make(PM)
    u0, u1 = orc.uniforms(seed, np.arange(N), 0, orc.PURPOSE_RESET, 0)
    np.testing.assert_array_equal(out["states"][off[:-1]][:, :2], np.stack([-1.0 + 2.0 * u0, -1.0 + 2.0 * u1], 1))
    for i in range(N):
        st, act, rw = out["states"][sl[i]], out["action"][sl[i]], out["reward"][sl[i]]
        for t in range(lengths[i]):
            env.state = st[t].copy()
            nxt, r, done, _ = env.step(act[t])
            assert abs(r - rw[t]) <= 1e-12 * max(1.0, abs(r)), (i, t, r, rw[t])
            if t + 1 < lengths[i]:
                np.testing.assert_allclose(nxt, st[t + 1], rtol=0, atol=1e-12)
                assert not done, (i, t)
            else:
                assert done == bool(out["terminated"][i]), (i, t)
        # actions: float32(z) * std + mean with the oracle's normals of (environment, step), entry j from block j
        z = uh.action_normals(seed, i, np.arange(lengths[i]), 2)
        prob = out["prob"][sl[i]]
        np.testing.assert_array_equal(act, orc.gauss_action(prob[:, :2], prob[:, 2:], z))
    np.testing.assert_allclose(out["prob"][:, 2:], np.broadcast_to(np.exp([-0.5, 0.3]), (off[-1], 2)), rtol=1e-6)
    # filters: the lockstep oracle over the raw observations (= the states) and the raw rewards
    raw = [out["states"][sl[i]] for i in range(N)]
    want, rs, pushed = orc.lockstep_zfilter(raw, lengths, (de.OB_STATE[0], de.OB_STATE[1], de.OB_STATE[2]))
    for i in range(N):
        np.testing.assert_allclose(out["observation"][sl[i]], want[i], rtol=0, atol=1e-10)
    assert out["ob_state"][0] == rs.n
    np.testing.assert_allclose(out["ob_state"][1], rs.M, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(out["ob_state"][2], rs.S, rtol=1e-10, atol=1e-12)
    rrs, _ = orc.lockstep_rewards([out["reward"][sl[i]] for i in range(N)], lengths, de.REW_STATE)
    assert out["rew_state"][0] == rrs.n
    np.testing.assert_allclose(out["rew_state"][1], rrs.M, rtol=1e-10)
    np.testing.assert_allclose(out["rew_state"][2], rrs.S, rtol=1e-10)
    # deterministic actions are the means
    det = DeviceRollouts(PM, N, 200).run(pol.net, seed, False, None, None)
    np.testing.assert_array_equal(det["action"], det["prob"][:, :2])


def test_point_mass_population_equals_host_path(monkeypatch):
    import examples.point_mass as pm
    import test_gpu_device_cem as dc
    from modular_rl_b200 import agentzoo, cem
    from oracle import rollout as orc
    env = pm.PointMassEnv()
    np.random.seed(0)
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[32, 32], filter=0))
    M, seed = 64, 31
    th = dc._thetas(agent.policy.dims, M, 0.5, seed=4)
    dev = cem.evaluate_population_device(env, agent, th, 200, seed)
    u0, u1 = orc.uniforms(seed, np.arange(M), 0, orc.PURPOSE_RESET, 0)
    starts = np.stack([-1.0 + 2.0 * u0, -1.0 + 2.0 * u1, np.zeros(M), np.zeros(M)], 1)
    made = [0]

    def reset(self):
        self.state = starts[made[0]].copy()
        made[0] += 1
        return np.array(self.state)
    monkeypatch.setattr(pm.PointMassEnv, "reset", reset)
    host = cem.evaluate_population(env, agent, th, 200)
    assert made[0] == M
    assert np.array_equal(host, dev), (host, dev)
    assert len(set(dev.tolist())) > 1


def test_policy_head_must_fit():
    from modular_rl_b200 import core
    from modular_rl_b200.device import DeviceRollouts
    ro = DeviceRollouts(PM, 8, 20)
    with pytest.raises(RuntimeError, match="DiagGauss head with 2 outputs"):
        ro.run(de._policy("cartpole").net, 1)                     # Categorical, 4 inputs: observations fit
    np.random.seed(0)
    three = core.StochPolicyMLP(4, [8], core.DiagGauss(3), "tanh")
    with pytest.raises(RuntimeError, match="DiagGauss head with 2 outputs"):
        ro.run(three.net, 1)
    with pytest.raises(RuntimeError, match="actions take 2 outputs"):
        ro.run_population([4, 8, 3], "tanh", np.zeros((4, 4 * 8 + 8 + 8 * 3 + 3), np.float32), 1)


def test_two_user_environments_in_one_process():
    from modular_rl_b200.device import DeviceRollouts
    cp = DeviceRollouts(uh.cartpole_user_env()(), 64, 100)
    pm = DeviceRollouts(PM, 64, 100)
    assert cp.categorical and not pm.categorical
    a = cp.run(de._policy("cartpole").net, 5)
    b = pm.run(_pm_policy().net, 5)
    a2 = cp.run(de._policy("cartpole").net, 5)
    assert a["action"].dtype == np.int32 and b["action"].shape[1] == 2
    assert np.array_equal(a["action"], a2["action"]) and np.array_equal(a["reward"], a2["reward"])


def test_run_pg_point_mass_learns(tmp_path):
    stdout = de._run_pg(["--env", PM, "--agent", "modular_rl.agentzoo.TrpoAgent", "--n_iter", "20",
                         "--timesteps_per_batch", "20000", "--seed", "0", "--gamma", "0.99", "--lam", "0.97",
                         "--device_envs", "256", "--outfile", str(tmp_path / "a.h5")])
    rews = [float(ln.split()[-1]) for ln in stdout.splitlines() if ln.startswith("EpRewMean")]
    assert len(rews) == 20
    # measured on a B200: -21106 at iteration 1 (the untrained policy drifts away), -9.5 over iterations 18-20
    assert np.mean(rews[-3:]) > -100.0 and np.mean(rews[-3:]) > 0.01 * rews[0], rews


def test_run_cem_point_mass_device_search(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "run_cem.py"), "--env", PM, "--agent",
                          "modular_rl.agentzoo.DeterministicAgent", "--device_envs", "--device_search", "--n_iter", "3",
                          "--batch_size", "64", "--snapshot_every", "3", "--outfile", str(tmp_path / "c.h5")],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "device_search: candidates drawn and refitted on the device" in out.stdout
    assert os.listdir(str(tmp_path / "c.h5.dir"))
