"""Population rounds of the device rollouts (rollout.cu POP mode, mrl_rollout_run_population,
DeviceRollouts.run_population, cem.evaluate_population_device, run_cem.py --device_envs) on the GPU: each environment
acts with its own parameter vector.  Rounds are replayed against the oracle (oracle/rollout.py resets and lockstep
ZFilter, envs.py dynamics, a float64 forward of each member's own theta), and scores are compared with the host
population path bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import test_gpu_device_envs as de

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

ENV_ID = {"cartpole": "CartPole-v0", "pendulum": "Pendulum-v0"}


def _dims(kind, hid=(64, 64)):
    return [4 if kind == "cartpole" else 3] + list(hid) + [2 if kind == "cartpole" else 1]


def _n_dense(dims):
    return sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(dims) - 1))


def _thetas(dims, M, scale=0.5, seed=0):
    return (np.random.default_rng(seed).standard_normal((M, _n_dense(dims))) * scale).astype(np.float32)


def _filters(kind, on=True):
    if not on:
        return None, None
    d = 4 if kind == "cartpole" else 3
    return ((de.OB_STATE[0], de.OB_STATE[1][:d], de.OB_STATE[2][:d]), True, True, 5.0), (de.REW_STATE, False, True, 10.0)


def _ro(kind, n_envs, limit):
    from modular_rl_b200.device import DeviceRollouts
    return DeviceRollouts(ENV_ID[kind], n_envs, limit)


def _run(kind, n_envs, limit, seed, dims, thetas, act="tanh", filters=True, want_rows=True, want_states=True, ro=None):
    ro = ro or _ro(kind, n_envs, limit)
    ob, rew = _filters(kind, filters)
    return ro.run_population(dims, act, thetas, seed, ob, rew, want_rows=want_rows, want_states=want_states)


def _check_population_round(kind, out, seed, dims, thetas, limit, act="tanh", filters=True, members=None):
    """Resets, dynamics, filters, each row's raw outputs against its own member's float64 forward, actions, scores."""
    from oracle import policy_math as pm
    from oracle import rollout as orc
    env = de._env(kind)
    lengths, term = out["lengths"], out["terminated"]
    off, sl = de._split(out)
    N = len(lengths)
    assert N == thetas.shape[0]
    assert off[-1] == len(out["reward"]) == len(out["observation"]) == len(out["prob"]) == len(out["action"])
    assert np.all((lengths >= 1) & (lengths <= limit))
    assert np.all((term == 1) | (lengths == limit))
    states = out["states"]
    idx = np.arange(N) if members is None else np.asarray(members)
    np.testing.assert_allclose(states[off[idx]], orc.reset_states(kind, seed, idx), rtol=0, atol=1e-15)
    for i in idx:
        S, A, R = states[sl[i]], out["action"][sl[i]], out["reward"][sl[i]]
        for t in range(lengths[i]):
            env.state = S[t].copy()
            _, r, done, _ = env.step(A[t] if kind == "cartpole" else A[t].astype(np.float64))
            assert abs(r - R[t]) <= 1e-12, (i, t, r, R[t])
            if t + 1 < lengths[i]:
                np.testing.assert_allclose(env.state, S[t + 1], rtol=0, atol=1e-12)
                assert not done, (i, t)
            else:
                assert done == bool(term[i]), (i, t)
    raw = [de._raw_obs(kind, states[sl[i]]) for i in range(N)]
    if filters:
        d = raw[0].shape[1]
        want, rs, pushed = orc.lockstep_zfilter(raw, lengths, (de.OB_STATE[0], de.OB_STATE[1][:d], de.OB_STATE[2][:d]))
        for i in range(N):
            np.testing.assert_allclose(out["observation"][sl[i]], want[i], rtol=0, atol=1e-10)
        for got, ref in ((out["ob_state"], rs), (out["ob_pushed"], pushed)):
            assert got[0] == ref.n
            np.testing.assert_allclose(got[1], ref.M, rtol=1e-10, atol=1e-12)
            np.testing.assert_allclose(got[2], ref.S, rtol=1e-10, atol=1e-12)
        rrs, rpushed = orc.lockstep_rewards([out["reward"][sl[i]] for i in range(N)], lengths, de.REW_STATE)
        for got, ref in ((out["rew_state"], rrs), (out["rew_pushed"], rpushed)):
            assert got[0] == ref.n
            np.testing.assert_allclose(got[1], ref.M, rtol=1e-10)
            np.testing.assert_allclose(got[2], ref.S, rtol=1e-10)
    else:
        for i in idx:
            np.testing.assert_allclose(out["observation"][sl[i]], raw[i], rtol=0, atol=1e-15)
    # raw outputs: a float64 forward of member i's own theta on the float32 observations (bound as _check_probs)
    spec = pm.NetSpec(tuple(dims), pm.CAT, act)
    for i in idx:
        x = out["observation"][sl[i]].astype(np.float32)
        hs, z = pm.forward(thetas[i, :_n_dense(dims)], spec, x)
        Ws, bs, _ = pm.split_params(np.asarray(thetas[i, :_n_dense(dims)], np.float64), spec)
        scale = (np.abs(hs[-1]) @ np.abs(Ws[-1]) + np.abs(bs[-1])).max(axis=1, keepdims=True)
        P, A = out["prob"][sl[i]], out["action"][sl[i]]
        got = P if kind == "cartpole" else P[:, :1]
        err = np.abs(got - z)
        assert np.all(err <= 1e-5 * (np.abs(z) + scale)), (i, float((err / (np.abs(z) + scale)).max()))
        if kind == "cartpole":
            np.testing.assert_array_equal(A, P.argmax(axis=1))
        else:
            np.testing.assert_array_equal(A[:, 0], P[:, 0])
            assert np.all(P[:, 1] == 1.0)
    # scores: the step-order float64 sum of each member's raw rewards
    for i in range(N):
        total = 0.0
        for r in out["reward"][sl[i]]:
            total += r
        assert out["returns"][i] == total, (i, out["returns"][i], total)


@pytest.mark.parametrize("kind,limit", [("cartpole", 200), ("pendulum", 50)])
def test_population_round_replays_against_oracle(kind, limit):
    dims = _dims(kind)
    th = _thetas(dims, 64, 0.5, seed=3)
    out = _run(kind, 64, limit, 1234, dims, th)
    _check_population_round(kind, out, 1234, dims, th, limit)
    assert len(set(out["lengths"].tolist())) > 1 or kind == "pendulum"   # distinct thetas, distinct episodes


def test_same_bits_as_host_population_path(monkeypatch):
    """cem.evaluate_population (one population forward per step on the host loop) with each environment reset to the
    device's start state gives exactly the device scores."""
    from modular_rl_b200 import agentzoo, cem, envs
    from oracle import rollout as orc
    env = envs.CartPoleEnv()
    np.random.seed(0)
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[64, 64], filter=0))
    dims = agent.policy.dims
    th = _thetas(dims, 48, 0.5, seed=11)
    seed = 2024
    dev = cem.evaluate_population_device(env, agent, th, 200, seed)
    starts = orc.reset_states("cartpole", seed, np.arange(48))
    made = [0]

    def reset(self):
        self.state = starts[made[0]].copy()
        made[0] += 1
        return np.array(self.state)
    monkeypatch.setattr(envs.CartPoleEnv, "reset", reset)
    host = cem.evaluate_population(env, agent, th, 200)
    assert made[0] == 48
    assert np.array_equal(host, dev), (host, dev)
    assert len(set(dev.tolist())) > 1


def test_agrees_with_shared_theta_round():
    """Every member with the Dense part of one DeterministicPolicy: the same round as mrl_rollout_run, maxprob."""
    from modular_rl_b200 import agentzoo, core
    np.random.seed(4)
    pol = agentzoo.DeterministicPolicy(3, [64, 64], core.DiagGauss(1))
    pol.set_from_flat(np.random.default_rng(4).standard_normal(pol.get_flat().size).astype(np.float32) * 0.5)
    th = np.tile(pol.get_flat()[None, :].astype(np.float32), (40, 1))
    ro = _ro("pendulum", 40, 60)
    ob, rew = _filters("pendulum")
    a = ro.run(pol.net, 99, False, ob, rew, want_states=True)
    b = ro.run_population(pol.dims, "tanh", th, 99, ob, rew, want_rows=True, want_states=True)
    for k in ("observation", "action", "reward", "lengths", "states", "prob"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("ob_state", "ob_pushed", "rew_state", "rew_pushed"):
        assert all(np.array_equal(x, y) for x, y in zip(a[k], b[k])), k


@pytest.mark.parametrize("hid,act", [((32,), "relu"), ((256,), "sigmoid"), ((32, 32, 32, 32, 32), "tanh")])
def test_net_shapes(hid, act):
    dims = _dims("cartpole", hid)
    th = _thetas(dims, 40, 0.3, seed=len(hid))
    out = _run("cartpole", 40, 60, 9, dims, th, act=act, filters=False)
    _check_population_round("cartpole", out, 9, dims, th, 60, act=act, filters=False)


def test_padding_members_and_device_thetas():
    import torch
    dims = _dims("pendulum", (32, 32))
    P = _n_dense(dims)
    ro = _ro("pendulum", 100, 30)
    th = _thetas(dims, 100, 0.5, seed=5)
    ref = _run("pendulum", 100, 30, 7, dims, th, ro=ro)
    padded = np.full((100, P + 13), np.nan, np.float32)
    padded[:, :P] = th
    got = _run("pendulum", 100, 30, 7, dims, padded, ro=ro)
    dev = _run("pendulum", 100, 30, 7, dims, torch.from_numpy(padded).cuda(), ro=ro)
    for k in ("returns", "observation", "action", "prob", "reward", "states", "lengths"):
        assert np.array_equal(ref[k], got[k]) and np.array_equal(ref[k], dev[k]), k
    # fewer members than the handle holds: member m of the small round is member m of the large one
    few = _run("pendulum", 100, 30, 7, dims, th[:33], ro=ro, filters=False)
    full = _run("pendulum", 100, 30, 7, dims, th, ro=ro, filters=False)
    assert few["lengths"].shape == (33,) and few["returns"].shape == (33,)
    assert np.array_equal(few["returns"], full["returns"][:33])
    _check_population_round("pendulum", few, 7, dims, th[:33], 30, filters=False)


def test_member_counts():
    from modular_rl_b200.device import DeviceRollouts
    mx = DeviceRollouts.max_envs()
    dims = _dims("cartpole")
    for n in (1, 33, mx):
        th = _thetas(dims, n, 0.5, seed=n)
        out = _run("cartpole", n, 40, 77 + n, dims, th)
        _check_population_round("cartpole", out, 77 + n, dims, th, 40, members=sorted({0, n // 3, n // 2, n - 1}))


def test_same_seed_same_bits_and_rows_optional():
    dims = _dims("cartpole")
    th = _thetas(dims, 200, 0.5, seed=8)
    ro = _ro("cartpole", 200, 200)
    a = _run("cartpole", 200, 200, 42, dims, th, ro=ro)
    b = _run("cartpole", 200, 200, 42, dims, th, ro=ro)
    c = _run("cartpole", 200, 200, 43, dims, th, ro=ro)
    for k in ("returns", "observation", "action", "prob", "reward", "states", "lengths"):
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["states"][:1], c["states"][:1]) and not np.array_equal(a["returns"], c["returns"])
    # without rows: the same scores, lengths and filter states, and no row arrays
    n = _run("cartpole", 200, 200, 42, dims, th, ro=ro, want_rows=False, want_states=False)
    assert "observation" not in n
    for k in ("returns", "lengths", "terminated"):
        assert np.array_equal(a[k], n[k]), k
    for k in ("ob_state", "rew_state"):
        assert all(np.array_equal(x, y) for x, y in zip(a[k], n[k])), k


def _raw_call(ro, dims, th, n_members=None, act=0, ld=None, want_rows=0, want_states=0, loc=None):
    from modular_rl_b200 import _lib as L
    th = np.ascontiguousarray(th, np.float32)
    arr = (C.c_int * len(dims))(*dims)
    ret = np.zeros(max(th.shape[0], 1))
    n = C.c_longlong()
    return L.check(L.lib().mrl_rollout_run_population(
        ro._h, len(dims) - 1, arr, act, L.ptr(th), th.shape[1] if ld is None else ld, L.HOST if loc is None else loc,
        th.shape[0] if n_members is None else n_members, 1, None, None, None, None, None, None, L.ptr(ret),
        want_rows, want_states, C.byref(n), None))


def test_rejections():
    from modular_rl_b200 import _lib as L
    ro = _ro("cartpole", 8, 10)
    dims = _dims("cartpole", (16,))
    th = _thetas(dims, 8)
    with pytest.raises(RuntimeError, match="CartPole observations have 4 entries, dims\\[0\\] = 3"):
        _raw_call(ro, [3, 16, 2], th)
    with pytest.raises(RuntimeError, match="CartPole actions take 2 outputs, dims\\[2\\] = 1"):
        _raw_call(ro, [4, 16, 1], th)
    with pytest.raises(RuntimeError, match="n_layers = 7; the rollout kernel runs 1..6 layers"):
        _raw_call(ro, [4] + [8] * 6 + [2], th)
    with pytest.raises(RuntimeError, match="dims\\[1\\] = 257; widths must be in 1..256"):
        _raw_call(ro, [4, 257, 2], np.zeros((8, 2000), np.float32))
    with pytest.raises(RuntimeError, match="unknown activation 3"):
        _raw_call(ro, dims, th, act=3)
    with pytest.raises(RuntimeError, match="ld_theta = 100 is smaller than the 114 Dense parameters"):
        _raw_call(ro, dims, th, ld=100)
    with pytest.raises(RuntimeError, match="n_members = 9; the handle runs 1..8 environments"):
        _raw_call(ro, dims, np.zeros((9, th.shape[1]), np.float32))
    with pytest.raises(RuntimeError, match="n_members = 0"):
        _raw_call(ro, dims, th, n_members=0)
    with pytest.raises(RuntimeError, match="theta_loc = 2 \\(MRL_HOST or MRL_DEVICE\\)"):
        _raw_call(ro, dims, th, loc=2)
    with pytest.raises(RuntimeError, match="theta_loc = MRL_DEVICE but thetas is not device memory of device"):
        _raw_call(ro, dims, th, loc=L.DEVICE)          # host memory passed as device memory
    # rows after a round without rows; lengths stay readable
    _raw_call(ro, dims, th)
    obs = np.empty((80, 4))
    with pytest.raises(RuntimeError, match="did not record rows"):
        L.check(L.lib().mrl_rollout_read(ro._h, None, None, L.ptr(obs), None, None, None, None))
    lengths = np.empty(8, np.int32)
    L.check(L.lib().mrl_rollout_read(ro._h, L.ptr(lengths), None, None, None, None, None, None))
    assert np.all((lengths >= 1) & (lengths <= 10))


def _count_population_launches(monkeypatch):
    from modular_rl_b200 import _lib as L, cem
    calls = []
    orig = cem.evaluate_population_device

    def counted(*a, **k):
        n0 = L.lib().mrl_launch_count()
        out = orig(*a, **k)
        calls.append(L.lib().mrl_launch_count() - n0)
        return out
    monkeypatch.setattr(cem, "evaluate_population_device", counted)
    return calls


def test_run_cem_algorithm_on_device(monkeypatch):
    from modular_rl_b200 import agentzoo, cem, device, envs
    monkeypatch.setattr(cem, "DEVICE_ENVS", True)
    launches = _count_population_launches(monkeypatch)
    lengths = []
    orig_run = device.DeviceRollouts.run_population

    def run_population(self, *a, **k):
        out = orig_run(self, *a, **k)
        lengths.append(int(out["lengths"].sum()))
        return out
    monkeypatch.setattr(device.DeviceRollouts, "run_population", run_population)
    env = envs.CartPoleEnv()
    np.random.seed(0)
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[64, 64]))
    n0 = agent.obfilter.rs.n
    infos = []
    cem.run_cem_algorithm(env, agent, dict(batch_size=64, n_iter=6, timestep_limit=200, seed=0), callback=infos.append)
    assert len(infos) == 6 and launches == [1] * 6
    assert agent.obfilter.rs.n == n0 + sum(lengths) and agent.rewfilter.rs.n == sum(lengths)
    assert max(info["ymean"] for info in infos[1:]) > infos[0]["ymean"]
    np.testing.assert_array_equal(agent.get_flat(), infos[-1]["th"].astype(np.float32))
    # Pendulum
    penv = envs.PendulumEnv()
    pagent = agentzoo.DeterministicAgent(penv.observation_space, penv.action_space, dict(hid_sizes=[16]))
    pinfos = []
    cem.run_cem_algorithm(penv, pagent, dict(batch_size=32, n_iter=2, timestep_limit=50), callback=pinfos.append)
    assert len(pinfos) == 2 and all(np.all(np.isfinite(i["ys"])) for i in pinfos)


def _run_cem(args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "run_cem.py")] + args, capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_run_cem_cli_device_envs(tmp_path):
    out = _run_cem(["--env", "CartPole-v0", "--agent", "modular_rl.agentzoo.DeterministicAgent", "--device_envs",
                    "--n_iter", "2", "--batch_size", "40", "--snapshot_every", "2", "--outfile", str(tmp_path / "c.h5")])
    assert out.returncode == 0, out.stderr[-2000:]
    assert "device_envs: one device rollout round per generation" in out.stdout
    assert os.listdir(str(tmp_path / "c.h5.dir"))
    bad = _run_cem(["--env", "Hopper-v1", "--agent", "modular_rl.agentzoo.DeterministicAgent", "--device_envs",
                    "--outfile", str(tmp_path / "d.h5")])
    assert bad.returncode == 2 and "CartPole-v0" in bad.stderr and "Pendulum-v0" in bad.stderr
    assert not os.path.exists(str(tmp_path / "d.h5.dir"))
