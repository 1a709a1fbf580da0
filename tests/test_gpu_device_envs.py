"""Device-resident rollouts (rollout.cu, core.do_rollouts_device, run_pg.py --device_envs) on the GPU, replayed
against the oracle: the Philox resets and draws of oracle/rollout.py, the dynamics of envs.py stepped from the
recorded states, the lockstep ZFilter over float64 RunningStat, and the policy forward of the library."""
import copy
import os
import subprocess
import sys
from itertools import count

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _policy(kind, hid_sizes=(64, 64), activation="tanh", scale=None, seed=0):
    from modular_rl_b200 import core
    probtype = core.Categorical(2) if kind == "cartpole" else core.DiagGauss(1)
    np.random.seed(seed)
    pol = core.StochPolicyMLP(4 if kind == "cartpole" else 3, list(hid_sizes), probtype, activation)
    if scale is not None:                 # weights large enough that the probabilities move away from 1/2
        th = pol.get_flat()
        pol.set_from_flat(np.random.default_rng(seed).standard_normal(th.size).astype(np.float32) * scale)
    return pol


def _env(kind):
    from modular_rl_b200 import envs
    return envs.CartPoleEnv() if kind == "cartpole" else envs.PendulumEnv()


def _raw_obs(kind, states):
    if kind == "cartpole":
        return states.copy()
    return np.stack([np.cos(states[:, 0]), np.sin(states[:, 0]), states[:, 1]], axis=1)


def _split(out):
    off = np.concatenate([[0], np.cumsum(out["lengths"], dtype=np.int64)])
    return off, [slice(off[i], off[i + 1]) for i in range(len(out["lengths"]))]


OB_STATE = (10.0, np.array([0.01, -0.02, 0.03, 0.5]), np.array([0.5, 2.0, 0.3, 4.0]))
REW_STATE = (7.0, np.array([0.9]), np.array([3.0]))


def _run(kind, n_envs, limit, seed, pol, stochastic=True, filters=True, want_states=True):
    from modular_rl_b200.device import DeviceRollouts
    ro = DeviceRollouts("CartPole-v0" if kind == "cartpole" else "Pendulum-v0", n_envs, limit)
    d = ro.ob_dim
    ob = ((OB_STATE[0], OB_STATE[1][:d], OB_STATE[2][:d]), True, True, 5.0) if filters else None
    rew = (REW_STATE, False, True, 10.0) if filters else None
    return ro.run(pol.net, seed, stochastic, ob, rew, want_states=want_states)


def _check_probs(kind, out, pol):
    """Prob rows against a float64 forward of the same float32 parameters on the float32 observations, elementwise,
    with a tolerance scaled by the magnitude of the terms that the last layer sums (a mean near zero is a sum that
    cancels, and only its absolute error is defined to FP32 rounding); and against the library's own forward
    (policy._act_prob) within 1e-5 relative in norm."""
    from conftest import relerr
    from oracle import policy_math as pm
    spec = pm.NetSpec(tuple(pol.dims), pm.CAT if kind == "cartpole" else pm.GAUSS, pol.activation)
    theta = pol.get_flat()
    x = out["observation"].astype(np.float32)
    hs, z = pm.forward(theta, spec, x)
    ref = pm.head_prob(theta, spec, z)
    Ws, bs, _ = pm.split_params(np.asarray(theta, np.float64), spec)
    scale = (np.abs(hs[-1]) @ np.abs(Ws[-1]) + np.abs(bs[-1])).max(axis=1, keepdims=True)
    err = np.abs(out["prob"] - ref)
    assert np.all(err <= 1e-5 * (np.abs(ref) + scale)), float((err / (np.abs(ref) + scale)).max())
    assert relerr(out["prob"], pol._act_prob(out["observation"])) < 1e-5


def _check_round(kind, out, seed, pol, limit, envs_checked=None, stochastic=True, filters=True):
    """Everything the oracle can say about one round (see the module docstring)."""
    from oracle import rollout as orc
    env = _env(kind)
    lengths, term = out["lengths"], out["terminated"]
    off, sl = _split(out)
    N = len(lengths)
    assert off[-1] == len(out["reward"]) == len(out["observation"]) == len(out["prob"]) == len(out["action"])
    assert np.all((lengths >= 1) & (lengths <= limit))
    assert np.all((term == 1) | (lengths == limit))
    if kind == "pendulum":
        assert not term.any() and np.all(lengths == limit)
    states = out["states"]
    idx = np.arange(N) if envs_checked is None else np.asarray(envs_checked)
    # resets
    np.testing.assert_allclose(states[off[idx]], orc.reset_states(kind, seed, idx), rtol=0, atol=1e-15)
    # dynamics: envs.py from each recorded (state, action)
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
    # filters: the lockstep ZFilter over every environment of the round
    raw = [_raw_obs(kind, states[sl[i]]) for i in range(N)]
    if filters:
        d = raw[0].shape[1]
        want, rs, pushed = orc.lockstep_zfilter(raw, lengths, (OB_STATE[0], OB_STATE[1][:d], OB_STATE[2][:d]))
        for i in range(N):
            np.testing.assert_allclose(out["observation"][sl[i]], want[i], rtol=0, atol=1e-10)
        for got, ref in ((out["ob_state"], rs), (out["ob_pushed"], pushed)):
            assert got[0] == ref.n
            np.testing.assert_allclose(got[1], ref.M, rtol=1e-10, atol=1e-12)
            np.testing.assert_allclose(got[2], ref.S, rtol=1e-10, atol=1e-12)
        rrs, rpushed = orc.lockstep_rewards([out["reward"][sl[i]] for i in range(N)], lengths, REW_STATE)
        for got, ref in ((out["rew_state"], rrs), (out["rew_pushed"], rpushed)):
            assert got[0] == ref.n
            np.testing.assert_allclose(got[1], ref.M, rtol=1e-10)
            np.testing.assert_allclose(got[2], ref.S, rtol=1e-10)
    else:
        for i in range(N):
            np.testing.assert_array_equal(out["observation"][sl[i]], raw[i]) if kind == "cartpole" else \
                np.testing.assert_allclose(out["observation"][sl[i]], raw[i], rtol=0, atol=1e-15)
    _check_probs(kind, out, pol)
    # actions
    for i in idx:
        t = np.arange(lengths[i])
        P, A = out["prob"][sl[i]], out["action"][sl[i]]
        if not stochastic:
            want = P.argmax(axis=1) if kind == "cartpole" else P[:, :1]
            np.testing.assert_array_equal(A, want)
        elif kind == "cartpole":
            u = orc.action_uniform(seed, i, t)
            assert [orc.categorical_action(P[k], u[k]) for k in range(len(t))] == list(A)
        else:
            want = orc.gauss_action(P[:, 0], P[:, 1], orc.action_normal(seed, i, t).astype(np.float32))
            np.testing.assert_allclose(A[:, 0], want, rtol=0, atol=1e-5)


@pytest.mark.parametrize("kind,limit", [("cartpole", 200), ("pendulum", 50)])
def test_round_replays_against_oracle(kind, limit):
    pol = _policy(kind, scale=0.5)
    out = _run(kind, 64, limit, 1234, pol)
    _check_round(kind, out, 1234, pol, limit)


@pytest.mark.parametrize("kind", ["cartpole", "pendulum"])
def test_deterministic_actions_are_maxprob(kind):
    pol = _policy(kind, scale=0.5)
    out = _run(kind, 16, 30, 5, pol, stochastic=False)
    _check_round(kind, out, 5, pol, 30, stochastic=False)


@pytest.mark.parametrize("hid,act", [((64, 64), "tanh"), ((32,), "relu"), ((256,), "sigmoid"),
                                     ((32, 32, 32, 32, 32), "tanh")])
def test_net_shapes(hid, act):
    """Every activation, the widest hidden layer (256) and the deepest net (6 layers) that mrl_net_create accepts for
    CartPole's 4 inputs and 2 outputs; wider hidden stacks such as [256, 128, 64] need more shared memory than the
    update kernels have and are rejected there, before any rollout."""
    pol = _policy("cartpole", hid, act, scale=0.3)
    out = _run("cartpole", 40, 60, 9, pol, filters=False)
    _check_round("cartpole", out, 9, pol, 60, envs_checked=[0, 17, 39], filters=False)


def test_n_envs_range_and_limit():
    from modular_rl_b200.device import DeviceRollouts
    mx = DeviceRollouts.max_envs()
    assert mx >= 4096
    pol = _policy("cartpole", scale=0.5)
    for n in (1, 33, 1000, mx):
        out = _run("cartpole", n, 40, 77 + n, pol)
        sample = sorted({0, n // 3, n // 2, n - 1})
        _check_round("cartpole", out, 77 + n, pol, 40, envs_checked=sample)
    with pytest.raises(RuntimeError, match="1..%d environments per round" % mx):
        DeviceRollouts("CartPole-v0", mx + 1, 40)


def test_wrong_policy_is_rejected():
    pol = _policy("pendulum")
    with pytest.raises(RuntimeError, match="CartPole observations have 4 entries, the policy takes 3"):
        _run("cartpole", 4, 10, 0, pol)
    from modular_rl_b200 import core
    np.random.seed(0)
    gauss4 = core.StochPolicyMLP(4, [8], core.DiagGauss(1))
    with pytest.raises(RuntimeError, match="CartPole needs a Categorical head with 2 outputs"):
        _run("cartpole", 4, 10, 0, gauss4)


def test_same_seed_same_bits():
    pol = _policy("pendulum", scale=0.5)
    a = _run("pendulum", 100, 40, 42, pol)
    b = _run("pendulum", 100, 40, 42, pol)
    c = _run("pendulum", 100, 40, 43, pol)
    for k in ("observation", "action", "prob", "reward", "states"):
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["states"], c["states"]) and not np.array_equal(a["action"], c["action"])
    for k in ("ob_state", "rew_state"):
        assert all(np.array_equal(x, y) for x, y in zip(a[k], b[k]))


def test_do_rollouts_device_rounds_and_wire_format(monkeypatch):
    from modular_rl_b200 import agentzoo, core, envs
    env = envs.CartPoleEnv()
    np.random.seed(0)
    agent = agentzoo.TrpoAgent(env.observation_space, env.action_space, dict(hid_sizes=[16], timestep_limit=40))
    seeds = count()
    n0 = agent.obfilter.rs.n
    paths = core.do_rollouts_device(env, agent, 40, 150, seeds, 8)
    rounds = len(paths) // 8
    assert len(paths) % 8 == 0 and next(seeds) == rounds          # one seed per round
    lens = [core.pathlength(p) for p in paths]
    assert sum(lens) > 150 and sum(lens[:-8]) <= 150                # strict stop after the round that crosses it
    assert agent.obfilter.rs.n == n0 + sum(lens) and agent.rewfilter.rs.n == sum(lens)
    host = core.do_rollouts_vectorized(copy.deepcopy(env), agent, 40, 10, count(), 2)
    assert list(paths[0]) == list(host[0])
    for k in host[0]:
        assert type(paths[0][k]) is type(host[0][k]), k
        if isinstance(host[0][k], np.ndarray):
            assert paths[0][k].dtype == host[0][k].dtype and paths[0][k].ndim == host[0][k].ndim, k
    # through get_paths, as run_pg.py --device_envs sets it
    monkeypatch.setattr(core, "DEVICE_ENVS", 8)
    got = core.get_paths(env, agent, dict(parallel=0, timesteps_per_batch=100, timestep_limit=40), count())
    assert sum(core.pathlength(p) for p in got) > 100
    core.compute_advantage(agent.baseline, got, 0.99, 0.97)
    # a Pendulum round writes the DiagGauss wire format
    penv = envs.PendulumEnv()
    pagent = agentzoo.TrpoAgent(penv.observation_space, penv.action_space, dict(hid_sizes=[16], timestep_limit=20))
    pp = core.do_rollouts_device(penv, pagent, 20, 30, count(), 2)
    hp = core.do_rollouts_vectorized(copy.deepcopy(penv), pagent, 20, 10, count(), 2)
    for k in ("observation", "action", "prob", "reward"):
        assert pp[0][k].dtype == hp[0][k].dtype and pp[0][k].shape == hp[0][k].shape, k


def _run_pg(args, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "run_pg.py")] + args, capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout


def test_run_pg_cartpole_learns_with_device_envs(tmp_path):
    """test_run_pg_cartpole_learns with the rollouts on the device."""
    stdout = _run_pg(["--env", "CartPole-v0", "--agent", "modular_rl.agentzoo.TrpoAgent", "--n_iter", "12",
                      "--timesteps_per_batch", "2000", "--seed", "0", "--cg_damping", "0.1", "--lam", "0.97",
                      "--device_envs", "64", "--outfile", str(tmp_path / "a.h5")])
    rews = [float(ln.split()[-1]) for ln in stdout.splitlines() if ln.startswith("EpRewMean")]
    assert len(rews) == 12
    assert max(rews[-3:]) > 2.0 * rews[0], rews
    kls = [float(ln.split()[-1]) for ln in stdout.splitlines() if ln.startswith("pol_kl_after")]
    assert all(0 < k < 0.03 for k in kls), kls


def test_coverage_smoke_pendulum_with_device_envs(tmp_path):
    stdout = _run_pg(["--snapshot_every=20", "--n_iter=1", "--cg_damping=0.1", "--timesteps_per_batch=5", "--lam=0.97",
                      "--agent=modular_rl.agentzoo.TrpoAgent", "--max_kl=0.01", "--env=Pendulum", "--gamma=0.98",
                      "--hid_sizes=10,5", "--device_envs=4", "--outfile", str(tmp_path / "b.h5")], timeout=600)
    assert "pol_surr_after" in stdout and "vf_EV_after" in stdout


@pytest.mark.parametrize("ranks", [2, 1])
def test_dp_device_envs(ranks):
    import test_gpu_data_parallel as dp
    dp._need_gpus(ranks)
    rc, out = dp._torchrun([os.path.join(ROOT, "tests", "dp_device_envs_check.py")], ranks=ranks)
    assert rc == 0 and "DP_DEVICE_ENVS_CHECK_OK" in out, out[-4000:]
