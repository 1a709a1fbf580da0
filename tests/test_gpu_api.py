"""The reference-facing Python API (agentzoo / updaters / compute_advantage / NnVf / ZFilter /
run_pg flow) on the GPU, checked against the oracle on the same paths.  These read like the tests
the reference would have for TrpoUpdater / compute_advantage: build `paths`, call the operator,
compare the returned dict / the in-place path entries."""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from conftest import relerr  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _make_paths(rng, n_paths, d0, policy, tmax=60):
    paths = []
    for i in range(n_paths):
        T = int(rng.integers(1, tmax + 1))
        ob = np.clip(rng.standard_normal((T, d0)), -5, 5)          # float64, as the ZFilter emits
        prob = policy._act_prob(ob)
        np.random.seed(100 + i)
        act = policy.probtype.sample(prob)
        paths.append(dict(observation=ob, action=act, prob=prob, reward=rng.standard_normal(T),
                          terminated=bool(rng.random() < 0.7)))
    return paths


def _oracle_spec(policy):
    from oracle import policy_math as pm
    from modular_rl_b200.core import DiagGauss
    head = pm.GAUSS if isinstance(policy.probtype, DiagGauss) else pm.CAT
    return pm.NetSpec(tuple(policy.dims), head)


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_compute_advantage_fit_and_trpo_updater(kind):
    from modular_rl_b200 import agentzoo, core, spaces
    from oracle import advantage as oadv, natgrad, policy_math as pm, valuefn
    np.random.seed(0)
    rng = np.random.default_rng(0)
    ob_space = spaces.Box(-np.ones(6), np.ones(6))
    ac_space = spaces.Box(-np.ones(2), np.ones(2)) if kind == "box" else spaces.Discrete(3)
    cfg = dict(hid_sizes=[16, 8], timestep_limit=60, cg_damping=0.1, max_kl=0.01, gamma=0.98, lam=0.95)
    agent = agentzoo.TrpoAgent(ob_space, ac_space, cfg)
    assert {o[0] for o in agent.options} >= {"cg_damping", "max_kl", "hid_sizes", "gamma", "lam", "filter"}
    paths = _make_paths(rng, 40, 6, agent.policy)
    opaths = copy.deepcopy(paths)

    # ---- compute_advantage (core.py:63-105), in place
    vf_theta = agent.baseline.reg.net.get_params()
    vspec = pm.NetSpec(tuple(agent.baseline.reg.net.dims), pm.VALUE)
    opredict = lambda p: valuefn.vf_forward(vf_theta, vspec, valuefn.preproc(p["observation"], 60),
                                            np.float64)[:, 0].astype(np.float32)
    core.compute_advantage(agent.baseline, paths, 0.98, 0.95)
    oadv.compute_advantage(opredict, opaths, 0.98, 0.95)
    for p, o in zip(paths, opaths):
        assert p["return"].dtype == np.float64 and p["advantage"].shape == o["advantage"].shape
        assert np.allclose(p["return"], o["return"], rtol=1e-12, atol=1e-12)
        assert np.allclose(p["baseline"], o["baseline"], rtol=1e-5, atol=1e-6)
    assert relerr(np.concatenate([p["advantage"] for p in paths]),
                  np.concatenate([o["advantage"] for o in opaths])) < 1e-5

    # ---- baseline.fit (core.py:652-657 -> 619-637 -> 674-697)
    for p, o in zip(paths, opaths):
        o["advantage"], o["return"], o["baseline"] = p["advantage"], p["return"], p["baseline"]
    vstats = agent.baseline.fit(paths)
    x = np.concatenate([valuefn.preproc(o["observation"], 60) for o in opaths])
    y = np.concatenate([o["return"] for o in opaths]).reshape(-1, 1)
    ostats, oth, _ = valuefn.regression_fit(vf_theta, vspec, x, y, mixfrac=0.1, maxiter=25)
    assert list(vstats)[:6] == ["loss_before", "loss_after", "mse_before", "mse_after", "l2_before", "l2_after"]
    for k in ("loss_before", "mse_before", "l2_before", "TargStdev", "PredStdevBefore", "EV_before"):
        assert np.isclose(vstats[k], ostats[k], rtol=1e-4, atol=1e-6), (k, vstats[k], ostats[k])
    assert vstats["loss_after"] < vstats["loss_before"]
    assert np.isclose(vstats["loss_after"], ostats["loss_after"], rtol=2e-2)     # L-BFGS path on float32 vs float64

    # ---- updater(paths) (trpo.py:72-140)
    theta = agent.policy.get_flat()
    spec = _oracle_spec(agent.policy)
    cat = lambda k: np.concatenate([o[k] for o in opaths])
    out = agent.updater(paths)
    ostats, oinfo = natgrad.trpo_update(theta, spec, cat("observation"), cat("action"), cat("advantage"),
                                        cat("prob"), 0.1, 0.01)
    assert list(out) == ["surr_before", "surr_after", "kl_before", "kl_after", "ent_before", "ent_after"]
    for k in out:
        assert np.isclose(out[k], ostats[k], rtol=1e-4, atol=1e-6), (k, out[k], ostats[k])
    assert relerr(agent.policy.get_flat(), oinfo["theta_new"]) < 5e-5   # ~1200 timesteps: CG amplifies f32 rounding of the Fvp
    assert agent.updater.last_info["success"] == int(oinfo["success"])


def test_ppo_lbfgs_updater_matches_oracle():
    from modular_rl_b200 import agentzoo, spaces
    from oracle import ppo_penalty
    np.random.seed(1)
    rng = np.random.default_rng(1)
    ob_space = spaces.Box(-np.ones(5), np.ones(5))
    agent = agentzoo.PpoLbfgsAgent(ob_space, spaces.Box(-np.ones(2), np.ones(2)),
                                   dict(hid_sizes=[12, 12], timestep_limit=50, maxiter=10))
    paths = _make_paths(rng, 30, 5, agent.policy, tmax=50)
    adv = rng.standard_normal(sum(len(p["reward"]) for p in paths))
    adv = (adv - adv.mean()) / adv.std()
    k = 0
    for p in paths:
        p["advantage"] = adv[k:k + len(p["reward"])]
        k += len(p["reward"])
    theta = agent.policy.get_flat()
    spec = _oracle_spec(agent.policy)
    cat = lambda key: np.concatenate([p[key] for p in paths])
    info = agent.updater(paths)
    oinfo, oth, oklc, _ = ppo_penalty.ppo_lbfgs_update(theta, spec, cat("observation"), cat("action"),
                                                       cat("advantage"), cat("prob"), maxiter=10)
    assert set(info) == set(oinfo)
    for key in ("surr_before", "kl_before", "ent_before"):
        assert np.isclose(info[key], oinfo[key], rtol=1e-4, atol=1e-6)
    assert info["surr_after"] < info["surr_before"]
    assert np.isclose(info["surr_after"], oinfo["surr_after"], rtol=5e-2, atol=1e-3)   # optimiser path, f32 vs f64
    assert agent.updater.kl_coeff == oklc


def test_discount_and_filter_batch(golden):
    from modular_rl_b200.filters import ZFilter
    from modular_rl_b200.misc_utils import discount
    y = discount(golden["disc_kat_x"], 0.99)                     # x.py:762 KAT through the scan kernel
    assert np.allclose(y, golden["disc_kat_y"], rtol=1e-14)
    for i in range(4):
        assert np.allclose(discount(golden[f"disc{i}_x"], float(golden[f"disc{i}_g"])), golden[f"disc{i}_y"],
                           rtol=1e-12, atol=1e-13)
    assert np.allclose(discount(golden["disc2d_x"], 0.9), golden["disc2d_y"], rtol=1e-12, atol=1e-13)
    X = golden["rs_x"]
    a, b = ZFilter((3,), clip=5), ZFilter((3,), clip=5)
    ya = np.array([a(x) for x in X])
    yb = np.concatenate([b.filter_batch(X[:13]), np.array([b(x) for x in X[13:20]]), b.filter_batch(X[20:])])
    assert np.allclose(ya, yb, rtol=1e-12, atol=1e-12) and a.rs.n == b.rs.n
    assert np.allclose(a.rs.mean, b.rs.mean, rtol=1e-13) and np.allclose(a.rs.var, b.rs.var, rtol=1e-12)


def test_run_pg_cartpole_learns(tmp_path):
    """BASELINE config 1: CartPole-v0 TrpoAgent through run_pg.py's own flags; a functional check
    (mean episode reward rises), not a throughput number."""
    cmd = [sys.executable, os.path.join(ROOT, "run_pg.py"), "--env", "CartPole-v0", "--agent",
           "modular_rl.agentzoo.TrpoAgent", "--n_iter", "12", "--timesteps_per_batch", "2000", "--seed", "0",
           "--cg_damping", "0.1", "--lam", "0.97", "--outfile", str(tmp_path / "a.h5")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    rews = [float(ln.split()[-1]) for ln in out.stdout.splitlines() if ln.startswith("EpRewMean")]
    assert len(rews) == 12
    assert max(rews[-3:]) > 2.0 * rews[0], rews
    kls = [float(ln.split()[-1]) for ln in out.stdout.splitlines() if ln.startswith("pol_kl_after")]
    assert all(0 < k < 0.03 for k in kls), kls


def test_coverage_smoke_pendulum(tmp_path):
    """coverage.sh:7 of the reference: one TRPO iteration on Pendulum with tiny settings."""
    outfile = str(tmp_path / "b.h5")
    cmd = [sys.executable, os.path.join(ROOT, "run_pg.py"), "--snapshot_every=20", "--n_iter=1", "--cg_damping=0.1",
           "--timesteps_per_batch=5", "--lam=0.97", "--agent=modular_rl.agentzoo.TrpoAgent", "--max_kl=0.01",
           "--env=Pendulum", "--gamma=0.98", "--hid_sizes=10,5", "--outfile", outfile]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "pol_surr_after" in out.stdout and "vf_EV_after" in out.stdout
    # --snapshot_every: the pickled agent lands next to the results (the reference stores the same bytes in
    # its hdf5 file, run_pg.py:141-142) and --load_snapshot resumes from it
    snap = outfile + ".dir/agent_snapshots/0001.pkl"
    assert os.path.exists(snap)
    from modular_rl_b200.misc_utils import load_agent_snapshot
    agent = load_agent_snapshot(snap)
    assert type(agent).__name__ == "TrpoAgent" and agent.policy.dims == [3, 10, 5, 1]
    # same --outfile: the snapshot is read before the previous run's results directory is cleared
    out = subprocess.run(cmd + ["--load_snapshot", outfile + ".dir"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "pol_surr_after" in out.stdout


@pytest.mark.parametrize("agent_name", ["TrpoAgent", "PpoLbfgsAgent", "PpoSgdAgent"])
def test_agent_pickle_roundtrip(agent_name):
    """Agent snapshots (EzPickle, misc_utils.py:163-189; run_pg.py:141-142): a pickled agent comes back with
    the same policy and value parameters, filter state and configuration, on fresh device handles, and its
    updater still runs."""
    import pickle
    from modular_rl_b200 import agentzoo, spaces
    from modular_rl_b200.core import compute_advantage
    rng = np.random.default_rng(5)
    np.random.seed(5)
    ob_space = spaces.Box(-np.ones(6), np.ones(6))
    ac_space = spaces.Box(-np.ones(2), np.ones(2))
    cfg = {"hid_sizes": [16, 8], "timestep_limit": 50, "max_kl": 0.02, "gamma": 0.97}
    agent = getattr(agentzoo, agent_name)(ob_space, ac_space, cfg)
    for _ in range(30):
        agent.obfilt(rng.standard_normal(6))
        agent.rewfilt(rng.standard_normal())
    agent.policy.set_params_flat(agent.policy.get_params_flat() + 0.01 * rng.standard_normal(agent.policy.net.P))
    blob = pickle.dumps(agent, -1)
    twin = pickle.loads(blob)
    assert type(twin) is type(agent) and twin.updater.stochpol is twin.policy
    np.testing.assert_array_equal(twin.policy.get_params_flat(), agent.policy.get_params_flat())
    np.testing.assert_array_equal(twin.baseline.reg.net.get_params(), agent.baseline.reg.net.get_params())
    assert twin.updater.cfg == agent.updater.cfg and twin.baseline.timestep_limit == 50
    assert twin.obfilter.rs.n == agent.obfilter.rs.n
    np.testing.assert_array_equal(twin.obfilter.rs.mean, agent.obfilter.rs.mean)
    ob = rng.standard_normal(6)
    np.testing.assert_array_equal(twin.policy.act(ob, stochastic=False)[1]["prob"],
                                  agent.policy.act(ob, stochastic=False)[1]["prob"])

    def make_paths(a):
        r = np.random.default_rng(9)
        paths = []
        for T in (20, 33, 50):
            obs = r.standard_normal((T, 6))
            prob = a.policy._act_prob(obs) if hasattr(a.policy, "_act_prob") else None
            act = prob[:, :2] + prob[:, 2:] * r.standard_normal((T, 2))
            paths.append(dict(observation=obs, action=act.astype(np.float32), prob=prob,
                              reward=r.standard_normal(T), terminated=bool(T < 50)))
        return paths

    stats = []
    for a in (agent, twin):
        paths = make_paths(a)
        compute_advantage(a.baseline, paths, gamma=0.97, lam=0.95)
        np.random.seed(11)                                    # PpoSgd shuffles minibatches with numpy's RNG
        stats.append(a.updater(paths))
    for k in stats[0]:
        assert stats[0][k] == stats[1][k], (k, stats[0][k], stats[1][k])
    np.testing.assert_array_equal(twin.policy.get_params_flat(), agent.policy.get_params_flat())


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_deterministic_agent_and_cem(kind):
    """DeterministicAgent (agentzoo.py:63-81,117-123): linear-output MLP acted on through maxprob; its flat
    vector has no logstd; run_cem_algorithm (cem.py:63-98) drives it and leaves the elite mean loaded."""
    import pickle
    from oracle import policy_math as pm
    from modular_rl_b200 import agentzoo, spaces
    from modular_rl_b200.cem import run_cem_algorithm
    from modular_rl_b200.envs import make
    rng = np.random.default_rng(3)
    np.random.seed(3)
    ob_space = spaces.Box(-np.ones(5), np.ones(5))
    ac_space = spaces.Box(-np.ones(2), np.ones(2)) if kind == "box" else spaces.Discrete(3)
    agent = agentzoo.DeterministicAgent(ob_space, ac_space, {"hid_sizes": [12, 6], "filter": 0})
    dout = 2 if kind == "box" else 3
    th = agent.get_flat()
    assert th.size == 5 * 12 + 12 + 12 * 6 + 6 + 6 * dout + dout and agent.stochastic is False
    th = (0.5 * rng.standard_normal(th.size)).astype(np.float32)
    agent.set_from_flat(th)
    np.testing.assert_array_equal(agent.get_flat(), th)
    spec = pm.NetSpec((5, 12, 6, dout), pm.CAT)      # a head without logstd: the bare Dense stack
    obs = rng.standard_normal((9, 5))
    _, z = pm.forward(th.astype(np.float64), spec, obs)
    for i in range(9):
        a, info = agent.act(obs[i])
        if kind == "box":
            assert relerr(a, z[i]) < 1e-5 and info["prob"].shape == (2,)
        else:
            assert a == int(np.argmax(z[i]))
    twin = pickle.loads(pickle.dumps(agent, -1))
    np.testing.assert_array_equal(twin.get_flat(), th)
    with pytest.raises(ValueError):
        agent.policy.act(obs[0], stochastic=True)

    env = make("Pendulum" if kind == "box" else "CartPole-v0")
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, {"hid_sizes": [8]})
    infos = []
    np.random.seed(0)
    run_cem_algorithm(env, agent, usercfg=dict(batch_size=24, n_iter=4, elite_frac=0.25, timestep_limit=100,
                                               extra_std=0.01), callback=infos.append)
    assert len(infos) == 4 and infos[0]["ys"].shape == (24,)
    np.testing.assert_allclose(agent.get_flat(), infos[-1]["th"].astype(np.float32))
    assert all(np.isfinite(i["ys"]).all() for i in infos)
    if kind == "discrete":          # CartPole: elite selection lengthens the episodes within a few iterations
        assert max(i["ymean"] for i in infos[1:]) > infos[0]["ymean"]


def test_run_cem_cli(tmp_path):
    outfile = str(tmp_path / "cem.h5")
    cmd = [sys.executable, os.path.join(ROOT, "run_cem.py"), "--env=CartPole-v0",
           "--agent=modular_rl.agentzoo.DeterministicAgent", "--n_iter=2", "--batch_size=10", "--hid_sizes=8",
           "--snapshot_every=2", "--outfile", outfile]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "Iteration 1" in out.stdout and "ymean" in out.stdout
    assert os.path.exists(outfile + ".dir/agent_snapshots/0002.pkl")


def test_multi_gpu_parity_two_ranks():
    """Sharded batch over 2 GPUs == full batch (skipped on a 1-GPU box; the CPU-side algebra is
    covered by tests/test_host_logic.py with gloo)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0 and "MULTI_GPU_CHECK_OK" in out.stdout, (out.stdout[-3000:], out.stderr[-3000:])


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_act_batch_matches_act(kind):
    """Batched rollout-side inference: act_batch(obs) rows == act(ob) row by row (same probabilities, and the
    same actions when the numpy generator is reseeded), and the ZFilter block scan == per-sample calls."""
    from modular_rl_b200 import agentzoo, filters, spaces
    rng = np.random.default_rng(1)
    ob_space = spaces.Box(-np.ones(7), np.ones(7))
    ac_space = spaces.Box(-np.ones(3), np.ones(3)) if kind == "box" else spaces.Discrete(4)
    agent = agentzoo.TrpoAgent(ob_space, ac_space, dict(hid_sizes=[16, 8], timestep_limit=50))
    obs = rng.standard_normal((37, 7))
    z1, z2 = filters.ZFilter((7,), clip=5), filters.ZFilter((7,), clip=5)
    fobs = z1.filter_batch(obs)
    assert np.allclose(fobs, np.stack([z2(o) for o in obs]), rtol=1e-10, atol=1e-12)
    pol = agent.policy
    _, info = pol.act_batch(fobs, stochastic=False)
    rows = np.stack([pol.act(o, stochastic=False)[1]["prob"] for o in fobs])
    assert np.allclose(info["prob"], rows, rtol=1e-6, atol=1e-7)
    # against the oracle's forward (float64) at the device's float32 parameters, not only CUDA against CUDA
    from oracle import policy_math as pm
    spec = _oracle_spec(pol)
    th = pol.get_flat()
    _, z = pm.forward(th, spec, fobs.astype(np.float32))
    want = pm.head_prob(th, spec, z)
    assert np.linalg.norm(info["prob"] - want) / np.linalg.norm(want) < 1e-5
    np.random.seed(5)
    a_batch, _ = pol.act_batch(fobs[:1], stochastic=True)
    np.random.seed(5)
    a_one, _ = pol.act(fobs[0], stochastic=True)
    assert np.allclose(a_batch[0], a_one)
    det, _ = pol.act_batch(fobs, stochastic=False)
    assert len(det) == 37


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_ppo_sgd_updater_matches_oracle(kind):
    """PpoSgdUpdater (ppo.py:115-228): minibatch-128 Adam on the penalised surrogate, against the oracle
    restatement with the same numpy permutation stream."""
    from modular_rl_b200 import agentzoo, spaces
    from oracle.ppo_sgd import Adam, ppo_sgd_update
    rng = np.random.default_rng(2)
    ob_space = spaces.Box(-np.ones(6), np.ones(6))
    ac_space = spaces.Box(-np.ones(2), np.ones(2)) if kind == "box" else spaces.Discrete(3)
    agent = agentzoo.PpoSgdAgent(ob_space, ac_space, dict(hid_sizes=[16, 8], timestep_limit=60, epochs=2,
                                                            stepsize=1e-3))
    paths = _make_paths(rng, 12, 6, agent.policy)
    for p in paths:
        p["advantage"] = rng.standard_normal(len(p["reward"]))
    theta = agent.policy.get_flat().astype(np.float64)
    spec = _oracle_spec(agent.policy)
    cat = lambda k: np.concatenate([p[k] for p in paths])
    np.random.seed(7)
    out = agent.updater(paths)
    np.random.seed(7)
    oinfo, oth, oklc, n_mb = ppo_sgd_update(theta, spec, cat("observation"), cat("action"), cat("advantage"),
                                            Adam(theta.size, 1e-3), epochs=2)
    assert list(out) == list(oinfo)
    for k in out:
        assert np.isclose(out[k], oinfo[k], rtol=2e-3, atol=2e-5), (k, out[k], oinfo[k])
    assert agent.updater.kl_coeff == oklc
    # Adam normalises the gradient, so float32 noise in near-zero components moves a parameter by O(stepsize)
    th = agent.policy.get_flat()
    assert np.abs(th - oth).max() < 5e-3 and relerr(th, oth) < 2e-3


# ----------------------------------------------------------------------------- SURVEY 8f rank 1 / rank 4 (round 2)
@pytest.mark.parametrize("act", ["tanh", "relu", "sigmoid"])
def test_population_forward_matches_oracle(act):
    """mrl_population_forward: every member's own theta on its own observation, one launch, against the oracle's
    float64 forward member by member."""
    from modular_rl_b200 import device
    from oracle import policy_math as pm
    rng = np.random.default_rng(3)
    dims = (9, 33, 20, 4)
    spec = pm.NetSpec(dims, pm.VALUE, act)
    P = pm.num_params(spec)
    M = 37
    ths = (0.4 * rng.standard_normal((M, P))).astype(np.float32)
    obs = rng.standard_normal((M, dims[0])).astype(np.float32)
    out = device.population_forward(dims, act, ths, obs)
    want = np.stack([pm.forward(ths[m], spec, obs[m:m + 1])[1][0] for m in range(M)])
    assert out.shape == (M, dims[-1])
    assert np.linalg.norm(out - want) / np.linalg.norm(want) < 1e-5
    # row stride larger than P (a population matrix with padding) and a single member
    pad = np.concatenate([ths, np.zeros((M, 5), np.float32)], axis=1)
    assert np.array_equal(device.population_forward(dims, act, pad, obs), out)
    assert np.array_equal(device.population_forward(dims, act, ths[:1], obs[:1]), out[:1])


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_rollouts_vectorized(kind):
    """Lockstep rollouts through act_batch / filter_batch: with one environment identical to the serial `rollout`
    (same observations after filtering, actions, probabilities and filter state); with several, every path is a valid
    rollout and the filters have seen every step once."""
    import copy
    from modular_rl_b200 import agentzoo, core, envs
    env = envs.CartPoleEnv() if kind == "discrete" else envs.PendulumEnv()
    cfg = dict(hid_sizes=[16, 8], timestep_limit=40)
    np.random.seed(0)
    a1 = agentzoo.TrpoAgent(env.observation_space, env.action_space, cfg)
    a2 = copy.deepcopy(a1)
    np.random.seed(11)
    p_serial = core.rollout(copy.deepcopy(env), a1, 40)
    np.random.seed(11)
    (p_vec,) = core.rollouts_vectorized([copy.deepcopy(env)], a2, 40)
    assert p_serial["terminated"] == p_vec["terminated"]
    for k in ("observation", "action", "reward", "prob"):
        assert np.allclose(p_serial[k], p_vec[k], rtol=1e-6, atol=1e-7), k
    assert a1.obfilter.rs.n == a2.obfilter.rs.n and np.allclose(a1.obfilter.rs.mean, a2.obfilter.rs.mean, rtol=1e-12)
    n0 = a2.obfilter.rs.n
    paths = core.rollouts_vectorized([copy.deepcopy(env) for _ in range(5)], a2, 40)
    assert len(paths) == 5
    steps = sum(core.pathlength(p) for p in paths)
    assert a2.obfilter.rs.n == n0 + steps
    for p in paths:
        T = core.pathlength(p)
        assert p["observation"].shape[0] == T == len(p["reward"]) == p["prob"].shape[0] and 1 <= T <= 40
    # the policy-gradient loop takes the lockstep rollouts when core.VEC_ENVS > 1 (run_pg.py --vec_envs): same dict keys downstream
    from itertools import count
    got = core.do_rollouts_vectorized(copy.deepcopy(env), a2, 40, 150, count(), 4)
    assert sum(core.pathlength(p) for p in got) > 150 and len(got) % 4 == 0
    core.compute_advantage(a2.baseline, got, 0.99, 0.97)
    assert all("advantage" in p for p in got)


def test_cem_population_evaluation_matches_sequential():
    """parallel=1 in run_cem_algorithm: one population-batched forward per environment step for all candidates; with
    the filters off the scores equal those of one rollout per candidate (cem.py:88-91)."""
    import copy
    from modular_rl_b200 import agentzoo, cem, core, envs
    env = envs.CartPoleEnv()
    np.random.seed(0)
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[8], filter=0))
    th0 = agent.get_flat()
    rng = np.random.default_rng(4)
    ths = th0[None, :] + 0.5 * rng.standard_normal((12, th0.size))
    np.random.seed(21)
    seq = []
    for th in ths:
        agent.set_from_flat(th)
        seq.append(core.rollout(copy.deepcopy(env), agent, 60)["reward"].sum())
    np.random.seed(21)
    pop = cem.evaluate_population(env, agent, ths, 60)
    # the environments draw their start states from numpy's global generator: sequentially one reset per rollout,
    # in lockstep all resets first - the same draws in the same order because CartPole's dynamics draw nothing
    assert np.array_equal(np.asarray(seq), pop)
    def f(th):
        raise AssertionError("cem must use f.population when it is given")
    f.population = lambda t: cem.evaluate_population(env, agent, t, 30)
    infos = list(cem.cem(f, th0, 8, 2, 0.25))
    assert len(infos) == 2 and infos[0]["ys"].shape == (8,)


@pytest.mark.parametrize("head", [0, 1])
def test_batch_gather_matches_oracle_on_the_subset(head):
    """mrl_batch_gather: a minibatch gathered on the device from the resident batch gives the oracle's loss and
    gradient on ob[idx] (ppo.py:194-199 slices numpy arrays); 1e-5 as everywhere."""
    from modular_rl_b200 import device, synth
    from oracle import policy_math as pm
    dims = (13, 32, 16, 3) if head == 0 else (13, 32, 16, 5)
    wl = synth.Workload("g", dims, head, 1000, 100, 5)
    spec = pm.NetSpec(dims, pm.GAUSS if head == 0 else pm.CAT)

    def fwd(th, ob):
        _, z = pm.forward(th, spec, ob)
        return z if head == 0 else pm.softmax(z)
    d = synth.policy_batch(wl, fwd)
    theta = synth.perturb(d["theta"], 0.03, 2)
    net = device.DeviceNet(dims, head)
    full = device.DeviceBatch(dims[0], True)
    full.set_obs(d["ob"]).set_policy_inputs(head, dims[-1], d["act"], d["adv"], d["oldprob"])
    net.set_params(theta)
    rng = np.random.default_rng(1)
    for n in (128, 77, 1, 300):
        idx = rng.permutation(1000)[:n].astype(np.int32)
        mb = device.DeviceBatch(dims[0], True).gather_from(full, idx)
        pen, g, ls = net.ppo_lossgrad(mb, 0.5, 1e-4, False)
        open_, og = pm.ppo_lossgrad(theta, spec, d["ob"][idx], d["act"][idx], d["adv"][idx], d["oldprob"][idx], 0.5, 1e-4)
        assert np.linalg.norm(g - og) / np.linalg.norm(og) < 2e-5, n
        ols, _, _ = pm.surr_kl_grads(theta, spec, d["ob"][idx], d["act"][idx], d["adv"][idx], d["oldprob"][idx], ratio="lik")
        assert np.allclose(ls, ols, rtol=1e-5, atol=2e-7), (n, ls, ols)
    # the source batch is untouched
    _, g_full, _ = net.ppo_lossgrad(full, 0.5, 1e-4, False)
    _, og_full = pm.ppo_lossgrad(theta, spec, d["ob"], d["act"], d["adv"], d["oldprob"], 0.5, 1e-4)
    assert np.linalg.norm(g_full - og_full) / np.linalg.norm(og_full) < 2e-5
