"""Nets whose fused mid_* kernels do not fit in shared memory (two hidden layers wider than about 88 units, three or
more hidden layers of 64, ...): mrl_net_create sends layers >= 2 to the layer-by-layer path (mlp_layers.cu).  Every
entry point on such nets against the float64 oracle, with the tolerances of test_gpu_parity.test_synthetic_shapes;
the limits that still reject a net; device rollouts and CEM populations with wide policies; the CLIs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import test_gpu_device_envs as de
from conftest import relerr

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-5

# dims, head (0 DiagGauss, 1 Categorical), N, activation.  Each one needs more shared memory than the fused reverse
# sweep can have on a B200 (mid_backward_smem + 2 KB > 232 448 B) and fits the layer-1 tensor-memory budget.
SHAPES = {
    "cat_128x2": ((4, 128, 128, 2), 1, 3000, "tanh"),
    "gauss_256x2": ((11, 256, 256, 3), 0, 2500, "tanh"),
    "gauss_256_128_64_relu": ((17, 256, 128, 64, 6), 0, 2000, "relu"),
    "cat_96x4_sigmoid": ((6, 96, 96, 96, 96, 3), 1, 1500, "sigmoid"),
    "gauss_64x5": ((17, 64, 64, 64, 64, 64, 6), 0, 1800, "tanh"),
    "cat_200_240": ((200, 240, 64, 5), 1, 1200, "tanh"),
    "gauss_one_hidden": ((12, 256, 33), 0, 1000, "tanh"),
}


@pytest.fixture(scope="module")
def dev():
    from modular_rl_b200 import _lib, device
    _lib.lib()
    return device


def _case(dims, head, N, act, seed=11):
    from modular_rl_b200 import synth
    from oracle import policy_math as pm
    wl = synth.Workload("wide", dims, head, N, min(200, N), seed)
    spec = pm.NetSpec(dims, pm.GAUSS if head == 0 else pm.CAT, act)

    def fwd(th, ob):
        _, z = pm.forward(th, spec, ob)
        return z if head == 0 else pm.softmax(z)
    data = synth.policy_batch(wl, fwd)
    return spec, synth.perturb(data["theta"], 0.02, 5), data


def _bind(dev, spec, head, d, theta):
    net = dev.DeviceNet(spec.dims, head, spec.activation)
    batch = dev.DeviceBatch(spec.dims[0], with_time_feature=True)
    batch.set_obs(d["ob"])
    N = d["ob"].shape[0]
    batch.set_paths(np.array([0, N], np.int64), np.array([1], np.uint8), 1000.0)
    batch.set_policy_inputs(head, spec.dims[-1], d["act"], d["adv"], d["oldprob"])
    net.set_params(theta)
    return net, batch


@pytest.mark.parametrize("name", list(SHAPES))
def test_wide_shapes(dev, name):
    from oracle import natgrad, policy_math as pm
    dims, head, N, act = SHAPES[name]
    spec, theta, d = _case(dims, head, N, act)
    net, batch = _bind(dev, spec, head, d, theta)
    args = (d["ob"], d["act"], d["adv"], d["oldprob"])
    ls = net.losses(batch)
    assert np.allclose(ls, pm.losses(theta, spec, *args), rtol=TOL, atol=2e-7)
    g, _ = net.policy_gradient(batch)
    assert relerr(g, pm.policy_gradient(theta, spec, *args)) < TOL
    v = np.random.default_rng(3).standard_normal(net.P).astype(np.float32)
    f = net.fvp(batch, v)
    assert relerr(f, pm.fisher_vector_product(theta, spec, d["ob"], v)) < TOL
    assert np.array_equal(net.fvp(batch, v), f)
    out = net.forward(batch)
    _, z = pm.forward(theta, spec, d["ob"])
    assert relerr(out, z if head == 0 else pm.softmax(z)) < TOL
    stats, info = net.trpo_step(batch, cg_damping=0.1, max_kl=0.01)
    ostats, oinfo = natgrad.trpo_update(theta, spec, *args, 0.1, 0.01)
    assert info["success"] == int(oinfo["success"]) and info["accepted_index"] == oinfo["accepted_index"]
    assert info["cg_iters_run"] == oinfo["cg_iters_run"]
    sd, fs, _ = net.trpo_vectors()
    # step-direction rule of test_synthetic_shapes: 1e-5, or as close to float64 as the reference's float32 path
    _, o32 = natgrad.trpo_update(theta, spec, *args, 0.1, 0.01, dtype=np.float32)
    floor = relerr(o32["stepdir"], oinfo["stepdir"])
    assert relerr(sd, oinfo["stepdir"]) < max(TOL, 1.5 * floor)
    assert relerr(fs, oinfo["fullstep"]) < max(TOL, 1.5 * floor)
    assert relerr(net.get_params(), oinfo["theta_new"]) < 1e-5
    want = np.array([ostats[k] for k in ("surr_before", "surr_after", "kl_before", "kl_after",
                                         "ent_before", "ent_after")])
    assert np.allclose(stats, want, rtol=1e-4, atol=1e-6), (stats, want)


# 1, 63, 64, 65 timesteps; 1000 (the last 8-timestep group of the last tile is partial); 70 001 (many slabs)
@pytest.mark.parametrize("name", ["gauss_256x2", "cat_128x2"])
@pytest.mark.parametrize("N", [1, 63, 64, 65, 1000, 70_001])
def test_batch_sizes(dev, name, N):
    from oracle import policy_math as pm
    dims, head, _, act = SHAPES[name]
    spec, theta, d = _case(dims, head, N, act, seed=N % 97)
    # synth standardises the advantages, which leaves NaN for a single timestep: draw them directly
    d["adv"] = np.random.default_rng(N).standard_normal(N).astype(np.float32)
    net, batch = _bind(dev, spec, head, d, theta)
    args = (d["ob"], d["act"], d["adv"], d["oldprob"])
    assert np.allclose(net.losses(batch), pm.losses(theta, spec, *args), rtol=TOL, atol=2e-7)
    g, _ = net.policy_gradient(batch)
    assert relerr(g, pm.policy_gradient(theta, spec, *args)) < TOL
    v = np.random.default_rng(5).standard_normal(net.P).astype(np.float32)
    f = net.fvp(batch, v)
    assert relerr(f, pm.fisher_vector_product(theta, spec, d["ob"], v)) < TOL
    g2, _ = net.policy_gradient(batch)
    assert np.array_equal(g2, g) and np.array_equal(net.fvp(batch, v), f)


@pytest.mark.parametrize("vdims,N", [((5, 256, 256, 1), 4001), ((13, 128, 128, 128, 1), 3000)])
def test_vf_lossgrad_and_fit(dev, vdims, N):
    from modular_rl_b200 import core, synth
    from oracle import policy_math as pm, valuefn as vf
    rng = np.random.default_rng(3)
    off = np.asarray(synth.make_paths(N, 300, rng)[0], np.int64)
    ob = synth.make_obs(N, vdims[0] - 1, rng)
    y = rng.standard_normal(N)
    theta = synth.init_params(vdims, synth.VALUE, rng, last_scale=1.0)
    net = dev.DeviceNet(vdims, 2)
    b = dev.DeviceBatch(vdims[0] - 1, with_time_feature=True)
    b.set_obs(ob).set_paths(off, np.ones(len(off) - 1, np.uint8), 300.0)
    b.set_vf_target(y)
    net.set_params(theta)
    spec = pm.NetSpec(vdims, pm.VALUE)
    tidx = np.concatenate([np.arange(off[i + 1] - off[i]) for i in range(len(off) - 1)])
    x = np.concatenate([ob.astype(np.float64), (tidx / 300.0)[:, None]], axis=1)
    assert relerr(net.forward(b), vf.vf_forward(theta, spec, x)) < TOL
    ls, g = net.vf_lossgrad(b, 1e-3)
    _, og = vf.vf_lossgrad(theta, spec, x, y.reshape(-1, 1), l2coeff=1e-3)
    assert np.allclose(ls, vf.vf_losses(theta, spec, x, y.reshape(-1, 1), l2coeff=1e-3), rtol=TOL)
    assert relerr(g, og) < TOL
    # one NnVf.fit (L-BFGS on float32) against the float64 regression
    vfn = core.NnVf(net, 300, dict(mixfrac=0.1, maxiter=25))
    paths = [dict(observation=ob[off[i]:off[i + 1]], **{"return": y[off[i]:off[i + 1]]}) for i in range(len(off) - 1)]
    vstats = vfn.fit(paths)
    ostats, _, _ = vf.regression_fit(theta.astype(np.float64), spec, x, y.reshape(-1, 1), mixfrac=0.1, maxiter=25)
    for k in ("loss_before", "mse_before", "l2_before", "TargStdev", "PredStdevBefore", "EV_before"):
        assert np.isclose(vstats[k], ostats[k], rtol=1e-4, atol=1e-6), (k, vstats[k], ostats[k])
    assert vstats["loss_after"] < vstats["loss_before"]
    assert np.isclose(vstats["loss_after"], ostats["loss_after"], rtol=2e-2)


@pytest.mark.parametrize("name", ["gauss_256x2", "cat_128x2"])
@pytest.mark.parametrize("rev", [False, True])
def test_ppo_lossgrad(dev, name, rev):
    from oracle import policy_math as pm
    dims, head, N, act = SHAPES[name]
    spec, theta, d = _case(dims, head, N, act)
    net, batch = _bind(dev, spec, head, d, theta)
    args = (d["ob"], d["act"], d["adv"], d["oldprob"])
    klc, cutoff = 0.7, 1e-4
    pen, g, _ = net.ppo_lossgrad(batch, klc, cutoff, rev)
    open_, og = pm.ppo_lossgrad(theta, spec, *args, klc, cutoff, reverse_kl=rev)
    ols, _, _ = pm.surr_kl_grads(theta, spec, *args, ratio="lik", reverse_kl=rev)
    dpen_dkl = klc + 2000.0 * (ols[1] > cutoff) * (ols[1] - cutoff)
    assert abs(pen - open_) < TOL * (abs(ols[0]) + abs(dpen_dkl) * ols[1]) + 1e-7
    assert relerr(g, og) < 2 * TOL


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_ppo_sgd_updater(kind):
    """PpoSgdUpdater (minibatch gather + Adam) on a 256-256 policy against oracle/ppo_sgd.py, same permutations."""
    from modular_rl_b200 import agentzoo, spaces
    from oracle import policy_math as pm
    from oracle.ppo_sgd import Adam, ppo_sgd_update
    from modular_rl_b200.core import DiagGauss
    import test_gpu_api as api
    rng = np.random.default_rng(2)
    ob_space = spaces.Box(-np.ones(6), np.ones(6))
    ac_space = spaces.Box(-np.ones(2), np.ones(2)) if kind == "box" else spaces.Discrete(3)
    agent = agentzoo.PpoSgdAgent(ob_space, ac_space, dict(hid_sizes=[256, 256], timestep_limit=60, epochs=2,
                                                            stepsize=1e-3))
    paths = api._make_paths(rng, 12, 6, agent.policy)
    for p in paths:
        p["advantage"] = rng.standard_normal(len(p["reward"]))
    theta = agent.policy.get_flat().astype(np.float64)
    spec = pm.NetSpec(tuple(agent.policy.dims), pm.GAUSS if isinstance(agent.policy.probtype, DiagGauss) else pm.CAT)
    cat = lambda k: np.concatenate([p[k] for p in paths])
    np.random.seed(7)
    out = agent.updater(paths)
    np.random.seed(7)
    oinfo, oth, oklc, _ = ppo_sgd_update(theta, spec, cat("observation"), cat("action"), cat("advantage"),
                                         Adam(theta.size, 1e-3), epochs=2)
    assert list(out) == list(oinfo)
    for k in out:
        assert np.isclose(out[k], oinfo[k], rtol=2e-3, atol=2e-5), (k, out[k], oinfo[k])
    assert agent.updater.kl_coeff == oklc
    th = agent.policy.get_flat()
    assert np.abs(th - oth).max() < 5e-3 and relerr(th, oth) < 2e-3


@pytest.mark.parametrize("dims,msg", [
    ((4, 257, 2), "layer width 257 > 256"),
    ((4, 64, 65), "output dim 65 > 64"),
    ((4, 16, 16, 16, 16, 16, 16, 2), "1..6 layers"),
    ((376, 160, 64, 17), "exceeds the TMEM budget"),
])
def test_limits_still_reject(dev, dims, msg):
    with pytest.raises(RuntimeError, match=msg):
        dev.DeviceNet(dims, 0)


def test_device_rollout_round_with_wide_policy():
    """4-256-256-2: 67 586 floats of theta (264 KB), read through L2 by the rollout kernel."""
    pol = de._policy("cartpole", (256, 256), "tanh", scale=0.1)
    assert pol.get_flat().size == 67_586
    out = de._run("cartpole", 64, 100, 31, pol)
    de._check_round("cartpole", out, 31, pol, 100, envs_checked=[0, 21, 63])


def test_population_round_with_wide_policy(monkeypatch):
    """DeterministicAgent hid_sizes=[256, 256]: device scores bit-identical to cem.evaluate_population started from
    the device's reset states."""
    from modular_rl_b200 import agentzoo, cem, envs
    from oracle import rollout as orc
    env = envs.CartPoleEnv()
    np.random.seed(0)
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[256, 256], filter=0))
    dims = agent.policy.dims
    P = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(dims) - 1))
    th = (np.random.default_rng(12).standard_normal((24, P)) * 0.1).astype(np.float32)
    seed = 77
    dev_scores = cem.evaluate_population_device(env, agent, th, 200, seed)
    starts = orc.reset_states("cartpole", seed, np.arange(24))
    made = [0]

    def reset(self):
        self.state = starts[made[0]].copy()
        made[0] += 1
        return np.array(self.state)
    monkeypatch.setattr(envs.CartPoleEnv, "reset", reset)
    host = cem.evaluate_population(env, agent, th, 200)
    assert made[0] == 24
    assert np.array_equal(host, dev_scores), (host, dev_scores)


def test_run_pg_cartpole_128x2_learns(tmp_path):
    """run_pg.py --hid_sizes 128,128 with device rollouts.  The threshold comes from one measured run on a B200, in
    which EpRewMean went from 22.4 to 200 over the 8 iterations; the check asks for twice the first iteration."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "run_pg.py"), "--env", "CartPole-v0", "--agent",
                          "modular_rl.agentzoo.TrpoAgent", "--hid_sizes", "128,128", "--n_iter", "8",
                          "--timesteps_per_batch", "2000", "--seed", "0", "--cg_damping", "0.1", "--lam", "0.97",
                          "--device_envs", "256", "--outfile", str(tmp_path / "a.h5")],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    rews = [float(ln.split()[-1]) for ln in out.stdout.splitlines() if ln.startswith("EpRewMean")]
    assert len(rews) == 8
    assert max(rews[-3:]) > 2.0 * rews[0], rews


def test_run_cem_256x2_device_envs(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "run_cem.py"), "--env", "CartPole-v0", "--agent",
                          "modular_rl.agentzoo.DeterministicAgent", "--hid_sizes", "256,256", "--device_envs",
                          "--n_iter", "2", "--batch_size", "40", "--outfile", str(tmp_path / "c.h5")],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "device_envs: one device rollout round per generation" in out.stdout
