"""PPO with the clipped surrogate objective on the GPU: the loss, clipfrac and gradient of every kernel path against
the float64 oracle (oracle/ppo_clip.py), the eps = inf limit against the surrogate, a whole PpoClipUpdater call
against the oracle's replay, agent snapshots, and learning runs of run_pg.py."""
import pickle

import numpy as np
import pytest

import test_gpu_api as api
import test_gpu_device_envs as de
from conftest import relerr

pytestmark = pytest.mark.gpu

EPS = 0.2
# dims, head (0 DiagGauss, 1 Categorical), activation, kernel path of layers >= 2
NETS = {
    "chain_gauss": ((11, 64, 64, 3), 0, "tanh"),          # register chains (mlp_chain.cu)
    "chain_cat": ((6, 64, 64, 4), 1, "tanh"),
    "mid_gauss_relu": ((11, 64, 64, 3), 0, "relu"),       # fused mid_* kernels (mlp_mid.cu)
    "mid_cat_3hidden": ((6, 32, 32, 32, 5), 1, "tanh"),
    "layers_gauss": ((11, 256, 256, 3), 0, "tanh"),       # layer by layer (mlp_layers.cu)
    "layers_cat": ((4, 128, 128, 2), 1, "tanh"),
}
N = 3001          # several slabs, not a multiple of 64


def _case(name, seed=1):
    """Float32 inputs, an old policy and parameters moved away from it until 10 - 60 % of the rows are clipped;
    rows whose float64 ratio is within 1e-4 of a clip boundary are dropped."""
    from oracle import policy_math as pm, ppo_clip
    dims, head, act_fn = NETS[name]
    spec = pm.NetSpec(dims, pm.GAUSS if head == 0 else pm.CAT, act_fn)
    rng = np.random.default_rng(seed)
    old = pm.init_params(spec, rng, last_scale=1.0)
    ob = rng.standard_normal((N, dims[0])).astype(np.float32)
    _, z0 = pm.forward(old, spec, ob)
    oldprob = pm.head_prob(old.astype(np.float64), spec, z0).astype(np.float32)
    d = dims[-1]
    if head == 0:
        act = (oldprob[:, :d] + oldprob[:, d:] * rng.standard_normal((N, d))).astype(np.float32)
    else:
        p = oldprob.astype(np.float64)
        act = np.array([rng.choice(d, p=q / q.sum()) for q in p], np.int32)
    adv = rng.standard_normal(N).astype(np.float32)
    step = rng.standard_normal(old.size).astype(np.float32)
    for scale in (0.01, 0.02, 0.04, 0.08, 0.16, 0.32):
        theta = (old + scale * step).astype(np.float32)
        r = ppo_clip.ratio(theta.astype(np.float64), spec, ob, act, oldprob)
        if np.mean((r < 1 - EPS) | (r > 1 + EPS)) >= 0.15:
            break
    keep = (np.abs(r - (1 - EPS)) > 1e-4) & (np.abs(r - (1 + EPS)) > 1e-4)
    return spec, head, theta, ob[keep], act[keep], adv[keep], oldprob[keep]


def _bind(spec, head, theta, ob, act, adv, oldprob):
    from modular_rl_b200 import device
    net = device.DeviceNet(spec.dims, head, spec.activation)
    batch = device.DeviceBatch(spec.dims[0], with_time_feature=True)
    batch.set_obs(ob)
    batch.set_paths(np.array([0, len(ob)], np.int64), np.array([1], np.uint8), 1000.0)
    batch.set_policy_inputs(head, spec.dims[-1], act, adv, oldprob)
    net.set_params(theta)
    return net, batch


@pytest.mark.parametrize("name", list(NETS))
def test_lossgrad_matches_oracle(name):
    from oracle import ppo_clip
    spec, head, theta, ob, act, adv, oldprob = _case(name)
    r = ppo_clip.ratio(theta.astype(np.float64), spec, ob, act, oldprob)
    out = (r < 1 - EPS) | (r > 1 + EPS)
    assert 0.10 <= out.mean() <= 0.60 and (out & (adv > 0)).any() and (out & (adv < 0)).any(), out.mean()
    assert np.min(np.abs(np.concatenate([r - (1 - EPS), r - (1 + EPS)]))) > 1e-4
    net, batch = _bind(spec, head, theta, ob, act, adv, oldprob)
    g, ls = net.ppo_clip_lossgrad(batch, EPS)
    ols, og = ppo_clip.clip_lossgrad(theta, spec, ob, act, adv, oldprob, EPS)
    assert np.allclose(ls[:3], ols[:3], rtol=1e-5, atol=1e-7), (ls, ols)
    assert round(ls[3] * len(ob)) == out.sum() and abs(ls[3] - ols[3]) <= 1e-15, (ls[3], ols[3])   # same rows
    assert relerr(g, og) < 1e-5
    _, ls2 = net.ppo_clip_lossgrad(batch, EPS, want_grad=False)
    assert np.array_equal(ls2, ls)
    g2, _ = net.ppo_clip_lossgrad(batch, EPS)
    assert np.array_equal(g2, g)


@pytest.mark.parametrize("name", list(NETS))
def test_no_clipping_is_the_surrogate(name):
    spec, head, theta, ob, act, adv, oldprob = _case(name, seed=2)
    net, batch = _bind(spec, head, theta, ob, act, adv, oldprob)
    g, ls = net.ppo_clip_lossgrad(batch, float("inf"))
    _, sg, sls = net.ppo_lossgrad(batch, 0.0, 1e300)
    assert ls[3] == 0.0
    assert abs(ls[0] - sls[0]) <= 1e-6 * abs(sls[0]) and np.allclose(ls[1:3], sls[1:3], rtol=1e-6)
    assert relerr(g, sg) < 1e-6


def test_rejections():
    from modular_rl_b200 import device
    spec, head, theta, ob, act, adv, oldprob = _case("chain_cat")
    net, batch = _bind(spec, head, theta, ob, act, adv, oldprob)
    for bad in (0.0, -1.0, float("nan")):
        with pytest.raises(RuntimeError, match="clip_eps must be > 0"):
            net.ppo_clip_lossgrad(batch, bad)
        with pytest.raises(RuntimeError, match="clip_eps must be > 0"):
            net.ppo_clip_sgd_step(batch, bad, 1e-3)
    vf = device.DeviceNet((spec.dims[0], 8, 1), 2)
    with pytest.raises(RuntimeError, match="value net"):
        vf.ppo_clip_lossgrad(batch, EPS)
    with pytest.raises(RuntimeError, match="value net"):
        vf.ppo_clip_sgd_step(batch, EPS, 1e-3)


def _agent_and_paths(kind, cfg, seed=2):
    from modular_rl_b200 import agentzoo, spaces
    rng = np.random.default_rng(seed)
    ob_space = spaces.Box(-np.ones(6), np.ones(6))
    ac_space = spaces.Box(-np.ones(2), np.ones(2)) if kind == "box" else spaces.Discrete(3)
    agent = agentzoo.PpoClipAgent(ob_space, ac_space, dict(hid_sizes=[16, 8], timestep_limit=60, **cfg))
    paths = api._make_paths(rng, 12, 6, agent.policy)
    for p in paths:
        p["advantage"] = rng.standard_normal(len(p["reward"]))
    return agent, paths


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_updater_matches_oracle_replay(kind):
    from oracle.ppo_clip import ppo_clip_update
    from oracle.ppo_sgd import Adam
    agent, paths = _agent_and_paths(kind, dict(epochs=2, minibatch_size=64, stepsize=1e-2))
    cat = lambda k: np.concatenate([p[k] for p in paths])
    n = len(cat("reward"))
    assert n % 64 != 0 and n > 128
    theta = agent.policy.get_flat()
    spec = api._oracle_spec(agent.policy)
    np.random.seed(7)
    info = agent.updater(paths)
    np.random.seed(7)
    oinfo, oth = ppo_clip_update(theta, spec, cat("observation"), cat("action"), cat("advantage"),
                                 Adam(theta.size, 1e-2, dtype=np.float32), clip_eps=0.2, epochs=2, minibatch_size=64)
    assert list(info) == list(oinfo)
    for k in info:
        assert np.isclose(info[k], oinfo[k], rtol=1e-5, atol=1e-7), (k, info[k], oinfo[k])
    assert info["clipfrac"] > 0
    assert relerr(agent.policy.get_flat(), oth) < 1e-5


@pytest.mark.parametrize("kind", ["box", "discrete"])
def test_snapshot_twin_updates_bit_identically(kind):
    agent, paths = _agent_and_paths(kind, dict(epochs=3, minibatch_size=32, stepsize=1e-2))
    rng = np.random.default_rng(4)
    agent.policy.set_params_flat(agent.policy.get_params_flat() + 0.05 * rng.standard_normal(agent.policy.net.P))
    twin = pickle.loads(pickle.dumps(agent, -1))
    assert type(twin).__name__ == "PpoClipAgent" and twin.updater.cfg == agent.updater.cfg
    infos = []
    for a in (agent, twin):
        np.random.seed(11)
        infos.append(a.updater(paths))
    for k in infos[0]:
        assert infos[0][k] == infos[1][k], (k, infos[0][k], infos[1][k])
    assert infos[0]["clipfrac"] > 0
    np.testing.assert_array_equal(twin.policy.get_params_flat(), agent.policy.get_params_flat())


def _rews(stdout):
    return [float(ln.split()[-1]) for ln in stdout.splitlines() if ln.startswith("EpRewMean")]


def test_run_pg_cartpole_learns(tmp_path):
    """CartPole-v0 with device rollouts.  Measured on an NVIDIA B200 (1000 W power limit), EpRewMean per iteration:
    21.4, 35.7, 66.4, 132, 186, 199, 200, 200, 200, 200."""
    stdout = de._run_pg(["--env", "CartPole-v0", "--agent", "modular_rl.agentzoo.PpoClipAgent", "--n_iter", "10",
                         "--timesteps_per_batch", "5000", "--seed", "0", "--lam", "0.95", "--device_envs", "256",
                         "--outfile", str(tmp_path / "a.h5")])
    rews = _rews(stdout)
    assert len(rews) == 10
    assert "clipfrac" in stdout
    assert np.mean(rews[-3:]) > 150.0, rews


def test_run_pg_point_mass_improves(tmp_path):
    """PointMass-v0 (DiagGauss d = 2) with device rollouts.  Measured on an NVIDIA B200 (1000 W power limit),
    EpRewMean per iteration: -21106, -12606, -6768, -3336, -1573, -557, -213, -98.5."""
    stdout = de._run_pg(["--env", "examples.point_mass:PointMass-v0", "--agent", "modular_rl.agentzoo.PpoClipAgent",
                         "--n_iter", "8", "--timesteps_per_batch", "20000", "--seed", "0", "--gamma", "0.99",
                         "--lam", "0.97", "--device_envs", "256", "--outfile", str(tmp_path / "b.h5")])
    rews = _rews(stdout)
    assert len(rews) == 8
    assert np.mean(rews[-2:]) > -1000.0, rews
