"""PPO with the clipped surrogate objective, on the CPU: the oracle's closed-form loss, gradient and clipfrac against
torch float64 autograd of the textbook expression, the eps = inf limit, the updater's option table, the
data-parallel rejection, and the argument checks of the two C entry points (no device needed)."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from oracle import policy_math as pm
from oracle import ppo_clip

EPS = 0.2
CASES = [("gauss", 1), ("gauss", 3), ("cat", 2), ("cat", 5)]


def _point(head, d, seed, N=400):
    """A net, its inputs and an old policy far enough from it that rows fall on all sides of the gate; rows within
    1e-6 of a clip boundary are dropped (there the two sides of the gate differ by one row's share)."""
    rng = np.random.default_rng(seed)
    spec = pm.NetSpec((5, 12, 7, d), pm.GAUSS if head == "gauss" else pm.CAT)
    theta = pm.init_params(spec, rng, last_scale=1.0).astype(np.float64)
    ob = rng.standard_normal((N, 5))
    old = theta + 0.3 * rng.standard_normal(theta.size)
    _, z0 = pm.forward(old, spec, ob)
    oldprob = pm.head_prob(old, spec, z0)
    if head == "gauss":
        act = oldprob[:, :d] + oldprob[:, d:] * rng.standard_normal((N, d))
    else:
        act = np.array([rng.choice(d, p=p / p.sum()) for p in oldprob])
    adv = rng.standard_normal(N)
    r = ppo_clip.ratio(theta, spec, ob, act, oldprob)
    keep = (np.abs(r - (1 - EPS)) > 1e-6) & (np.abs(r - (1 + EPS)) > 1e-6)
    return spec, theta, ob[keep], act[keep], adv[keep], oldprob[keep]


def _torch_loss(theta, spec, ob, act, adv, oldprob, eps):
    import torch
    th = torch.tensor(theta, dtype=torch.float64, requires_grad=True)
    pos, h = 0, torch.tensor(ob, dtype=torch.float64)
    L = spec.n_layers
    for l in range(L):
        din, dout = spec.dims[l], spec.dims[l + 1]
        W = th[pos:pos + din * dout].reshape(din, dout); pos += din * dout
        b = th[pos:pos + dout]; pos += dout
        h = h @ W + b
        if l < L - 1:
            h = torch.tanh(h)
    old = torch.tensor(oldprob, dtype=torch.float64)
    if spec.head == pm.GAUSS:
        d = spec.dims[-1]
        logstd = th[pos:pos + d]
        a = torch.tensor(act, dtype=torch.float64)
        lp = (-0.5 * ((a - h) / torch.exp(logstd)) ** 2 - logstd).sum(1)
        olp = (-0.5 * ((a - old[:, :d]) / old[:, d:]) ** 2 - torch.log(old[:, d:])).sum(1)
        r = torch.exp(lp - olp)
    else:
        idx = torch.tensor(np.asarray(act, np.int64))
        p = torch.softmax(h, 1)
        r = p[torch.arange(len(idx)), idx] / old[torch.arange(len(idx)), idx]
    A = torch.tensor(adv, dtype=torch.float64)
    loss = -(torch.minimum(r * A, torch.clamp(r, 1 - eps, 1 + eps) * A)).mean()
    loss.backward()
    return loss.item(), th.grad.numpy()


@pytest.mark.parametrize("head,d", CASES)
def test_oracle_matches_torch_autograd(head, d):
    spec, theta, ob, act, adv, oldprob = _point(head, d, seed=d + 10 * (head == "cat"))
    r = ppo_clip.ratio(theta, spec, ob, act, oldprob)
    lo, hi = 1 - EPS, 1 + EPS
    sides = [(adv > 0) & (r > hi), (adv < 0) & (r < lo), (adv > 0) & (r < lo), (adv < 0) & (r > hi),
             (r > lo) & (r < hi)]
    assert all(s.any() for s in sides), [int(s.sum()) for s in sides]
    ls, g = ppo_clip.clip_lossgrad(theta, spec, ob, act, adv, oldprob, EPS)
    tl, tg = _torch_loss(theta, spec, ob, act, adv, oldprob, EPS)
    assert abs(ls[0] - tl) <= 1e-10 * max(1.0, abs(tl))
    assert np.linalg.norm(g - tg) <= 1e-10 * np.linalg.norm(tg)
    assert ls[3] == ((r < lo) | (r > hi)).mean() and 0 < ls[3] < 1
    want = pm.surr_kl_grads(theta, spec, ob, act, adv, oldprob, ratio="lik")[0]
    assert np.allclose(ls[1:3], want[1:3], rtol=1e-12)          # KL[old, new] and entropy as the surrogate reports


@pytest.mark.parametrize("head,d", CASES)
def test_oracle_without_clipping_is_the_surrogate(head, d):
    spec, theta, ob, act, adv, oldprob = _point(head, d, seed=3 + d)
    ls, g = ppo_clip.clip_lossgrad(theta, spec, ob, act, adv, oldprob, math.inf)
    want_ls, want_g, _ = pm.surr_kl_grads(theta, spec, ob, act, adv, oldprob, ratio="lik")
    assert ls[3] == 0.0 and abs(ls[0] - want_ls[0]) <= 1e-12 * abs(want_ls[0])
    assert np.linalg.norm(g - want_g) <= 1e-12 * np.linalg.norm(want_g)


def test_option_table_and_defaults():
    from modular_rl_b200 import agentzoo
    from modular_rl_b200.ppo import PpoClipUpdater
    opts = {name: (typ, default) for name, typ, default, _ in PpoClipUpdater.options}
    assert opts == {"clip_param": (float, 0.2), "epochs": (int, 10), "stepsize": (float, 3e-4),
                    "minibatch_size": (int, 64)}
    names = [o[0] for o in agentzoo.PpoClipAgent.options]
    assert len(names) == len(set(names))
    assert names == [o[0] for o in agentzoo.MLP_OPTIONS + agentzoo.PG_OPTIONS + PpoClipUpdater.options
                     + agentzoo.FILTER_OPTIONS]


def test_rejected_in_data_parallel_training(monkeypatch):
    from modular_rl_b200 import agentzoo, envs
    env = envs.make("CartPole-v0")
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(NotImplementedError, match="PpoClipAgent"):
        agentzoo.PpoClipAgent(env.observation_space, env.action_space, {})


@pytest.fixture(scope="module")
def lib():
    from modular_rl_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.lib()


@pytest.mark.parametrize("bad", [0.0, -0.1, float("nan"), 1e-60])
def test_abi_rejects_clip_eps(lib, bad):
    ls = (C.c_double * 4)()
    assert lib.mrl_net_ppo_clip_lossgrad(None, None, bad, None, ls, None) != 0
    assert b"mrl_net_ppo_clip_lossgrad: clip_eps must be > 0" in lib.mrl_last_error()
    assert lib.mrl_net_ppo_clip_sgd_step(None, None, bad, 1e-3, 0.9, 0.999, 1e-8, None) != 0
    assert b"mrl_net_ppo_clip_sgd_step: clip_eps must be > 0" in lib.mrl_last_error()


@pytest.mark.parametrize("eps", [0.2, float("inf")])
def test_abi_rejects_null_handles(lib, eps):
    ls = (C.c_double * 4)()
    assert lib.mrl_net_ppo_clip_lossgrad(None, None, eps, None, ls, None) != 0
    assert b"mrl_net_ppo_clip_lossgrad: null net or batch" in lib.mrl_last_error()
    assert lib.mrl_net_ppo_clip_sgd_step(None, None, eps, 1e-3, 0.9, 0.999, 1e-8, None) != 0
    assert b"mrl_net_ppo_clip_sgd_step: null net or batch" in lib.mrl_last_error()
