"""Oracle (test infrastructure): PPO with the clipped surrogate objective, in closed form through the MLP of
policy_math, and a replay of one PpoClipUpdater call.

    L(theta) = -(1/N) sum_t min(r_t A_t, clip(r_t, 1 - eps, 1 + eps) A_t),   r_t = pi(a_t | s_t) / pi_old(a_t | s_t)

A row carries the surrogate's gradient -(1/N) A_t dr_t/dtheta unless (A_t > 0 and r_t > 1 + eps) or
(A_t < 0 and r_t < 1 - eps); at r_t = 1 +- eps it does (torch autograd of torch.minimum / torch.clamp gives the
same).  clipfrac is the fraction of rows with r_t outside [1 - eps, 1 + eps].  eps = inf is the plain surrogate.
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np

from . import policy_math as pm
from .ppo_sgd import Adam, _oldprob


def ratio(theta, spec, ob, act, oldprob, dtype=np.float64):
    """r_t as the device forms it: exp(logp - logp_old) (DiagGauss), p_a / p0_a (Categorical)."""
    _, z = pm.forward(theta, spec, ob, dtype)
    prob = pm.head_prob(np.asarray(theta, dtype), spec, z, dtype)
    oldprob = np.asarray(oldprob, dtype)
    if spec.head == pm.GAUSS:
        d = spec.dims[-1]
        a = np.asarray(act, dtype)
        return np.exp(pm.gauss_loglik(a, prob, d) - pm.gauss_loglik(a, oldprob, d))
    return pm.cat_lik(np.asarray(act), prob) / pm.cat_lik(np.asarray(act), oldprob)


def clip_lossgrad(theta, spec, ob, act, adv, oldprob, clip_eps, dtype=np.float64):
    """-> (losses [surr, kl, ent, clipfrac], gradient of surr [P]); kl = mean KL[old, new]."""
    th = np.asarray(theta, dtype)
    Ws, _, _ = pm.split_params(th, spec)
    hs, z = pm.forward(th, spec, ob, dtype)
    prob = pm.head_prob(th, spec, z, dtype)
    oldprob = np.asarray(oldprob, dtype)
    adv = np.asarray(adv, dtype)
    N = ob.shape[0]
    d = spec.dims[-1]
    r = ratio(th, spec, ob, act, oldprob, dtype)
    lo, hi = 1.0 - clip_eps, 1.0 + clip_eps
    obj = np.minimum(r * adv, np.clip(r, lo, hi) * adv)
    gated = ((adv > 0) & (r > hi)) | ((adv < 0) & (r < lo))
    w = np.where(gated, 0.0, -r * adv / N)[:, None]
    if spec.head == pm.GAUSS:
        a = np.asarray(act, dtype)
        std = prob[:, d:]
        dz = w * (a - z) / np.square(std)
        dls = (w * (np.square((a - z) / std) - 1.0)).sum(axis=0)
        g = pm._backprop(spec, Ws, hs, dz, dls)
    else:
        onehot = np.zeros_like(prob)
        onehot[np.arange(N), np.asarray(act).astype(np.int64)] = 1.0
        g = pm._backprop(spec, Ws, hs, w * (onehot - prob))
    ls = np.array([-obj.mean(), pm.kl_rows(spec, oldprob, prob).mean(), pm.entropy_rows(spec, prob).mean(),
                   ((r < lo) | (r > hi)).mean()], np.float64)
    return ls, g


def ppo_clip_update(theta, spec, ob, act, adv, adam: Adam, clip_eps=0.2, epochs=10, minibatch_size=64,
                    oldprob=None, dtype=np.float64):
    """Replays one PpoClipUpdater call -> (info OrderedDict, theta_new).  The permutations come from numpy's global
    generator in the updater's order; each minibatch's gradient is taken in `dtype` at the current parameters and
    applied by `adam` (pass Adam(..., dtype=np.float32) for the device's float32 step).  oldprob: the old policy's
    prob rows (default: a forward pass at theta)."""
    N = ob.shape[0]
    theta = np.asarray(theta, adam.f)
    if oldprob is None:
        oldprob = _oldprob(theta, spec, ob, dtype)
    before, _ = clip_lossgrad(theta, spec, ob, act, adv, oldprob, clip_eps, dtype)
    for _ in range(epochs):
        perm = np.random.permutation(N)
        for istart in range(0, N, minibatch_size):
            idx = perm[istart:istart + minibatch_size]
            _, g = clip_lossgrad(theta, spec, ob[idx], act[idx], adv[idx], oldprob[idx], clip_eps, dtype)
            theta = adam.step(theta, g)
    after, _ = clip_lossgrad(theta, spec, ob, act, adv, oldprob, clip_eps, dtype)
    info = OrderedDict()
    for name, lb, la in zip(("surr", "kl", "ent"), before[:3], after[:3]):
        info[name + "_before"] = lb
        info[name + "_after"] = la
        info[name + "_change"] = la - lb
    info["clipfrac"] = after[3]
    return info, theta
