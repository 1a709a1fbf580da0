"""numpy restatement of the cross-entropy method's device search (modular_rl_b200/csrc/cem_search.cu, DESIGN.md 4b
"Device search"): the candidate normals, the draw, the stable elite rule and the refit.

Normals: Philox4x32-10 (oracle/rollout.py) keyed by the generation's round seed, counter (member m, pair p = j // 2,
purpose 2, block 0); the block gives (u0, u1) and z[m, 2p] = r cos(2 pi u1), z[m, 2p + 1] = r sin(2 pi u1) with
r = sqrt(-2 log(1 - u0)), all in float64.  The device evaluates cos(2 pi u1) as cospi(2 u1), without rounding the
argument, and its log / sincospi are within an ulp or two of numpy's: draws agree to a few float64 ulp, not bits.
"""
import numpy as np

from .rollout import philox4x32_10, seed_key, u53

PURPOSE_DRAW = 2


def normals(seed, members, P):
    """z float64 [len(members), P] of the given members."""
    members = np.asarray(members, np.uint64)
    pairs = np.arange((P + 1) // 2, dtype=np.uint64)
    m, p = np.meshgrid(members, pairs, indexing="ij")
    ctr = np.stack([m, p, np.full(m.shape, PURPOSE_DRAW, np.uint64), np.zeros(m.shape, np.uint64)], axis=-1)
    x = philox4x32_10(ctr, seed_key(seed))
    u0, u1 = u53(x[..., 0], x[..., 1]), u53(x[..., 2], x[..., 3])
    r = np.sqrt(-2.0 * np.log(1.0 - u0))
    z = np.empty((len(members), 2 * len(pairs)))
    z[:, 0::2] = r * np.cos(2.0 * np.pi * u1)
    z[:, 1::2] = r * np.sin(2.0 * np.pi * u1)
    return z[:, :P]


def deviation(var, extra_var, noise_left):
    """_GaussianSearch.draw's dev = sqrt(var + extra_var * noise_left)."""
    return np.sqrt(np.asarray(var, np.float64) + extra_var * noise_left)


def candidates(mean, dev, seed, members, chunk=512):
    """float64 rows mean + dev * z of the given members (chunks of `chunk` members bound the temporaries)."""
    members = np.asarray(members)
    mean, dev = np.asarray(mean, np.float64), np.asarray(dev, np.float64)
    out = np.empty((len(members), mean.size))
    for i in range(0, len(members), chunk):
        out[i:i + chunk] = mean[None, :] + dev[None, :] * normals(seed, members[i:i + chunk], mean.size)
    return out


def draw(mean, var, extra_var, noise_left, seed, M):
    """-> (float64 rows [M, P], dev [P]); the device stores the rows rounded to float32."""
    dev = deviation(var, extra_var, noise_left)
    return candidates(mean, dev, seed, np.arange(M)), dev


def elite(scores, keep):
    """np.argsort(scores, kind="stable")[-keep:] in ascending order: ties to the higher index, NaN last; keep == 0
    (numpy's [-0:]) and keep > M select every member."""
    if keep < 0:
        raise ValueError("keep = %d is negative" % keep)
    scores = np.asarray(scores, np.float64)
    n = scores.size if keep == 0 or keep > scores.size else keep
    key_nan = np.isnan(scores)
    # the rule spelled out: sort by (is NaN, score, index); np.lexsort sorts by its last key first
    order = np.lexsort((np.arange(scores.size), np.where(key_nan, 0.0, scores), key_nan))
    return order[scores.size - n:]


def refit(mean, dev, seed, scores, keep):
    """New (mean, var) of the elite rows recomputed in float64, in elite order: best.mean(axis=0), best.var(axis=0)."""
    best = candidates(mean, dev, seed, elite(scores, keep))
    return best.mean(axis=0), best.var(axis=0)
