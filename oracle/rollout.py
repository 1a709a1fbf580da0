"""numpy restatement of the device rollouts' random stream, reset draws, action rule and lockstep ZFilter
(modular_rl_b200/csrc/rollout.cu, DESIGN.md "Device rollouts").  The dynamics reference is envs.py itself.

Philox4x32-10 (Salmon et al., SC'11; the constants and round of Random123 and curand_philox4x32_x.h), keyed by the
round seed (low word, high word), counter (environment, step, purpose, block).  A uniform takes two output words
(hi, lo): (hi << 21 | lo >> 11) * 2**-53.  Block words (x0, x1) give u0, (x2, x3) give u1.
  reset    purpose 0, step 0: CartPole blocks 0, 1 -> 4 uniforms; Pendulum block 0 -> (u0, u1)
  action   purpose 1, block 0: Categorical u0; DiagGauss z = sqrt(-2 log(1 - u0)) cos(2 pi u1)
"""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)
PURPOSE_RESET, PURPOSE_ACTION = 0, 1


def philox4x32_10(ctr, key):
    """ctr: uint32 [..., 4]; key: (k0, k1) -> uint32 [..., 4]."""
    c = np.asarray(ctr, np.uint64).copy()
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for i in range(10):
        if i:
            k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
        p0 = M0 * c[..., 0]
        p1 = M1 * c[..., 2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c = np.stack([hi1 ^ c[..., 1] ^ np.uint64(k0), lo1, hi0 ^ c[..., 3] ^ np.uint64(k1), lo0], axis=-1)
    return c.astype(np.uint32)


def seed_key(seed):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return seed & 0xFFFFFFFF, seed >> 32


def u53(hi, lo):
    hi = np.asarray(hi, np.uint64)
    lo = np.asarray(lo, np.uint64)
    return ((hi << np.uint64(21)) | (lo >> np.uint64(11))).astype(np.float64) * 2.0 ** -53


def uniforms(seed, env, step, purpose, block=0):
    """(u0, u1) of one counter block; env / step may be arrays."""
    env, step = np.broadcast_arrays(np.asarray(env, np.uint64), np.asarray(step, np.uint64))
    ctr = np.stack([env, step, np.full(env.shape, purpose, np.uint64), np.full(env.shape, block, np.uint64)], axis=-1)
    x = philox4x32_10(ctr, seed_key(seed))
    return u53(x[..., 0], x[..., 1]), u53(x[..., 2], x[..., 3])


def reset_states(kind, seed, envs):
    """Start states of environments `envs` (array of indices) of a round: [len(envs), state_dim]."""
    envs = np.asarray(envs)
    if kind == "cartpole":
        a0, a1 = uniforms(seed, envs, 0, PURPOSE_RESET, 0)
        b0, b1 = uniforms(seed, envs, 0, PURPOSE_RESET, 1)
        u = np.stack([a0, a1, b0, b1], axis=-1)
        return -0.05 + (0.05 - -0.05) * u
    u0, u1 = uniforms(seed, envs, 0, PURPOSE_RESET, 0)
    return np.stack([-np.pi + (np.pi - -np.pi) * u0, -1.0 + (1.0 - -1.0) * u1], axis=-1)


def action_uniform(seed, env, step):
    return uniforms(seed, env, step, PURPOSE_ACTION, 0)[0]


def action_normal(seed, env, step):
    u0, u1 = uniforms(seed, env, step, PURPOSE_ACTION, 0)
    return np.sqrt(-2.0 * np.log(1.0 - u0)) * np.cos(2.0 * np.pi * u1)


def categorical_action(prob_row, u):
    """argmax(cumsum(p) > u) with the cumulative sum in float32 (distributions.categorical_sample)."""
    return int(np.argmax(np.cumsum(np.asarray(prob_row, np.float32)) > u))


def gauss_action(mean, std, z):
    return np.float32(z) * np.asarray(std, np.float32) + np.asarray(mean, np.float32)


class RunningStat(object):
    """running_stat.py:4-33 in float64."""

    def __init__(self, d, state=None):
        self.n, self.M, self.S = 0, np.zeros(d), np.zeros(d)
        if state is not None:
            self.n, self.M, self.S = int(state[0]), np.array(state[1], np.float64).reshape(d), np.array(state[2], np.float64).reshape(d)

    def push(self, x):
        x = np.asarray(x, np.float64)
        self.n += 1
        if self.n == 1:
            self.M[...] = x
            return
        old = self.M.copy()
        self.M[...] = old + (x - old) / self.n
        self.S[...] = self.S + (x - old) * (x - self.M)

    @property
    def std(self):
        return np.sqrt(self.S / (self.n - 1) if self.n > 1 else np.square(self.M))


def lockstep_zfilter(raw, lengths, state, demean=True, destd=True, clip=5.0):
    """raw: per environment an array [length_i, d] of raw observations.  Step t pushes the observations of the
    environments with length_i > t in index order, each normalised right after its own push.
    -> (filtered rows per environment, final RunningStat, RunningStat of the pushed samples alone)."""
    d = raw[0].shape[1]
    rs, pushed = RunningStat(d, state), RunningStat(d)
    out = [np.empty_like(r) for r in raw]
    for t in range(max(lengths)):
        for i, L in enumerate(lengths):
            if L > t:
                x = raw[i][t]
                rs.push(x)
                pushed.push(x)
                y = x
                if demean:
                    y = y - rs.M
                if destd:
                    y = y / (rs.std + 1e-8)
                if clip:
                    y = np.clip(y, -clip, clip)
                out[i][t] = y
    return out, rs, pushed


def lockstep_rewards(rewards, lengths, state):
    """The reward filter's statistics: step t pushes the rewards of the environments with length_i > t in index order."""
    rs, pushed = RunningStat(1, state), RunningStat(1)
    for t in range(max(lengths)):
        for i, L in enumerate(lengths):
            if L > t:
                rs.push([rewards[i][t]])
                pushed.push([rewards[i][t]])
    return rs, pushed
