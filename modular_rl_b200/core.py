"""Host-side mirror of the reference's core.py for the policy-update path.

Same names, arguments and error behaviour as the reference (file:line cited per item), but every
batch quantity is computed by libmrl_b200.so on the GPU: there is no Theano graph, no per-path
Python loop around the value net or the discounted scans, and no CPU fallback.

What lives here
  compute_advantage        core.py:63-105   -> one value-net forward + one segmented scan kernel
  run_policy_gradient_algorithm / rollout / do_rollouts_serial / get_paths   core.py:118-239 (callers)
  StochPolicy / StochPolicyMLP (the reference's StochPolicyKeras)            core.py:245-336
  ProbType / Categorical / DiagGauss                                         core.py:272-438
  NnRegression / NnVf / LbfgsOptimizer / EzFlat                              core.py:518-697
"""
import itertools
import time
from collections import OrderedDict, defaultdict
from importlib import import_module

import os

import numpy as np
import scipy.optimize

from . import _lib as L
from . import distributions
from . import parallel
from .device import DeviceBatch, DeviceNet, DeviceRollouts
from .misc_utils import *  # noqa: F401,F403  (the reference star-imports misc_utils too)
from .misc_utils import EzPickle, explained_variance, explained_variance_2d, update_default_config

concat = np.concatenate
floatX = "float32"          # the device computes in float32 (keras_theano_setup.py:5, SURVEY A.4)


# ================================================================
# Make agent
# ================================================================

def get_agent_cls(name):
    p, m = name.rsplit('.', 1)
    mod = import_module(p)
    return getattr(mod, m)


# ================================================================
# Stats
# ================================================================

def episode_arrays(paths):
    """-> (total reward, length) of every path."""
    reward_key = "reward_raw" if "reward_raw" in paths[0] else "reward"
    episoderewards = np.array([path[reward_key].sum() for path in paths])
    pathlengths = np.array([pathlength(path) for path in paths])
    return episoderewards, pathlengths


def add_episode_stats(stats, paths):
    add_episode_arrays(stats, *episode_arrays(paths))


def add_episode_arrays(stats, episoderewards, pathlengths):
    """add_episode_stats from the per-episode arrays (data-parallel training gathers these, not the paths)."""
    stats["EpisodeRewards"] = episoderewards
    stats["EpisodeLengths"] = pathlengths
    stats["NumEpBatch"] = len(episoderewards)
    stats["EpRewMean"] = episoderewards.mean()
    stats["EpRewSEM"] = episoderewards.std() / np.sqrt(len(episoderewards))
    stats["EpRewMax"] = episoderewards.max()
    stats["EpLenMean"] = pathlengths.mean()
    stats["EpLenMax"] = pathlengths.max()
    stats["RewPerStep"] = episoderewards.sum() / pathlengths.sum()


def add_prefixed_stats(stats, prefix, d):
    for k, v in d.items():
        stats[prefix + "_" + k] = v


# ================================================================
# Paths -> device batch
# ================================================================

class _BatchCache(object):
    """compute_advantage, baseline.fit and updater are called one after the other on the same
    `paths` list (core.py:139-159).  The observations are by far the largest upload, so the
    DeviceBatch built for a list of paths is kept until a different list shows up."""

    def __init__(self):
        self.key = None
        self.batch = None
        self.keep = None
        self.offsets = None

    def get(self, paths, timestep_limit):
        """timestep_limit=None: the caller ignores the time feature (policy nets read the first ob_dim
        columns only), so a batch cached for the same paths under ANY limit is reused - the update must not
        re-upload the observations compute_advantage / NnVf.fit already bound."""
        obs = [path["observation"] for path in paths]
        okey = (tuple(id(o) for o in obs), tuple(o.shape for o in obs))
        if timestep_limit is None:
            if self.key is not None and self.key[:2] == okey:
                return self.batch, self.offsets
            timestep_limit = 1.0
        key = okey + (float(timestep_limit),)
        if key[:2] == (self.key or (None, None))[:2] and key != self.key:
            # same observations, other limit: only the time feature / path table is rebuilt
            self.batch.set_paths(self.offsets, self.terminated, float(timestep_limit))
            self.key = key
        elif key != self.key:
            lens = np.array([len(o) for o in obs], np.int64)
            offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
            terminated = np.array([bool(path.get("terminated", True)) for path in paths], np.uint8)
            ob_no = obs[0] if len(obs) == 1 else concat(obs)
            ob_no = np.asarray(ob_no).reshape(int(offsets[-1]), -1)
            batch = self.batch
            if batch is None or batch.ob_dim != ob_no.shape[1]:
                batch = DeviceBatch(ob_no.shape[1], with_time_feature=True)
            batch.set_obs(ob_no)                     # float64 from the ZFilter is cast to float32 ONCE
            batch.set_paths(offsets, terminated, float(timestep_limit))
            self.key, self.batch, self.keep, self.offsets = key, batch, obs, offsets
            self.terminated = terminated
        return self.batch, self.offsets


_batch_cache = _BatchCache()


def batch_for_paths(paths, timestep_limit=1.0):
    """-> (DeviceBatch with observations + trajectory structure bound, offsets int64[n_paths+1]).  For this rank's
    paths of a data-parallel iteration the batch is told the timestep count of all ranks (the device sums divide
    by it)."""
    batch, offsets = _batch_cache.get(paths, None if timestep_limit is None else (timestep_limit if timestep_limit else 1.0))
    n_total = parallel.global_timesteps(paths)
    if n_total is not None:
        batch.set_global_n(n_total)
    return batch, offsets


def _split(flat, offsets):
    return [flat[offsets[i]:offsets[i + 1]] for i in range(len(offsets) - 1)]


# ================================================================
# Policy Gradients
# ================================================================

def compute_advantage(vf, paths, gamma, lam):
    """Writes path["return"], path["baseline"], path["advantage"] in place (core.py:63-105).
    return = discount(reward, gamma); delta_t = r_t + gamma*V_{t+1} - V_t with V after the last step
    = 0 if terminated else V of the last visited state; advantage = discount(delta, gamma*lam),
    then standardised over the whole batch with the population std and no epsilon."""
    limit = getattr(vf, "timestep_limit", 1.0)
    batch, offsets = batch_for_paths(paths, limit)
    if isinstance(vf, NnVf):
        base = vf.predict_batch(batch)                       # one forward over all paths
    else:                                                    # any Baseline with predict(path)
        base = concat([np.asarray(vf.predict(path)) for path in paths])
    reward = concat([np.asarray(path["reward"], np.float64) for path in paths])
    comm = parallel.context().comm if parallel.global_timesteps(paths) is not None else None
    ret, adv = batch.gae(reward, base, gamma, lam, standardize=True, comm=comm)   # comm: moments of all ranks
    for path, r, b, a in zip(paths, _split(ret, offsets), _split(base, offsets), _split(adv, offsets)):
        path["return"] = r
        path["baseline"] = b
        path["advantage"] = a


PG_OPTIONS = [
    ("timestep_limit", int, 0, "maximum length of trajectories"),
    ("n_iter", int, 200, "number of batch"),
    ("parallel", int, 0, "collect trajectories in parallel"),
    ("timesteps_per_batch", int, 100, ""),
    ("gamma", float, 0.99, "discount"),
    ("lam", float, 1.0, "lambda parameter from generalized advantage estimation"),
]


def run_policy_gradient_algorithm(env, agent, usercfg=None, callback=None):
    """rollouts -> compute_advantage -> baseline.fit -> updater (core.py:118-171, canonical order;
    the fork's TensorFlow cross-check lines are not part of the contract, SURVEY section 0)."""
    cfg = update_default_config(PG_OPTIONS, usercfg)
    cfg.update(usercfg)
    print("policy gradient config", cfg)
    if cfg["parallel"]:
        raise NotImplementedError
    tstart = time.time()
    # data-parallel training (parallel.init_data_parallel ran): each rank collects its share of the trajectories,
    # the filters and episode statistics are merged over ranks, the updates sum over ranks inside the library
    dp = parallel.context() is not None
    if dp:
        parallel.attach_agent(agent)
    seed_iter = parallel.seed_stream()           # itertools.count() in one process
    for _ in range(cfg["n_iter"]):
        starts = parallel.begin_rollouts(agent) if dp else None
        paths = get_paths(env, agent, cfg, seed_iter)
        episodes = parallel.sync_rollouts(agent, paths, starts) if dp else None
        compute_advantage(agent.baseline, paths, gamma=cfg["gamma"], lam=cfg["lam"])
        vf_stats = agent.baseline.fit(paths)
        pol_stats = agent.updater(paths)
        stats = OrderedDict()
        if dp:
            add_episode_arrays(stats, episodes["rewards"], episodes["lengths"])
        else:
            add_episode_stats(stats, paths)
        add_prefixed_stats(stats, "vf", vf_stats)
        add_prefixed_stats(stats, "pol", pol_stats)
        stats["TimeElapsed"] = time.time() - tstart
        if callback:
            callback(stats)


# Environments stepped in lockstep per rollout round (one batched device forward + one ZFilter block scan per step).
# 0 / 1 = the reference's serial rollouts.  Not an agent option - the reference's option tables stay unchanged -
# but a process setting: MRL_VEC_ENVS in the environment or run_pg.py --vec_envs.
VEC_ENVS = int(os.environ.get("MRL_VEC_ENVS", "0") or 0)
# Environments per device-resident rollout round (0: host rollouts): the whole round of a built-in environment runs in
# one kernel launch (do_rollouts_device).  Resets and action noise come from the device's Philox stream, not numpy's,
# so the numbers differ from a host run with the same seed.  MRL_DEVICE_ENVS or run_pg.py --device_envs.
DEVICE_ENVS = int(os.environ.get("MRL_DEVICE_ENVS", "0") or 0)


def get_paths(env, agent, cfg, seed_iter):
    if cfg["parallel"]:
        raise NotImplementedError
    n_timesteps = cfg["timesteps_per_batch"]
    if parallel.context() is not None:           # this rank's share of the batch
        n_timesteps = parallel.rank_quota(n_timesteps, parallel.context().world)
    if DEVICE_ENVS > 0:
        if VEC_ENVS > 0:
            raise ValueError("device rollouts (DEVICE_ENVS = %d) and host lockstep rollouts (VEC_ENVS = %d) are both set; "
                             "choose one" % (DEVICE_ENVS, VEC_ENVS))
        return do_rollouts_device(env, agent, cfg["timestep_limit"], n_timesteps, seed_iter, DEVICE_ENVS)
    if VEC_ENVS > 1:
        return do_rollouts_vectorized(env, agent, cfg["timestep_limit"], n_timesteps, seed_iter, VEC_ENVS)
    return do_rollouts_serial(env, agent, cfg["timestep_limit"], n_timesteps, seed_iter)


def _filter_block(filt, X):
    """N consecutive filt(x) calls on a block (ZFilter: one Welford scan on the device; anything else: per row)."""
    return filt.filter_batch(X) if hasattr(filt, "filter_batch") else np.stack([filt(x) for x in X])


def rollouts_vectorized(envs, agent, timestep_limit):
    """len(envs) rollouts in lockstep (SURVEY section 8f rank 1): per step ONE ZFilter block scan and ONE device
    forward for all live environments (`ZFilter.filter_batch`, `StochPolicy.act_batch`) instead of a batch-1 `act`
    per environment step (core.py:193).  Returns one path dict per environment with the keys of `rollout`.  With one
    environment the result is identical to `rollout` (same filter updates, same numpy draws); with several the running
    filter statistics see the observations in lockstep order instead of episode after episode."""
    K = len(envs)
    obs = [env.reset() for env in envs]
    data = [defaultdict(list) for _ in range(K)]
    terminated = [False] * K
    live = list(range(K))
    stochastic = getattr(agent, "stochastic", True)
    for _ in range(timestep_limit):
        if not live:
            break
        block = _filter_block(agent.obfilter, np.stack([np.asarray(obs[i], np.float64) for i in live]))
        actions, info = agent.policy.act_batch(block, stochastic=stochastic)
        rews = []
        still = []
        for j, i in enumerate(live):
            data[i]["observation"].append(block[j])
            data[i]["action"].append(actions[j])
            for (k, v) in info.items():
                data[i][k].append(v[j])
            ob, rew, done, envinfo = envs[i].step(actions[j])
            obs[i] = ob
            data[i]["reward"].append(rew)
            rews.append(rew)
            for (k, v) in envinfo.items():
                data[i][k].append(v)
            if done:
                terminated[i] = True
            else:
                still.append(i)
        _filter_block(agent.rewfilter, np.asarray(rews, np.float64))     # only advances its statistics (SURVEY A.5)
        live = still
    paths = []
    for i in range(K):
        d = {k: np.array(v) for (k, v) in data[i].items()}
        d["terminated"] = terminated[i]
        paths.append(d)
    return paths


def do_rollouts_vectorized(env, agent, timestep_limit, n_timesteps, seed_iter, n_envs):
    """Rounds of n_envs lockstep rollouts until more than n_timesteps are collected (the strict test of
    core.py:219); numpy is reseeded once per round from the same counter `do_rollouts_serial` draws from."""
    import copy
    envs = [env] + [copy.deepcopy(env) for _ in range(n_envs - 1)]
    paths = []
    timesteps_sofar = 0
    while True:
        np.random.seed(next(seed_iter))
        for path in rollouts_vectorized(envs, agent, timestep_limit):
            paths.append(path)
            timesteps_sofar += pathlength(path)
        if timesteps_sofar > n_timesteps:
            break
    return paths


def _device_filter(filt, what):
    """ZFilter -> the filter; IDENTITY -> None; anything else has no device implementation."""
    from .filters import ZFilter
    if filt is IDENTITY:
        return None
    if isinstance(filt, ZFilter):
        return filt
    raise TypeError("device rollouts support a ZFilter or IDENTITY as the %s, not %r" % (what, filt))


def check_device_rollouts(env, agent):
    """Raise, before anything runs, for what do_rollouts_device cannot run: an environment without a device
    implementation, filters other than ZFilter / IDENTITY, a policy without a DeviceNet.  -> the env's device kind."""
    from . import envs
    kind = envs.device_kind(env)
    _device_filter(agent.obfilter, "observation filter")
    _device_filter(agent.rewfilter, "reward filter")
    if not isinstance(getattr(agent.policy, "net", None), DeviceNet):
        raise TypeError("device rollouts need a policy with a DeviceNet (StochPolicyMLP); %s has none"
                        % type(agent.policy).__name__)
    return kind


_device_rollouts = {}        # (kind, n_envs, timestep_limit, device) -> DeviceRollouts: buffers kept across iterations


def _filter_arg(filt):
    return None if filt is None else (filt.rs.state(), filt.demean, filt.destd, filt.clip)


def _advance_filter(filt, state, pushed):
    """The filter takes the state after the round; a data-parallel iteration also merges the round's own samples into
    `pushed` (parallel.sync_rollouts exchanges that)."""
    filt.rs.set_state(*state)
    if filt.pushed is not None:
        filt.pushed.set_state(*parallel.merge_filter_states(filt.pushed.state(), [pushed]))


def device_paths(out, categorical):
    """Path dicts with the keys and dtypes of rollouts_vectorized from the compacted arrays of DeviceRollouts.run."""
    offsets = np.concatenate([[0], np.cumsum(out["lengths"], dtype=np.int64)])
    act = out["action"].astype(np.int64) if categorical else out["action"]
    paths = []
    for i in range(len(out["lengths"])):
        a, b = offsets[i], offsets[i + 1]
        paths.append({"observation": out["observation"][a:b], "action": act[a:b], "prob": out["prob"][a:b],
                      "reward": out["reward"][a:b], "terminated": bool(out["terminated"][i])})
    return paths


def do_rollouts_device(env, agent, timestep_limit, n_timesteps, seed_iter, n_envs):
    """do_rollouts_vectorized with each round of n_envs environments run on the device in one kernel launch: one
    next(seed_iter) per round (the Philox key of its resets and action draws), rounds until more than n_timesteps are
    collected (strict, core.py:219)."""
    kind = check_device_rollouts(env, agent)
    net = agent.policy.net
    key = (kind, int(n_envs), int(timestep_limit), net.device)
    if key not in _device_rollouts:
        _device_rollouts[key] = DeviceRollouts(env, n_envs, timestep_limit, device=net.device)
    ro = _device_rollouts[key]
    obf = _device_filter(agent.obfilter, "observation filter")
    rwf = _device_filter(agent.rewfilter, "reward filter")
    stochastic = getattr(agent, "stochastic", True)
    paths = []
    timesteps_sofar = 0
    while True:
        out = ro.run(net, next(seed_iter), stochastic, _filter_arg(obf), _filter_arg(rwf))
        if obf is not None:
            _advance_filter(obf, out["ob_state"], out["ob_pushed"])
        if rwf is not None:
            _advance_filter(rwf, out["rew_state"], out["rew_pushed"])
        paths += device_paths(out, ro.categorical)
        timesteps_sofar += len(out["reward"])
        if timesteps_sofar > n_timesteps:
            break
    return paths


def rollout(env, agent, timestep_limit):
    """Simulate the env and agent for timestep_limit steps (core.py:182-207).  The RAW reward is
    stored; rewfilt only advances its running statistics (SURVEY A.5)."""
    ob = env.reset()
    terminated = False
    data = defaultdict(list)
    for _ in range(timestep_limit):
        ob = agent.obfilt(ob)
        data["observation"].append(ob)
        action, agentinfo = agent.act(ob)
        data["action"].append(action)
        for (k, v) in agentinfo.items():
            data[k].append(v)
        ob, rew, done, envinfo = env.step(action)
        data["reward"].append(rew)
        rew = agent.rewfilt(rew)
        for (k, v) in envinfo.items():
            data[k].append(v)
        if done:
            terminated = True
            break
    data = {k: np.array(v) for (k, v) in data.items()}
    data["terminated"] = terminated
    return data


def do_rollouts_serial(env, agent, timestep_limit, n_timesteps, seed_iter):
    paths = []
    timesteps_sofar = 0
    while True:
        np.random.seed(next(seed_iter))
        path = rollout(env, agent, timestep_limit)
        paths.append(path)
        timesteps_sofar += pathlength(path)
        if timesteps_sofar > n_timesteps:        # strict, as the reference (core.py:219)
            break
    return paths


def pathlength(path):
    return len(path["action"])


def animate_rollout(env, agent, n_timesteps, delay=.01):
    ob = env.reset()
    env.render()
    for i in range(n_timesteps):
        a, _info = agent.act(ob)
        (ob, _rew, done, _info) = env.step(a)
        env.render()
        if done:
            print("terminated after %s timesteps" % i)
            break
        time.sleep(delay)


# ================================================================
# Probability types
# ================================================================

class ProbType(object):
    head = None

    def sampled_variable(self):
        raise NotImplementedError

    def prob_variable(self):
        raise NotImplementedError

    def likelihood(self, a, prob):
        raise NotImplementedError

    def loglikelihood(self, a, prob):
        raise NotImplementedError

    def kl(self, prob0, prob1):
        raise NotImplementedError

    def entropy(self, prob):
        raise NotImplementedError

    def maxprob(self, prob):
        raise NotImplementedError


class Categorical(ProbType):
    """prob row = class probabilities (core.py:339-365).  The batch reductions of likelihood / kl /
    entropy inside the updaters run in the CUDA heads; the array methods here are the same formulas for
    callers that hold explicit prob arrays."""
    head = L.CATEGORICAL

    def __init__(self, n):
        self.n = n

    def sampled_variable(self):
        return np.zeros((0,), np.int32)

    def prob_variable(self):
        return np.zeros((0, self.n), floatX)

    def likelihood(self, a, prob):
        return prob[np.arange(prob.shape[0]), np.asarray(a).astype(np.int64)]

    def loglikelihood(self, a, prob):
        return np.log(self.likelihood(a, prob))

    def kl(self, prob0, prob1):
        return (prob0 * np.log(prob0 / prob1)).sum(axis=1)

    def entropy(self, prob0):
        return - (prob0 * np.log(prob0)).sum(axis=1)

    def sample(self, prob):
        return distributions.categorical_sample(prob)

    def maxprob(self, prob):
        return prob.argmax(axis=1)


class DiagGauss(ProbType):
    """prob row = [mean (d), std (d)] (core.py:402-438)."""
    head = L.GAUSS

    def __init__(self, d):
        self.d = d

    def sampled_variable(self):
        return np.zeros((0, self.d), floatX)

    def prob_variable(self):
        return np.zeros((0, 2 * self.d), floatX)

    def loglikelihood(self, a, prob):
        mean0, std0 = prob[:, :self.d], prob[:, self.d:]
        return (- 0.5 * np.square((a - mean0) / std0).sum(axis=1) - 0.5 * np.log(2.0 * np.pi) * self.d
                - np.log(std0).sum(axis=1))

    def likelihood(self, a, prob):
        return np.exp(self.loglikelihood(a, prob))

    def kl(self, prob0, prob1):
        mean0, std0 = prob0[:, :self.d], prob0[:, self.d:]
        mean1, std1 = prob1[:, :self.d], prob1[:, self.d:]
        return (np.log(std1 / std0).sum(axis=1)
                + ((np.square(std0) + np.square(mean0 - mean1)) / (2.0 * np.square(std1))).sum(axis=1)
                - 0.5 * self.d)

    def entropy(self, prob):
        return np.log(prob[:, self.d:]).sum(axis=1) + .5 * np.log(2 * np.pi * np.e) * self.d

    def sample(self, prob):
        mean_nd, std_nd = prob[:, :self.d], prob[:, self.d:]
        return np.random.randn(prob.shape[0], self.d).astype(floatX) * std_nd + mean_nd

    def maxprob(self, prob):
        return prob[:, :self.d]


# ================================================================
# Flat parameter access
# ================================================================

class EzFlat(object):
    """get_params_flat / set_params_flat over a device-resident net (core.py:548-557).  The flat
    vector has the reference's order: per Dense layer [kernel (in,out) C-order, bias], logstd last."""

    def __init__(self, net):
        self._flat_net = net

    def set_params_flat(self, theta):
        self._flat_net.set_params(np.asarray(theta))      # cast to float32 on the device (core.py:540)

    def get_params_flat(self):
        return self._flat_net.get_params()


# ================================================================
# Stochastic policies
# ================================================================

def glorot_flat(dims, head, last_scale):
    """Keras-2.0.2 Dense defaults (glorot-uniform kernel, zero bias), last kernel scaled, logstd zeros
    (agentzoo.py:34-48, core.py:716), drawn from numpy's global RNG like Keras does."""
    chunks = []
    n = len(dims) - 1
    for l in range(n):
        lim = np.sqrt(6.0 / (dims[l] + dims[l + 1]))
        W = np.random.uniform(-lim, lim, size=(dims[l], dims[l + 1])).astype(floatX)
        if l == n - 1:
            W *= np.float32(last_scale)
        chunks += [W.ravel(), np.zeros(dims[l + 1], floatX)]
    if head == L.GAUSS:
        chunks.append(np.zeros(dims[-1], floatX))
    return concat(chunks)


class StochPolicy(object):
    @property
    def probtype(self):
        raise NotImplementedError

    def act(self, ob, stochastic=True):
        """(action, {"prob": row}) - the row becomes oldprob_np in the updaters (core.py:261-267)."""
        prob = self._act_prob(ob[None])
        if stochastic:
            return self.probtype.sample(prob)[0], {"prob": prob[0]}
        return self.probtype.maxprob(prob)[0], {"prob": prob[0]}

    def act_batch(self, ob_no, stochastic=True):
        """`act` for a block of observations (vectorised environments, SURVEY section 8f rank 1): ONE device
        forward for all rows instead of one batch-1 call per environment step (core.py:193).  Returns
        (actions [N, ...], {"prob": rows [N, K | 2d]}); row i is exactly what act(ob_no[i]) computes, the
        sampling draws come from the same numpy generator (core.py:432-435, distributions.py:3-13)."""
        prob = self._act_prob(np.asarray(ob_no))
        act = self.probtype.sample(prob) if stochastic else self.probtype.maxprob(prob)
        return act, {"prob": prob}


class StochPolicyMLP(StochPolicy, EzFlat):
    """The reference's StochPolicyKeras (core.py:296-336) with the Keras Sequential replaced by a
    device-resident MLP: Dense(h, activation) x len(hid_sizes), then Dense(d) + ConcatFixedStd
    (core.py:708-725) for Box actions or Dense(K, softmax) for Discrete ones."""

    def __init__(self, ob_dim, hid_sizes, probtype, activation="tanh", theta=None):
        self._probtype = probtype
        out = probtype.d if isinstance(probtype, DiagGauss) else probtype.n
        self.dims = [int(ob_dim)] + [int(h) for h in hid_sizes] + [int(out)]
        self.activation = activation
        self.net = DeviceNet(self.dims, probtype.head, activation)
        EzFlat.__init__(self, self.net)
        self.set_params_flat(glorot_flat(self.dims, probtype.head, 0.1) if theta is None else theta)
        self._act_batch = DeviceBatch(self.dims[0], with_time_feature=True)

    @property
    def probtype(self):
        return self._probtype

    def _act_prob(self, ob_no):
        ob_no = np.asarray(ob_no, np.float32).reshape(-1, self.dims[0])
        self._act_batch.set_obs(ob_no)
        return self.output_from_head(self.net.forward(self._act_batch))

    def output_from_head(self, out):
        """net output -> the reference's prob rows: [mean, std] or probabilities."""
        if isinstance(self._probtype, DiagGauss):
            d = self._probtype.d
            ver = self.net.theta_version          # act() runs per env step: download theta only after it changed
            if getattr(self, "_std_cache", (None, None))[0] != ver:
                self._std_cache = (ver, np.exp(self.get_params_flat()[-d:]))
            std = self._std_cache[1]
            return concat([out, np.broadcast_to(std[None, :], out.shape)], axis=1).astype(floatX)
        return out

    def get_flat(self):
        return self.get_params_flat()

    def set_from_flat(self, th):
        self.set_params_flat(th)

    def __getstate__(self):
        return dict(ob_dim=self.dims[0], hid_sizes=self.dims[1:-1], probtype=self._probtype,
                    activation=self.activation, theta=self.get_params_flat())

    def __setstate__(self, d):
        self.__init__(d["ob_dim"], d["hid_sizes"], d["probtype"], d["activation"], d["theta"])


StochPolicyKeras = StochPolicyMLP   # the name agentzoo / snapshots of the reference use


# ================================================================
# Value functions
# ================================================================

class Baseline(object):
    def fit(self, paths):
        raise NotImplementedError

    def predict(self, path):
        raise NotImplementedError


class LbfgsOptimizer(EzFlat):
    """scipy's L-BFGS-B on the host (the identical routine the reference calls, core.py:687) driving
    the device loss/gradient: every evaluation is one set_params + one fused forward/backward pass."""

    def __init__(self, net, maxiter=25, l2coeff=1e-3):
        EzFlat.__init__(self, net)
        self.net = net
        self.maxiter = maxiter
        self.l2coeff = l2coeff
        self.loss_names = ["loss", "mse", "l2"]

    def update(self, batch):
        thprev = self.get_params_flat().astype(np.float64)

        def lossandgrad(th):
            self.set_params_flat(th)
            ls, g = self.net.vf_lossgrad(batch, self.l2coeff)
            return ls[0], g

        losses_before, _ = self.net.vf_lossgrad(batch, self.l2coeff, want_grad=False)
        theta, _, opt_info = scipy.optimize.fmin_l_bfgs_b(lossandgrad, thprev, maxiter=self.maxiter)
        self.set_params_flat(theta)
        losses_after, _ = self.net.vf_lossgrad(batch, self.l2coeff, want_grad=False)
        info = OrderedDict()
        for (name, lossbefore, lossafter) in zip(self.loss_names, losses_before, losses_after):
            info[name + "_before"] = lossbefore
            info[name + "_after"] = lossafter
        self.last_opt_info = {k: v for k, v in opt_info.items() if k != "grad"}
        return info


class NnRegression(object):
    """Least-squares fit of a value MLP with target mixing (core.py:595-637):
    target = y*mixfrac + ypred_old*(1-mixfrac); loss = sum((target-pred)^2)/N + 1e-3*sum(theta^2).
    maxiter defaults to the upstream 25; the fork's HEAD has 2 (core.py:596) - pass it explicitly to
    reproduce that (SURVEY A.6)."""

    def __init__(self, net, mixfrac=1.0, maxiter=25):
        self.net = net
        self.mixfrac = mixfrac
        self.opt = LbfgsOptimizer(net, maxiter=maxiter)
        self.ez_for_net = self.opt
        self._xbatch = None

    def predict(self, x_nx):
        x_nx = np.asarray(x_nx)
        if self._xbatch is None or self._xbatch.ob_dim != x_nx.shape[1]:
            self._xbatch = DeviceBatch(x_nx.shape[1], with_time_feature=False)
        self._xbatch.set_obs(x_nx)
        return self.net.forward(self._xbatch)

    def fit(self, x_nx, ytarg_ny):
        ypredold_ny = self.predict(x_nx)                     # leaves x bound in self._xbatch
        return self._fit_bound(self._xbatch, np.asarray(ytarg_ny), ypredold_ny)

    def _fit_bound(self, batch, ytarg_ny, ypredold_ny, across_ranks=False):
        """across_ranks: `batch` is one rank's shard of a data-parallel batch; the loss and gradient already sum
        over ranks, the statistics are computed from the moments of all ranks."""
        nY = ytarg_ny.shape[1]
        target = ytarg_ny * self.mixfrac + ypredold_ny * (1 - self.mixfrac)
        batch.set_vf_target(target[:, 0])
        out = self.opt.update(batch)
        yprednew_ny = self.net.forward(batch)
        if across_ranks:
            out.update(parallel.regression_stats(ypredold_ny, yprednew_ny, ytarg_ny))
            return out
        out["PredStdevBefore"] = ypredold_ny.std()
        out["PredStdevAfter"] = yprednew_ny.std()
        out["TargStdev"] = ytarg_ny.std()
        if nY == 1:
            out["EV_before"] = explained_variance_2d(ypredold_ny, ytarg_ny)[0]
            out["EV_after"] = explained_variance_2d(yprednew_ny, ytarg_ny)[0]
        else:
            out["EV_avg"] = explained_variance(yprednew_ny.ravel(), ytarg_ny.ravel())
        return out


class NnVf(Baseline):
    """Neural value function on [observation, t/timestep_limit] (core.py:643-660)."""

    def __init__(self, net, timestep_limit, regression_params):
        self.reg = NnRegression(net, **regression_params)
        self.timestep_limit = timestep_limit

    def preproc(self, ob_no):
        ob_no = np.asarray(ob_no)
        return concat([ob_no, np.arange(len(ob_no)).reshape(-1, 1) / float(self.timestep_limit)], axis=1)

    def predict_batch(self, batch):
        """Values of every timestep of a bound batch (the time feature is built on the device)."""
        return self.reg.net.forward(batch)[:, 0]

    def predict(self, path):
        batch, _ = batch_for_paths([path], self.timestep_limit)
        return self.predict_batch(batch)

    def fit(self, paths):
        batch, _ = batch_for_paths(paths, self.timestep_limit)
        vtarg_n1 = concat([path["return"] for path in paths]).reshape(-1, 1)
        ypredold = self.reg.net.forward(batch)
        return self.reg._fit_bound(batch, vtarg_n1, ypredold, parallel.global_timesteps(paths) is not None)


def make_value_net(ob_dim, hid_sizes, activation="tanh"):
    """vfnet of agentzoo.py:53-59: input ob_dim+1 (time feature), same hidden sizes, Dense(1); the last
    kernel is NOT scaled."""
    dims = [int(ob_dim) + 1] + [int(h) for h in hid_sizes] + [1]
    net = DeviceNet(dims, L.VALUE, activation)
    net.set_params(glorot_flat(dims, L.VALUE, 1.0))
    return net


# ================================================================
# Video monitoring
# ================================================================

def VIDEO_NEVER(_):
    return False


def VIDEO_ALWAYS(_):
    return True
