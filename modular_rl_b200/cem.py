"""Noisy cross-entropy method over the flat parameter vector of a DeterministicAgent - the reference's
modular_rl/cem.py API (cem, CEM_OPTIONS, run_cem_algorithm), SURVEY section 8f rank 4.

Every population member is scored by one rollout with its theta loaded into the device-resident net
(`agent.set_from_flat`), so the per-step `act` is the same device forward the policy-gradient agents use.
The search arithmetic itself is a few numpy lines on the host, as in the reference.  With DEVICE_ENVS on, a
generation of a built-in environment is scored by one device rollout round instead (evaluate_population_device), and
with DEVICE_SEARCH on as well the search runs on the device too (_DeviceGaussianSearch)."""
from __future__ import print_function

import itertools

import numpy as np

from .core import _filter_block, rollout
from .misc_utils import update_default_config

try:
    from tabulate import tabulate
except ImportError:  # pragma: no cover
    def tabulate(rows):
        return "\n".join(" ".join("%10.4g" % v for v in r) for r in rows)


def evaluate_population(env, agent, ths, timestep_limit):
    """Total reward of one rollout per candidate theta, all candidates in lockstep: per step ONE launch evaluates every
    live member's net on its own observation (`mrl_population_forward`) - the population-batched forward of SURVEY
    section 8f rank 4; the reference scores the candidates one rollout after another (cem.py:43-44,88-91).  The
    environments are copies of `env`; the agent's filters see the observations of a step as one block."""
    import copy
    from .core import Categorical
    from .device import population_forward
    pol = agent.policy
    ths = np.asarray(ths, np.float32)
    M = ths.shape[0]
    envs = [copy.deepcopy(env) for _ in range(M)]
    obs = [e.reset() for e in envs]
    total = np.zeros(M)
    live = list(range(M))
    discrete = isinstance(pol.probtype, Categorical)
    for _ in range(timestep_limit):
        if not live:
            break
        block = _filter_block(agent.obfilter, np.stack([np.asarray(obs[i], np.float64) for i in live]))
        out = population_forward(pol.dims, pol.activation, ths[live], block)
        acts = out.argmax(axis=1) if discrete else out          # maxprob of the deterministic policy (core.py:364-365,437-438)
        rews, still = [], []
        for j, i in enumerate(live):
            ob, rew, done, _ = envs[i].step(acts[j])
            obs[i] = ob
            total[i] += rew
            rews.append(rew)
            if not done:
                still.append(i)
        _filter_block(agent.rewfilter, np.asarray(rews, np.float64))
        live = still
    return total


# Score each generation of a built-in environment with one device rollout round (evaluate_population_device) instead
# of host rollouts.  Not a CEM option - the reference's option table stays unchanged - but a process setting:
# run_cem.py --device_envs.
DEVICE_ENVS = False


def evaluate_population_device(env, agent, ths, timestep_limit, seed):
    """evaluate_population with the whole population run on the device in ONE kernel launch: environment m of the
    round acts with ths[m] (the argmax of the raw outputs / the raw output), its score is the float64 sum of its raw
    rewards in step order, and the agent's filters take the states after the round.  `seed` keys the Philox stream of
    the round's resets, so start states come from the device and not from numpy's generator (which this call never
    touches).  `ths` may be the DeviceRows of a _DeviceGaussianSearch draw, which the round reads in place.  Raises
    before any device call for an environment, filter or policy the device cannot run."""
    from .core import _advance_filter, _device_filter, _device_rollouts, _filter_arg, check_device_rollouts
    from .device import DeviceRollouts, DeviceRows
    kind = check_device_rollouts(env, agent)
    pol = agent.policy
    if not isinstance(ths, DeviceRows):
        ths = np.asarray(ths, np.float32)
    key = (kind, int(ths.shape[0]), int(timestep_limit), pol.net.device)
    if key not in _device_rollouts:
        _device_rollouts[key] = DeviceRollouts(env, ths.shape[0], timestep_limit, device=pol.net.device)
    obf = _device_filter(agent.obfilter, "observation filter")
    rwf = _device_filter(agent.rewfilter, "reward filter")
    out = _device_rollouts[key].run_population(pol.dims, pol.activation, ths, seed, _filter_arg(obf), _filter_arg(rwf))
    if obf is not None:
        _advance_filter(obf, out["ob_state"], out["ob_pushed"])
    if rwf is not None:
        _advance_filter(rwf, out["rew_state"], out["rew_pushed"])
    return out["returns"]


class _GaussianSearch(object):
    """Diagonal-Gaussian search distribution of the noisy cross-entropy method (cem.py:10-50).  `var` is the elite
    VARIANCE (the reference's `th_std`, which starts as ones * initial_std); a generation is drawn with deviation
    sqrt(var + extra_std^2 * max(1 - generation / std_decay_time, 0)).  One `np.random.randn(batch, dim)` call per
    generation keeps the reference's random stream (pinned bit-exactly by tests/golden/cem_vectors.npz)."""

    def __init__(self, mean, initial_std, extra_std, std_decay_time):
        self.mean = np.asarray(mean, np.float64)
        self.var = np.full(self.mean.size, 1.0) * initial_std
        self.extra_var = np.square(extra_std)
        self.decay = float(std_decay_time)
        self.generation = 0

    def noise_left(self):
        return max(1.0 - self.generation / self.decay, 0)

    def draw(self, count):
        self.dev = np.sqrt(self.var + self.extra_var * self.noise_left())
        return self.mean[None, :] + self.dev[None, :] * np.random.randn(count, self.mean.size)

    def refit(self, candidates, scores, keep):
        best = candidates[scores.argsort()[-keep:]]
        self.mean, self.var = best.mean(axis=0), best.var(axis=0)
        self.generation += 1


# Draw and refit each generation on the device (_DeviceGaussianSearch) instead of with numpy.  Needs DEVICE_ENVS: the
# candidates stay in device memory and only the population round reads them.  A process setting like DEVICE_ENVS:
# run_cem.py --device_search.
DEVICE_SEARCH = False


class _DeviceGaussianSearch(object):
    """_GaussianSearch with the distribution on the device (device.DeviceSearch): `draw` fills the device's candidate
    rows and returns them as DeviceRows, `refit` ranks the M scores and refits mean and variance there.  The normals of
    generation g come from the device's Philox stream keyed by seed + g, the round seed evaluate_population_device gets
    for that generation, so numpy's generator is never touched.  `mean` and `dev` are host float64 copies (the info
    dict's th and std).  The elite rule is np.argsort(scores, kind="stable")[-keep:] (ties to the higher index, NaN
    last); the host search's default argsort may pick a different member among tied scores."""

    def __init__(self, mean, initial_std, extra_std, std_decay_time, batch_size, seed, device):
        from .device import DeviceSearch
        mean = np.asarray(mean, np.float64)
        self.search = DeviceSearch(mean.size, batch_size, device)
        self.search.set_mean(mean)
        self.search.set_var(np.full(mean.size, 1.0) * initial_std)
        self.mean = mean
        self.extra_var = np.square(extra_std)
        self.decay = float(std_decay_time)
        self.seed = int(seed)
        self.generation = 0

    def noise_left(self):
        return max(1.0 - self.generation / self.decay, 0)

    def draw(self, count):
        if count != self.search.M:
            raise ValueError("the device search draws %d candidates per generation, not %d" % (self.search.M, count))
        self.dev = self.search.draw(self.seed + self.generation, self.extra_var, self.noise_left())
        return self.search.rows

    def refit(self, candidates, scores, keep):
        if keep < 0:
            raise ValueError("elite_frac is negative: round(batch_size * elite_frac) = %d elite members" % keep)
        self.search.refit(np.asarray(scores, np.float64), keep)
        self.mean = self.search.get_mean()
        self.generation += 1


def _score(f, ths, pool):
    population = getattr(f, "population", None)
    if population is not None:
        return np.asarray(population(ths))                      # all candidates in one lockstep evaluation
    return np.array([f(th) for th in ths] if pool is None else pool.map(f, ths))


def cem(f, th_mean, batch_size, n_iter, elite_frac, initial_std=1.0, extra_std=0.0, std_decay_time=1.0, pool=None,
        search=None):
    """Generator of one info dict per iteration - the reference's `cem` signature and info keys (cem.py:10-50):
    keep the round(batch_size * elite_frac) best of each generation and refit the search distribution to them.  An
    objective that has a `population` attribute is scored with one call for the whole generation.  `search`: the
    search distribution, already set up from th_mean and the std options (default: the host _GaussianSearch)."""
    if search is None:
        search = _GaussianSearch(th_mean, initial_std, extra_std, std_decay_time)
    keep = int(np.round(batch_size * elite_frac))
    for _ in range(n_iter):
        print("extra var", search.noise_left())
        ths = search.draw(batch_size)
        ys = _score(f, ths, pool)
        assert ys.ndim == 1
        search.refit(ths, ys, keep)
        yield {"ys": ys, "th": search.mean, "ymean": ys.mean(), "std": search.dev}


CEM_OPTIONS = [
    ("batch_size", int, 200, "Number of episodes per batch"),
    ("n_iter", int, 200, "Number of iterations"),
    ("elite_frac", float, 0.2, "fraction of parameter settings used to fit pop"),
    ("initial_std", float, 1.0, "initial standard deviation for parameters"),
    ("extra_std", float, 0.0, "extra stdev added"),
    ("std_decay_time", float, -1.0, "number of timesteps that extra stdev decays over. negative => n_iter/2"),
    ("timestep_limit", int, 0, "maximum length of trajectories"),
    ("parallel", int, 0, "collect trajectories in parallel"),
]


def run_cem_algorithm(env, agent, usercfg=None, callback=None):
    """cem.py:63-98.  `parallel=1`: the reference forks a process pool around a CPU Theano function (every worker with
    its own copy of the agent and its filters); a forked child cannot share this process's CUDA context, so here
    parallel=1 scores the whole population in lockstep with one population-batched device forward per environment step
    (`evaluate_population`).  parallel=0 scores one candidate after another as cem.py:43 does.

    DEVICE_ENVS on (the built-in environments of envs.py only): each generation is scored by one device rollout round
    (`evaluate_population_device`), its Philox seed a counter started from cfg["seed"], one value per generation.
    The host paths draw the environments' resets from numpy's global generator; the device path does not touch it,
    so the search's own randn calls are its only numpy draws.  Start states, scores and therefore later generations
    differ from a host run with the same seed (as with run_pg.py --device_envs); equal seeds give identical device
    runs.

    DEVICE_SEARCH on (needs DEVICE_ENVS): the candidates are drawn and the distribution refitted on the device
    (_DeviceGaussianSearch), the draws of generation g keyed by the same round seed as its rollouts.  numpy's
    generator is not used at all, and the numbers differ from a host search."""
    cfg = update_default_config(CEM_OPTIONS, usercfg)
    if cfg["std_decay_time"] < 0:
        cfg["std_decay_time"] = cfg["n_iter"] / 2
    if usercfg:
        cfg.update(usercfg)
    print("cem config", {k: cfg[k] for (k, _, _, _) in CEM_OPTIONS})
    if cfg["parallel"] and DEVICE_ENVS:
        raise ValueError("parallel=1 (host population path) and DEVICE_ENVS select different scoring paths; choose one")
    if cfg["parallel"]:
        print("parallel=1: population-batched evaluation (one device forward per step for all candidates)")
    if DEVICE_SEARCH and not DEVICE_ENVS:
        raise ValueError("DEVICE_SEARCH draws the candidates into device memory that only DEVICE_ENVS rounds read; "
                         "set both")
    if DEVICE_SEARCH and cfg["elite_frac"] < 0:
        raise ValueError("elite_frac = %g is negative" % cfg["elite_frac"])
    if DEVICE_ENVS:
        print("device_envs: one device rollout round per generation")
    if DEVICE_SEARCH:
        print("device_search: candidates drawn and refitted on the device")
    timestep_limit = cfg["timestep_limit"]

    def objective(th):
        agent.set_from_flat(th)
        path = rollout(env, agent, timestep_limit)
        return path["reward"].sum()
    if cfg["parallel"]:
        objective.population = lambda ths: evaluate_population(env, agent, ths, timestep_limit)
    if DEVICE_ENVS:
        seeds = itertools.count(int(cfg.get("seed", 0)))
        objective.population = lambda ths: evaluate_population_device(env, agent, ths, timestep_limit, next(seeds))

    th_mean = agent.get_flat()
    search = None
    if DEVICE_SEARCH:
        search = _DeviceGaussianSearch(th_mean, cfg["initial_std"], cfg["extra_std"], cfg["std_decay_time"],
                                       cfg["batch_size"], int(cfg.get("seed", 0)), agent.policy.net.device)
    for info in cem(objective, th_mean, cfg["batch_size"], cfg["n_iter"], cfg["elite_frac"],
                    cfg["initial_std"], cfg["extra_std"], cfg["std_decay_time"], search=search):
        if callback is not None:
            callback(info)
        ps = np.linspace(0, 100, 5)
        print(tabulate([ps, np.percentile(info["ys"].ravel(), ps), np.percentile(info["std"].ravel(), ps)]))
        agent.set_from_flat(info["th"])
