"""Host side of data-parallel training (run_pg.py under torchrun): the per-iteration exchange of filter states and
episode / value-function statistics over a gloo world of 2, the rank seed streams and quotas, and the configurations
that data-parallel training rejects.  The device sums are covered by tests/dp_training_check.py on 2 GPUs."""
import itertools
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OB_DIM = 3


def _rank_paths(rank):
    """Seeded paths of one rank (different counts and lengths per rank)."""
    rng = np.random.default_rng(100 + rank)
    paths = []
    for _ in range(3 + 2 * rank):
        T = int(rng.integers(5, 40))
        paths.append(dict(observation=rng.normal(1.0 + rank, 2.0, (T, OB_DIM)), action=np.zeros(T, np.int64),
                          reward=rng.normal(0.5, 1.0, T), terminated=bool(rng.integers(2))))
    return paths


def _start_samples():
    rng = np.random.default_rng(7)
    return rng.normal(-1.0, 3.0, (57, OB_DIM)), rng.normal(0.0, 5.0, 57)


class _Agent(object):
    def __init__(self):
        from modular_rl_b200.filters import ZFilter
        self.obfilter = ZFilter((OB_DIM,), clip=5)
        self.rewfilter = ZFilter((), demean=False, clip=10)


def _vf_shard(rank, world):
    rng = np.random.default_rng(3)
    N = 1001
    y = rng.normal(2.0, 4.0, (N, 1))
    old = y + rng.normal(0.0, 1.5, (N, 1))
    new = y + rng.normal(0.0, 0.5, (N, 1))
    lo, hi = (N * rank) // world, (N * (rank + 1)) // world
    return (old, new, y), (old[lo:hi], new[lo:hi], y[lo:hi])


def _worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from modular_rl_b200 import core, parallel
    from modular_rl_b200.misc_utils import explained_variance_2d

    # filters: identical start state on every rank, then each rank pushes its own samples
    agent = _Agent()
    obs0, rew0 = _start_samples()
    for o, r in zip(obs0, rew0):
        agent.obfilter(o)
        agent.rewfilter(r)
    starts = parallel.begin_rollouts(agent)
    paths = _rank_paths(rank)
    for p in paths:
        for o, r in zip(p["observation"], p["reward"]):
            agent.obfilter(o)
            agent.rewfilter(r)
    episodes = parallel.sync_rollouts(agent, paths, starts)
    assert agent.obfilter.pushed is None and agent.rewfilter.pushed is None
    assert parallel.global_timesteps(paths) is None          # no data-parallel context in this process
    np.savez(os.path.join(tmp, "rank%d.npz" % rank),
             ob=np.concatenate([[agent.obfilter.rs.n], agent.obfilter.rs.mean, agent.obfilter.rs._S]),
             rew=np.concatenate([[agent.rewfilter.rs.n], agent.rewfilter.rs.mean.ravel(), agent.rewfilter.rs._S.ravel()]))

    # episode statistics from the gathered arrays == add_episode_stats on the union of the paths
    union = [p for r in range(world) for p in _rank_paths(r)]
    got, want = {}, {}
    core.add_episode_arrays(got, episodes["rewards"], episodes["lengths"])
    core.add_episode_stats(want, union)
    assert list(got) == list(want)
    for k in want:
        np.testing.assert_array_equal(got[k], want[k])
    assert episodes["n_total"] == sum(len(p["action"]) for p in union)

    # value-function statistics merged from shards == the single-process formulas on the whole batch
    (old, new, y), (old_s, new_s, y_s) = _vf_shard(rank, world)
    stats = parallel.regression_stats(old_s, new_s, y_s)
    want = dict(PredStdevBefore=old.std(), PredStdevAfter=new.std(), TargStdev=y.std(),
                EV_before=explained_variance_2d(old, y)[0], EV_after=explained_variance_2d(new, y)[0])
    assert list(stats) == list(want)
    for k in want:
        assert abs(stats[k] - want[k]) <= 1e-12 * max(1.0, abs(want[k])), (k, stats[k], want[k])

    # start-up check of replicated parameters
    parallel.check_replicated({"policy parameters": np.arange(5, dtype=np.float32)})
    with pytest.raises(RuntimeError, match="np.random.seed"):
        parallel.check_replicated({"policy parameters": np.arange(5, dtype=np.float32) + rank})
    dist.barrier()
    dist.destroy_process_group()


def test_filter_episode_and_vf_stats_sync_gloo_world2(tmp_path):
    from modular_rl_b200.running_stat import RunningStat
    world = 2
    port = 29500 + (os.getpid() + 1000) % 2000
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r0, r1 = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    for k in ("ob", "rew"):
        assert np.array_equal(r0[k], r1[k])                 # bit-identical on both ranks
    # one RunningStat that saw the start samples, then rank 0's, then rank 1's
    ob_rs, rew_rs = RunningStat((OB_DIM,)), RunningStat(())
    obs0, rew0 = _start_samples()
    for o, r in zip(obs0, rew0):
        ob_rs.push(o)
        rew_rs.push(r)
    for rank in range(world):
        for p in _rank_paths(rank):
            for o, r in zip(p["observation"], p["reward"]):
                ob_rs.push(o)
                rew_rs.push(r)
    for got, rs in ((r0["ob"], ob_rs), (r0["rew"], rew_rs)):
        want = np.concatenate([[rs.n], rs.mean.ravel(), rs._S.ravel()])
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)


def test_seed_streams_and_quotas():
    from modular_rl_b200.parallel import rank_quota, seed_stream
    assert list(itertools.islice(seed_stream(0, 1), 100)) == list(itertools.islice(itertools.count(), 100))
    assert list(itertools.islice(seed_stream(), 10)) == list(range(10))      # no data-parallel context
    for world in (2, 3, 8):
        seen = set()
        for rank in range(world):
            mine = set(itertools.islice(seed_stream(rank, world), 200))
            assert len(mine) == 200 and not (mine & seen)
            seen |= mine
    for n in (1, 7, 100, 999, 1000, 50000):
        for world in (1, 2, 3, 8):
            q = rank_quota(n, world)
            assert q * world >= n and (q - 1) * world < n
    assert rank_quota(100, 1) == 100


def test_rollout_quota_is_per_rank(monkeypatch):
    """get_paths under a data-parallel context collects ceil(timesteps_per_batch / world), strictly exceeded."""
    from modular_rl_b200 import core, envs, parallel

    class _Stub(object):
        stochastic = True

        def __init__(self):
            self.obfilter = self.rewfilter = lambda x: x

        def obfilt(self, ob):
            return ob

        def rewfilt(self, rew):
            return rew

        def act(self, ob):
            return int(np.random.randint(2)), {"prob": np.array([0.5, 0.5], np.float32)}

    monkeypatch.setattr(parallel, "_context", parallel.DataParallel(1, 4, 0, None, None))
    cfg = dict(parallel=0, timestep_limit=50, timesteps_per_batch=203)
    seeds = parallel.seed_stream()
    assert next(itertools.islice(parallel.seed_stream(), 1, None)) == 5      # rank 1 of 4: 1, 5, 9, ...
    paths = core.get_paths(envs.make("CartPole-v0"), _Stub(), cfg, seeds)
    total = sum(len(p["action"]) for p in paths)
    assert total > 51 and total - len(paths[-1]["action"]) <= 51


def test_out_of_scope_configurations_raise(monkeypatch):
    from modular_rl_b200 import agentzoo, envs, parallel
    import run_cem
    env = envs.make("Pendulum-v0")
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(NotImplementedError, match="PpoSgdAgent"):
        agentzoo.PpoSgdAgent(env.observation_space, env.action_space, {})
    with pytest.raises(NotImplementedError, match="do_split=1"):
        agentzoo.PpoLbfgsAgent(env.observation_space, env.action_space, {"do_split": 1})
    with pytest.raises(NotImplementedError, match="run_cem.py"):
        run_cem.main(["--env", "CartPole-v0", "--agent", "modular_rl.agentzoo.DeterministicAgent"])
    monkeypatch.setenv("WORLD_SIZE", "1")
    parallel.reject_data_parallel("anything")                                  # one process: nothing to reject
