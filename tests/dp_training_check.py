#!/usr/bin/env python
"""Data-parallel training check, run under torchrun with one rank per GPU (2 or more; 1 rank drives the same code
paths without a peer):

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
      --master-port 29521 tests/dp_training_check.py

Three iterations of run_policy_gradient_algorithm for TrpoAgent on CartPole-v0 and PpoLbfgsAgent on Pendulum-v0.
After every iteration the policy parameters, the value-function parameters and both filter states must be
bit-identical on every rank.  In the last iteration each rank keeps its paths and the pickled agent from before the
update; rank 0 then replays compute_advantage + baseline.fit + updater in one process on the paths of all ranks,
and the statistics and new parameters must agree within 1e-5 relative (only the order of the sums differs).
MRL_NCCL_ONLY=1 selects NCCL instead of the peer-memory transport."""
import os
import pickle
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_ITER = 3
TOL = 1e-5


def _rel(a, b, floor=1e-2):
    """Relative difference; values below `floor` in magnitude (a surrogate or KL that is zero up to rounding at the
    old parameters) are compared against the floor."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), floor))


def _replicated_state(agent):
    parts = [agent.policy.get_flat(), agent.baseline.reg.net.get_params()]
    for f in (agent.obfilter, agent.rewfilter):
        n, M, S = f.rs.state()
        parts += [np.array([n]), M, S]
    return b"".join(np.ascontiguousarray(p).tobytes() for p in parts)


def run_case(name, env_id, cfg_overrides, vec_envs, failures):
    from modular_rl_b200 import agentzoo, core, parallel
    from modular_rl_b200.envs import make
    from modular_rl_b200.misc_utils import update_default_config
    ctx = parallel.context()
    env = make(env_id)
    agent_cls = getattr(agentzoo, name)
    usercfg = dict(timestep_limit=env.spec.max_episode_steps, n_iter=N_ITER, timesteps_per_batch=3000, **cfg_overrides)
    cfg = update_default_config(agent_cls.options, usercfg)
    np.random.seed(0)
    agent = agent_cls(env.observation_space, env.action_space, cfg)
    core.VEC_ENVS = vec_envs

    it = [0]
    kept = {}
    compute_advantage = core.compute_advantage

    def keep_last(vf, paths, gamma, lam):
        if it[0] == N_ITER - 1:
            kept["agent"] = pickle.dumps(agent, -1)
            kept["kl_coeff"] = getattr(agent.updater, "kl_coeff", None)
            kept["paths"] = [dict(p) for p in paths]
        return compute_advantage(vf, paths, gamma, lam)

    def callback(stats):
        it[0] += 1
        states = parallel.all_gather(_replicated_state(agent))
        if any(s != states[0] for s in states):
            failures.append("%s: ranks differ after iteration %d" % (name, it[0]))
        kept["stats"] = stats

    core.compute_advantage = keep_last
    try:
        core.run_policy_gradient_algorithm(env, agent, usercfg=cfg, callback=callback)
    finally:
        core.compute_advantage = compute_advantage
    if it[0] != N_ITER:
        failures.append("%s: %d iterations" % (name, it[0]))

    all_paths = parallel.all_gather(kept["paths"])
    if ctx.rank == 0:
        # one process, no communicator, no sharding: the same update on the concatenated paths
        parallel._context = None
        try:
            ref = pickle.loads(kept["agent"])
            if kept["kl_coeff"] is not None:
                ref.updater.kl_coeff = kept["kl_coeff"]
            paths = [p for r in all_paths for p in r]
            core.compute_advantage(ref.baseline, paths, gamma=cfg["gamma"], lam=cfg["lam"])
            vf_stats = ref.baseline.fit(paths)
            pol_stats = ref.updater(paths)
        finally:
            parallel._context = ctx
        got = kept["stats"]
        checks = {}
        for prefix, want in (("vf", vf_stats), ("pol", pol_stats)):
            for k, v in want.items():
                if k.endswith("_change"):          # a difference of two checked values
                    continue
                checks["%s_%s" % (prefix, k)] = _rel(got["%s_%s" % (prefix, k)], v)
        checks["theta"] = _rel(agent.policy.get_flat(), ref.policy.get_flat())
        checks["vf_theta"] = _rel(agent.baseline.reg.net.get_params(), ref.baseline.reg.net.get_params())
        checks["NumEpBatch"] = abs(got["NumEpBatch"] - len(paths))
        bad = {k: v for k, v in checks.items() if not v <= TOL}
        print(name, env_id, "ranks:", ctx.world, "timesteps:", sum(len(p["action"]) for p in paths),
              "max rel. diff to the one-process replay: %.3g" % max(checks.values()), flush=True)
        if bad:
            failures.append("%s: differs from the one-process replay: %s" % (name, bad))
    parallel.barrier()


def main():
    from modular_rl_b200 import parallel
    ctx = parallel.init_data_parallel()
    if ctx.rank == 0:
        print("transport:", "nvlink peer-memory push" if ctx.comm.p2p else "nccl", flush=True)
    failures = []
    run_case("TrpoAgent", "CartPole-v0", dict(cg_damping=0.1), 0, failures)            # serial rollouts
    run_case("PpoLbfgsAgent", "Pendulum-v0", {}, 4, failures)                          # 4 lockstep environments
    failures = [f for r in parallel.all_gather(failures) for f in r]
    parallel.shutdown_data_parallel()
    if failures:
        print("FAIL", failures, flush=True)
        sys.exit(1)
    if ctx.rank == 0:
        print("DP_TRAINING_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
