#!/usr/bin/env python
"""This script runs a policy gradient algorithm - same flags as the reference's run_pg.py
(GENERAL_OPTIONS + --env --agent --plot + the agent's own option table, parsed in two passes,
run_pg.py:79-102), with the policy update executed by the B200 library.

  python run_pg.py --env CartPole-v0 --agent modular_rl.agentzoo.TrpoAgent --n_iter 20 --timesteps_per_batch 5000

Under torchrun (WORLD_SIZE > 1) it trains data-parallel, one process per GPU: every rank collects its share of
--timesteps_per_batch and each update runs over the trajectories of all ranks.  Only rank 0 prints and writes
results and snapshots.

  torchrun --nproc-per-node 8 run_pg.py --env Pendulum-v0 --agent modular_rl.agentzoo.TrpoAgent --vec_envs 16 ...
"""
import argparse
import os
import pickle
import shutil
import sys

import numpy as np

from modular_rl import *  # noqa: F401,F403
from modular_rl_b200 import parallel
from modular_rl_b200.envs import make

try:
    from tabulate import tabulate
except ImportError:  # pragma: no cover
    def tabulate(rows):
        return "\n".join("%-24s %s" % (k, v) for k, v in rows)


def main():
    parser = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    update_argument_parser(parser, GENERAL_OPTIONS)
    parser.add_argument("--env", default="CartPole-v0")
    parser.add_argument("--agent", default="modular_rl.agentzoo.TrpoAgent")
    parser.add_argument("--plot", action="store_true")
    parser.add_argument("--vec_envs", type=int, default=0,
                        help="environments stepped in lockstep with one batched device forward per step "
                             "(0: serial rollouts as the reference); not an agent option")
    parser.add_argument("--device_envs", type=int, default=0,
                        help="environments per rollout round run on the GPU in one kernel launch (the built-in "
                             "environments, and user environments whose class has an envs.DeviceEnv, e.g. --env "
                             "examples.point_mass:PointMass-v0; 0: host rollouts); resets and action noise come from "
                             "the device's Philox stream, so results differ from a host run with the same --seed")
    args, _ = parser.parse_known_args([arg for arg in sys.argv[1:] if arg not in ('-h', '--help')])
    if args.device_envs and args.vec_envs:
        parser.error("--device_envs and --vec_envs select different rollout paths; give one")
    if args.device_envs < 0:
        parser.error("--device_envs must be >= 0")
    dp = parallel.init_data_parallel() if parallel.launched_data_parallel() else None
    root = parallel.is_root()
    if not root:
        sys.stdout = open(os.devnull, "w")          # the updaters' and the loop's lines come from rank 0 only
    env = make(args.env)
    env_spec = env.spec
    # read the snapshot before the results directory of a previous run (which may hold it) is cleared
    snapshot_agent = load_agent_snapshot(args.load_snapshot) if args.load_snapshot else None
    parallel.barrier()                               # every rank has read it before rank 0 clears the directory
    mondir = args.outfile + ".dir"
    if root:
        if os.path.exists(mondir):
            shutil.rmtree(mondir)
        os.makedirs(mondir)
    agent_ctor = get_agent_cls(args.agent)
    update_argument_parser(parser, agent_ctor.options)
    args = parser.parse_args()
    if args.timestep_limit == 0:
        args.timestep_limit = env_spec.max_episode_steps
    cfg = args.__dict__
    from modular_rl_b200 import core as _core
    if args.vec_envs > 1:
        _core.VEC_ENVS = args.vec_envs
    if args.device_envs:
        _core.DEVICE_ENVS = args.device_envs
    np.random.seed(args.seed)
    if args.load_snapshot:
        # the reference declares the flag (misc_utils.py:102) without reading it; here it resumes from a
        # pickled agent (.pkl / directory written below, or an hdf5 results file as sim_agent.py:41-52 reads)
        agent = snapshot_agent
        assert isinstance(agent, agent_ctor), "snapshot holds a %s" % type(agent).__name__
    else:
        agent = agent_ctor(env.observation_space, env.action_space, cfg)
    if args.device_envs:
        _core.check_device_rollouts(env, agent)     # an unsupported env / filter / policy fails before any rollout
    if args.use_hdf and root:
        hdf, diagnostics = prepare_h5_file(args)

    counter = [0]

    def callback(stats):
        counter[0] += 1
        print("*********** Iteration %i ****************" % counter[0])
        print(tabulate([(k, v) for k, v in stats.items() if np.asarray(v).size == 1]))
        if args.use_hdf:
            for (stat, val) in stats.items():
                if np.asarray(val).ndim == 0:
                    diagnostics[stat].append(val)
                else:
                    assert val.ndim == 1
                    diagnostics[stat].extend(val)
            if args.snapshot_every and ((counter[0] % args.snapshot_every == 0) or (counter[0] == args.n_iter)):
                hdf['/agent_snapshots/%0.4i' % counter[0]] = np.array(pickle.dumps(agent, -1))
        elif args.snapshot_every and ((counter[0] % args.snapshot_every == 0) or (counter[0] == args.n_iter)):
            save_agent_snapshot(agent, mondir, counter[0], env_id=env_spec.id)      # same bytes, one file per snapshot
        if args.plot:
            animate_rollout(env, agent, min(500, args.timestep_limit))

    run_policy_gradient_algorithm(env, agent, callback=callback if root else None, usercfg=cfg)

    if args.use_hdf and root:
        hdf['env_id'] = env_spec.id
    env.close()
    if dp is not None:
        parallel.shutdown_data_parallel()


if __name__ == "__main__":
    main()
