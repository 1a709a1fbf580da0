#!/usr/bin/env python
"""Cross-entropy-method driver with the reference's run_cem.py command line (GENERAL_OPTIONS, --env, --agent, --plot,
the agent's own options, CEM_OPTIONS - run_cem.py:13-30).  Candidates are scored through the device-resident
deterministic policy; with --parallel 1 the whole population is scored in lockstep by one population-batched forward
per environment step; with --device_envs (environments with a device implementation) each generation is one device
rollout round, and with --device_search as well the candidates are drawn and the search distribution refitted on the
device.

  python run_cem.py --env CartPole-v0 --agent modular_rl.agentzoo.DeterministicAgent --n_iter 10 --batch_size 40
"""
import argparse
import os
import pickle
import shutil
import sys

import numpy as np

import modular_rl as mrl
from modular_rl_b200 import parallel
from modular_rl_b200.envs import make


def _table(pairs):
    try:
        from tabulate import tabulate
        return tabulate(pairs)
    except ImportError:  # pragma: no cover
        return "\n".join("%-24s %s" % kv for kv in pairs)


def parse_cli(argv):
    """Two-stage parse as in the reference: the agent class named by --agent contributes its own options."""
    ap = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    mrl.update_argument_parser(ap, mrl.GENERAL_OPTIONS)
    ap.add_argument("--env", required=True)
    ap.add_argument("--agent", required=True)
    ap.add_argument("--plot", action="store_true")
    ap.add_argument("--device_envs", action="store_true",
                    help="score each generation in one GPU rollout round, one environment per candidate (the "
                         "built-in environments, and user environments whose class has an envs.DeviceEnv); resets "
                         "come from the device's Philox stream, so results differ from a host run with the same --seed")
    ap.add_argument("--device_search", action="store_true",
                    help="with --device_envs: draw each generation's candidates and refit the search distribution on "
                         "the GPU; the draws come from the device's Philox stream, not numpy's, so results differ "
                         "from a run without it")
    first, _ = ap.parse_known_args([a for a in argv if a not in ("-h", "--help")])
    agent_cls = mrl.get_agent_cls(first.agent)
    mrl.update_argument_parser(ap, agent_cls.options)
    mrl.update_argument_parser(ap, mrl.CEM_OPTIONS)
    args = ap.parse_args(argv)
    if args.device_search:
        if not args.device_envs:
            ap.error("--device_search needs --device_envs: only a device rollout round reads candidates in device memory")
        if args.elite_frac < 0:
            ap.error("--device_search: --elite_frac is %g; it must not be negative" % args.elite_frac)
    if args.device_envs:
        from modular_rl_b200.device import DeviceRollouts
        from modular_rl_b200.envs import device_kind
        if args.parallel:
            ap.error("--device_envs and --parallel 1 select different population paths; give one")
        if args.batch_size > DeviceRollouts.max_envs():
            ap.error("--device_envs runs a generation in one round of at most %d environments; --batch_size is %d"
                     % (DeviceRollouts.max_envs(), args.batch_size))
        try:
            device_kind(args.env)
        except ValueError as e:
            ap.error(str(e))
    return args, agent_cls


class IterationLog(object):
    """Per-iteration callback of run_cem_algorithm: diagnostics to hdf5, a table of the scalar stats, snapshots."""

    def __init__(self, args, env, agent, results_dir, hdf=None, diagnostics=None):
        self.args, self.env, self.agent, self.results_dir = args, env, agent, results_dir
        self.hdf, self.diagnostics = hdf, diagnostics
        self.done = 0

    def snapshot_due(self):
        every = self.args.snapshot_every
        return bool(every) and (self.done % every == 0 or self.done == self.args.n_iter)

    def __call__(self, stats):
        if self.diagnostics is not None:
            for key, val in stats.items():
                self.diagnostics[key].append(val)
        if self.args.plot:
            mrl.animate_rollout(self.env, self.agent, min(500, self.args.timestep_limit))
        print("*********** Iteration %i ****************" % self.done)
        print(_table([(k, v) for k, v in stats.items() if np.asarray(v).size == 1]))
        self.done += 1
        if self.snapshot_due():
            self.agent.set_from_flat(stats["th"])
            if self.hdf is not None:
                self.hdf["/agent_snapshots/%0.4i" % self.done] = np.array(pickle.dumps(self.agent, -1))
            else:
                mrl.save_agent_snapshot(self.agent, self.results_dir, self.done, env_id=self.env.spec.id)


def main(argv=None):
    parallel.reject_data_parallel("run_cem.py")
    args, agent_cls = parse_cli(sys.argv[1:] if argv is None else argv)
    env = make(args.env)
    # a snapshot may live in the results directory of the previous run: read it before that directory is cleared
    restored = mrl.load_agent_snapshot(args.load_snapshot) if args.load_snapshot else None
    results_dir = args.outfile + ".dir"
    shutil.rmtree(results_dir, ignore_errors=True)
    os.makedirs(results_dir)
    if args.timestep_limit == 0:
        args.timestep_limit = env.spec.max_episode_steps
    np.random.seed(args.seed)
    cfg = vars(args)
    agent = restored if restored is not None else agent_cls(env.observation_space, env.action_space, cfg)
    if args.device_envs:
        from modular_rl_b200 import cem, core
        core.check_device_rollouts(env, agent)     # an unsupported filter / policy fails before any rollout
        cem.DEVICE_ENVS = True
        cem.DEVICE_SEARCH = args.device_search
    hdf, diagnostics = mrl.prepare_h5_file(args) if args.use_hdf else (None, None)
    mrl.run_cem_algorithm(env, agent, callback=IterationLog(args, env, agent, results_dir, hdf, diagnostics), usercfg=cfg)
    if hdf is not None:
        hdf["env_id"] = env.spec.id
    env.close()


if __name__ == "__main__":
    main()
