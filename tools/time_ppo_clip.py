#!/usr/bin/env python
"""Time PPO with the clipped surrogate objective (ppo.PpoClipUpdater) at the sizes users run it with device
rollouts: one whole updater call (default options: 10 epochs of minibatches of 64) and the per-minibatch device step
(gather + mrl_net_ppo_clip_sgd_step), each timed with CUDA events around work that ends in a device synchronise.
A report, not a check.

  python tools/time_ppo_clip.py --out profiles/r08a_ppo_clip_timing.json

Writes one JSON with the card name and power limit read in the same run."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

CASES = [   # name, observation / action spaces, hidden sizes, timesteps
    ("pendulum_3-64-64-1_50k", 3, ("box", 1), [64, 64], 50_000),
    ("hopper_11-64-64-3_50k", 11, ("box", 3), [64, 64], 50_000),
]


def make_case(ob_dim, ac, hid, N):
    from modular_rl_b200 import agentzoo, spaces
    rng = np.random.default_rng(0)
    ob_space = spaces.Box(-np.ones(ob_dim), np.ones(ob_dim))
    ac_space = spaces.Box(-np.ones(ac[1]), np.ones(ac[1])) if ac[0] == "box" else spaces.Discrete(ac[1])
    agent = agentzoo.PpoClipAgent(ob_space, ac_space, dict(hid_sizes=hid, timestep_limit=1000))
    paths, left = [], N
    while left:
        T = min(left, 1000)
        ob = rng.standard_normal((T, ob_dim))
        prob = agent.policy._act_prob(ob)
        paths.append(dict(observation=ob, action=agent.policy.probtype.sample(prob), prob=prob,
                          advantage=rng.standard_normal(T)))
        left -= T
    return agent, paths


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=2000, help="minibatch steps per timed window")
    args = ap.parse_args()
    import torch
    from time_dp_training import card
    name, watts = card()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    report = dict(card=name, power_limit_w=watts, options=dict(clip_param=0.2, epochs=10, minibatch_size=64,
                                                              stepsize=3e-4), cases=[])
    for cname, ob_dim, ac, hid, N in CASES:
        agent, paths = make_case(ob_dim, ac, hid, N)
        up = agent.updater
        np.random.seed(0)
        up(paths)                                              # warm-up: module loads, buffer growth
        calls = []
        for _ in range(args.reps):
            a, b = ev(), ev()
            a.record()
            up(paths)
            b.record()
            torch.cuda.synchronize()
            calls.append(a.elapsed_time(b))
        # the minibatch step alone: gather from a resident device permutation + the device step, no host sync
        net, full, mb = agent.policy.net, up._full, up._mb
        perm = torch.from_numpy(np.random.permutation(N).astype(np.int32)).cuda()
        n_mb = (N + 63) // 64
        for i in range(50):
            net.ppo_clip_sgd_step(mb.gather_from(full, perm[(i % n_mb) * 64:(i % n_mb) * 64 + 64]), 0.2, 3e-4)
        torch.cuda.synchronize()
        steps = []
        for _ in range(args.reps):
            a, b = ev(), ev()
            a.record()
            for i in range(args.steps):
                j = (i % (n_mb - 1)) * 64
                net.ppo_clip_sgd_step(mb.gather_from(full, perm[j:j + 64]), 0.2, 3e-4)
            b.record()
            torch.cuda.synchronize()
            steps.append(a.elapsed_time(b) * 1e3 / args.steps)
        row = dict(case=cname, dims=[ob_dim] + hid + [ac[1]], timesteps=N, minibatches_per_call=10 * n_mb,
                   median_ms_per_call=float(np.median(calls)), spread_ms_per_call=[min(calls), max(calls)],
                   median_us_per_minibatch_step=float(np.median(steps)),
                   spread_us_per_minibatch_step=[min(steps), max(steps)], reps=args.reps)
        print(json.dumps(row), flush=True)
        report["cases"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
