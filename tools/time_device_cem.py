#!/usr/bin/env python
"""Wall time per cross-entropy-method generation (cem.run_cem_algorithm) with the population scored on the host one
candidate after another (parallel=0), on the host in lockstep with one population forward per step (parallel=1), and
in one device rollout round (cem.DEVICE_ENVS, run_cem.py --device_envs), the last also with the search drawn and
refitted on the device (cem.DEVICE_SEARCH, run_cem.py --device_search).  DeterministicAgent, hid_sizes 64,64, filters
on, the environment's own timestep limit (200 for both).  For the device paths the rollout kernel's time per generation
comes from the library's CUDA-event profiler (kind "rollout") in a second, profiled run, as does the time of the
search kernels (kind "cem_search": the draw, the rank and the refit) with --device_search, and is also given per step of
the round (the longest episode's length, plus the final scan).  The host paths are timed at the smallest batch size
only unless --host_sizes says otherwise: at 200 candidates a parallel=0 generation already takes seconds, and both
host paths grow linearly with the population.  Medians are over the generations after the first (a warm-up).
A report, not a check.

  python tools/time_device_cem.py --out device_cem_timing.json

The card name and power limit are read in the same call and stored next to the times."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def generations(env_id, path, batch_size, n_iter, profile=False):
    """Seconds per generation (all n_iter) and, for the device path, the kernel's (ms, launches, steps per round)."""
    from modular_rl_b200 import _lib as L, agentzoo, cem, device
    from modular_rl_b200.envs import make
    lib = L.lib()
    env = make(env_id)
    np.random.seed(0)
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[64, 64], filter=1))
    steps = []
    orig = device.DeviceRollouts.run_population

    def run_population(self, *a, **k):
        out = orig(self, *a, **k)
        steps.append(int(out["lengths"].max()) + 1)
        return out
    device.DeviceRollouts.run_population = run_population
    cem.DEVICE_ENVS = path in ("device", "device_search")
    cem.DEVICE_SEARCH = path == "device_search"
    stamps = [time.perf_counter()]

    def callback(info):
        stamps.append(time.perf_counter())
        if profile and len(stamps) == 2:          # kernel times from generation 2 on (the first loads modules)
            lib.mrl_profile_enable(1)
    try:
        cem.run_cem_algorithm(env, agent, dict(batch_size=batch_size, n_iter=n_iter, parallel=int(path == "parallel1"),
                                               timestep_limit=env.spec.max_episode_steps, seed=0), callback=callback)
    finally:
        cem.DEVICE_ENVS = cem.DEVICE_SEARCH = False
        device.DeviceRollouts.run_population = orig
    kern = None
    if profile:
        nk = lib.mrl_profile_kinds()
        pms, pcnt = (C.c_double * nk)(), (C.c_longlong * nk)()
        L.check(lib.mrl_profile_read(pms, pcnt))
        lib.mrl_profile_enable(0)
        byname = {lib.mrl_profile_kind_name(k).decode(): (pms[k], pcnt[k]) for k in range(nk)}
        kern = byname["rollout"] + (steps[1:], byname["cem_search"])
    return list(np.diff(stamps)), kern


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--envs", default="CartPole-v0,Pendulum-v0")
    ap.add_argument("--sizes", default="200,1000,4096")
    ap.add_argument("--host_sizes", default="200", help="batch sizes at which the two host paths are timed")
    ap.add_argument("--n_iter", type=int, default=6, help="device path; the first generation is a warm-up")
    ap.add_argument("--host_n_iter", type=int, default=3)
    args = ap.parse_args()

    from time_dp_training import card
    name, watts = card()
    report = dict(card=name, power_limit_w=watts, agent="DeterministicAgent", hid_sizes=[64, 64], filter=1,
                  summary="median seconds per generation over generations 2..n_iter; kernel: CUDA events, profiled run",
                  runs=[])
    host_sizes = {int(s) for s in args.host_sizes.split(",") if s}
    for env_id in args.envs.split(","):
        for size in (int(s) for s in args.sizes.split(",")):
            for path in ("parallel0", "parallel1", "device", "device_search"):
                if path.startswith("parallel") and size not in host_sizes:
                    continue
                n_iter = args.host_n_iter if path.startswith("parallel") else args.n_iter
                secs, _ = generations(env_id, path, size, n_iter)
                run = dict(env=env_id, batch_size=size, path=path, generations_timed=len(secs) - 1,
                           s_per_generation=float(np.median(secs[1:])))
                if not path.startswith("parallel"):
                    _, (ms, cnt, steps, (sms, _)) = generations(env_id, path, size, n_iter, profile=True)
                    run.update(kernel_ms_per_generation=ms / cnt, launches_timed=cnt,
                               steps_per_round=float(np.mean(steps)),
                               kernel_us_per_step=1e3 * ms / float(np.sum(steps)))
                    if path == "device_search":
                        run.update(search_kernels_ms_per_generation=sms / cnt)
                report["runs"].append(run)
                print(json.dumps(run), flush=True)
                with open(args.out, "w") as f:          # after every run: a later failure keeps what was measured
                    json.dump(report, f, indent=1)
    print(json.dumps(dict(card=name, power_limit_w=watts)), flush=True)


if __name__ == "__main__":
    main()
