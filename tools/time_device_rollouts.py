#!/usr/bin/env python
"""Wall time of run_pg.py training iterations with host lockstep rollouts (--vec_envs 16) against device-resident
rollouts (--device_envs 256, 1024, 4096), split into rollouts, advantage + value-function fit and policy update, plus
the rollout kernel's time per round from CUDA events (the library's profiler, kind "rollout").  One process per
configuration; the medians are over iterations 2..n_iter (the first is a warm-up).  A report, not a check.

  python tools/time_device_rollouts.py --out device_rollouts_timing.json      # Pendulum-v0, TrpoAgent, 50 000 steps

The card name and power limit are read in the same call and stored next to the times."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def worker(args, run_pg_argv):
    import run_pg
    from modular_rl_b200 import _lib as L, core, ppo, trpo

    lib = L.lib()
    iters = []

    def timed(phase, fn, starts_iteration=False):
        def wrapped(*a, **k):
            if starts_iteration:
                if len(iters) == 1:              # kernel times from iteration 2 on (the first launch loads modules)
                    lib.mrl_profile_enable(1)
                iters.append(dict(rollouts=0.0, advantage_vf=0.0, update=0.0, t0=time.perf_counter()))
            t = time.perf_counter()
            out = fn(*a, **k)
            now = time.perf_counter()
            iters[-1][phase] += now - t
            iters[-1]["total"] = now - iters[-1]["t0"]
            return out
        return wrapped

    core.get_paths = timed("rollouts", core.get_paths, starts_iteration=True)
    core.compute_advantage = timed("advantage_vf", core.compute_advantage)
    core.NnVf.fit = timed("advantage_vf", core.NnVf.fit)
    trpo.TrpoUpdater.__call__ = timed("update", trpo.TrpoUpdater.__call__)
    ppo.PpoLbfgsUpdater.__call__ = timed("update", ppo.PpoLbfgsUpdater.__call__)
    sys.argv = ["run_pg.py"] + run_pg_argv
    run_pg.main()
    nk = lib.mrl_profile_kinds()
    pms, pcnt = (C.c_double * nk)(), (C.c_longlong * nk)()
    L.check(lib.mrl_profile_read(pms, pcnt))
    lib.mrl_profile_enable(0)
    kern = {lib.mrl_profile_kind_name(k).decode(): (pms[k], pcnt[k]) for k in range(nk)}
    ms, cnt = kern.get("rollout", (0.0, 0))
    with open(args.worker_out, "w") as f:
        json.dump(dict(iterations=[{k: v for k, v in it.items() if k != "t0"} for it in iters],
                       rollout_kernel_ms_per_round=(ms / cnt) if cnt else None, rollout_rounds_timed=cnt), f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--env", default="Pendulum-v0")
    ap.add_argument("--agent", default="modular_rl.agentzoo.TrpoAgent")
    ap.add_argument("--timesteps_per_batch", type=int, default=50000)
    ap.add_argument("--vec_envs", type=int, default=16)
    ap.add_argument("--device_envs", default="256,1024,4096")
    ap.add_argument("--n_iter", type=int, default=4, help="the first iteration is a warm-up and not summarised")
    ap.add_argument("--timeout", type=int, default=1200)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--worker_out")
    ap.add_argument("--rollout_flag", default="")
    args = ap.parse_args()

    with tempfile.TemporaryDirectory() as tmp:
        base = ["--env", args.env, "--agent", args.agent, "--timesteps_per_batch", str(args.timesteps_per_batch),
                "--n_iter", str(args.n_iter), "--cg_damping", "0.1", "--outfile", os.path.join(tmp, "run.h5")]
        if args.worker:
            return worker(args, base + args.rollout_flag.split())

        from time_dp_training import card
        name, watts = card()
        report = dict(card=name, power_limit_w=watts, env=args.env, agent=args.agent,
                      timesteps_per_batch=args.timesteps_per_batch, n_iter=args.n_iter,
                      summary="median over iterations 2..%d, seconds (kernel: ms per round)" % args.n_iter, runs=[])
        configs = [("--vec_envs %d" % args.vec_envs)] + ["--device_envs %s" % n for n in args.device_envs.split(",")]
        for flag in configs:
            wout = os.path.join(tmp, "w.json")
            cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--worker_out", wout, "--out", args.out,
                   "--env", args.env, "--agent", args.agent, "--timesteps_per_batch", str(args.timesteps_per_batch),
                   "--n_iter", str(args.n_iter), "--rollout_flag=" + flag]
            p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=args.timeout)
            if p.returncode != 0:
                report["runs"].append(dict(config=flag, result="failed", log=(p.stdout + p.stderr)[-3000:]))
                continue
            w = json.load(open(wout))
            its = w["iterations"][1:]
            med = {k: float(np.median([it[k] for it in its])) for k in ("rollouts", "advantage_vf", "update", "total")}
            report["runs"].append(dict(config=flag, rollout_kernel_ms_per_round=w["rollout_kernel_ms_per_round"],
                                       rollout_rounds_timed=w["rollout_rounds_timed"], **med))
            print(json.dumps(report["runs"][-1]), flush=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
        print(json.dumps(dict(card=name, power_limit_w=watts)), flush=True)


if __name__ == "__main__":
    main()
