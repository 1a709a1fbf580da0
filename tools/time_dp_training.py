#!/usr/bin/env python
"""Wall time of whole run_pg.py training iterations at 1, 2 and 8 ranks (one per GPU, torchrun), split into
rollouts (including the wait for the other ranks' filter states), advantage + value-function fit, and policy
update.  A report, not a check: rank counts above the number of visible GPUs are recorded as "not measured".

  python tools/time_dp_training.py --out dp_timing.json            # Pendulum-v0, TrpoAgent, --vec_envs 16

The card name and power limit are read in the same call and stored next to the times."""
import argparse
import json
import os
import socket
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    """(name, power limit in W) of GPU 0, or (None, None)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        name = pynvml.nvmlDeviceGetName(h)
        return (name.decode() if isinstance(name, bytes) else name), pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception:
        pass
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
        name, watts = [s.strip() for s in line.split(",")]
        return name, float(watts)
    except Exception:
        return None, None


def worker(args, run_pg_argv):
    """One rank: run_pg.main() with its phases timed on the host (each phase ends in a device synchronisation:
    the rollouts read actions back, the fit and the update return host statistics)."""
    import run_pg
    from modular_rl_b200 import core, parallel, ppo, trpo

    iters = []

    def timed(phase, fn, starts_iteration=False):
        def wrapped(*a, **k):
            if starts_iteration:
                iters.append(dict(rollouts=0.0, advantage_vf=0.0, update=0.0, t0=time.perf_counter()))
            t = time.perf_counter()
            out = fn(*a, **k)
            now = time.perf_counter()
            iters[-1][phase] += now - t
            iters[-1]["total"] = now - iters[-1]["t0"]
            return out
        return wrapped

    core.get_paths = timed("rollouts", core.get_paths, starts_iteration=True)
    parallel.sync_rollouts = timed("rollouts", parallel.sync_rollouts)
    core.compute_advantage = timed("advantage_vf", core.compute_advantage)
    core.NnVf.fit = timed("advantage_vf", core.NnVf.fit)
    trpo.TrpoUpdater.__call__ = timed("update", trpo.TrpoUpdater.__call__)
    ppo.PpoLbfgsUpdater.__call__ = timed("update", ppo.PpoLbfgsUpdater.__call__)

    sys.argv = ["run_pg.py"] + run_pg_argv
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    run_pg.main()
    if rank == 0:
        with open(args.worker_out, "w") as f:
            json.dump(dict(ranks=world, iterations=[{k: v for k, v in it.items() if k != "t0"} for it in iters]), f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--ranks", default="1,2,8")
    ap.add_argument("--env", default="Pendulum-v0")
    ap.add_argument("--agent", default="modular_rl.agentzoo.TrpoAgent")
    ap.add_argument("--timesteps_per_batch", type=int, default=50000)
    ap.add_argument("--vec_envs", type=int, default=16)
    ap.add_argument("--n_iter", type=int, default=4, help="the first iteration is a warm-up and not summarised")
    ap.add_argument("--timeout", type=int, default=900)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--worker_out")
    args = ap.parse_args()

    with tempfile.TemporaryDirectory() as tmp:
        run_pg_argv = ["--env", args.env, "--agent", args.agent, "--timesteps_per_batch", str(args.timesteps_per_batch),
                       "--vec_envs", str(args.vec_envs), "--n_iter", str(args.n_iter), "--cg_damping", "0.1",
                       "--outfile", os.path.join(tmp, "run.h5")]
        if args.worker:
            return worker(args, run_pg_argv)

        import torch
        n_gpu = torch.cuda.device_count()
        name, watts = card()
        report = dict(card=name, power_limit_w=watts, visible_gpus=n_gpu, env=args.env, agent=args.agent,
                      timesteps_per_batch=args.timesteps_per_batch, vec_envs_per_rank=args.vec_envs,
                      n_iter=args.n_iter, runs=[])
        for w in [int(x) for x in args.ranks.split(",")]:
            if w > n_gpu:
                report["runs"].append(dict(ranks=w, result="not measured (%d GPUs visible)" % n_gpu))
                continue
            wout = os.path.join(tmp, "w%d.json" % w)
            with socket.socket() as s:
                s.bind(("127.0.0.1", 0))
                port = s.getsockname()[1]
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(w),
                   "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__), "--worker",
                   "--worker_out", wout, "--out", args.out, "--env", args.env, "--agent", args.agent,
                   "--timesteps_per_batch", str(args.timesteps_per_batch), "--vec_envs", str(args.vec_envs),
                   "--n_iter", str(args.n_iter)]
            p = subprocess.Popen(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                                 start_new_session=True)
            try:
                log, _ = p.communicate(timeout=args.timeout)
            except subprocess.TimeoutExpired:
                import signal
                os.killpg(p.pid, signal.SIGKILL)
                log, _ = p.communicate()
            if p.returncode != 0 or not os.path.exists(wout):
                report["runs"].append(dict(ranks=w, result="not measured (run failed, exit %s)" % p.returncode,
                                           log_tail=log[-3000:]))
                continue
            with open(wout) as f:
                run = json.load(f)
            import numpy as np
            steady = run["iterations"][1:] or run["iterations"]
            run["median_s"] = {k: float(np.median([it[k] for it in steady]))
                               for k in ("rollouts", "advantage_vf", "update", "total")}
            report["runs"].append(run)
            print("ranks %d: median per iteration %s" % (w, {k: "%.3f s" % v for k, v in run["median_s"].items()}),
                  flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)
    print("card: %s, power limit %s W -> %s" % (name, watts, args.out))


if __name__ == "__main__":
    main()
