#!/usr/bin/env python
"""bench.py - TRPO update timesteps/s (Fvp + CG + line search + GAE) on B200.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank/GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py ... --dump-outputs DIR       (+ the last timed step's outputs as DIR/<name>.npy)

One "step" = one full policy update on one synthetic batch of the named workload:
value-net forward (NnVf.predict) -> GAE + standardise (compute_advantage, core.py:63-105) ->
TrpoUpdater.__call__ (trpo.py:72-140: gradient, 10 CG Fisher-vector products, shs product,
backtracking line search).  Parameters are reset to the same theta before every step so that
all steps do identical work.

`value`: inputs resident in HBM when the timed region starts.  `e2e`: the same update through
the C ABI with HOST (pinned) buffers - observations, actions, old probabilities, rewards and
parameters are copied host->device and returns/advantages/stats device->host inside the timed
region.  Multi-GPU: the 1M-timestep batch is sharded over the ranks (strong scaling); partial
sums are combined with NCCL all-reduces; CG runs replicated.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

HOST_CORES = len(os.sched_getaffinity(0))
# torch.distributed.run exports OMP_NUM_THREADS=1 to every rank.  The CPU legs of this file (the reference arm and
# rank 0's oracle checks) run while the other ranks idle, so they get the box's cores back - set BEFORE numpy loads
# its BLAS; the thread count actually in use is read back with threadpoolctl and reported.
if int(os.environ.get("RANK", "0")) == 0:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(HOST_CORES)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(cg_damping=0.1, max_kl=0.01, gamma=0.995, lam=0.97)   # battery-trpo.yaml:7-11
METRIC = "trpo_update_timesteps_per_sec"
UNIT = "timesteps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="humanoid",
                    help="humanoid (configs[2], default) | hopper (configs[1]) | walker_ppo (configs[3]) | cat_vf (configs[4]) | any synth.WORKLOADS name")
    ap.add_argument("--timesteps", type=int, default=0, help="total timesteps (default: the workload's)")
    ap.add_argument("--cpu-sample", type=int, default=100_000, help="timesteps of the CPU baseline sample (b200 arm)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="reference arm: wall-clock budget of the K+W sampled steps")
    ap.add_argument("--verify", default="quick", choices=["none", "quick", "full"],
                    help="parity legs outside the timed region, on the FULL batch against the fp64 oracle: "
                         "quick = losses, gradient, one Fvp, advantages; full = + the oracle's whole update (step direction, stats)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--nccl-only", action="store_true", help="sum over ranks with NCCL instead of the NVLink peer-memory exchange")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy "
                         "(float32 / float64; the inputs are seeded, so two builds can be compared array by array)")
    return ap.parse_args()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, integers widened to float64, at most DUMP_LIMIT_BYTES in all."""
    arrays = {k: np.asarray(v, np.float32 if np.asarray(v).dtype == np.float32 else np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_desc(wl, n_total):
    hid = "-".join(str(d) for d in wl.dims[1:-1])
    head = "DiagGauss" if wl.head == 0 else "Categorical"
    return (f"{wl.name}: obs {wl.dims[0]}, act {wl.dims[-1]}, {hid} tanh MLP, {head}, {n_total} timesteps; "
            "step = VF predict + GAE + standardise + TRPO update (1 grad, 10 CG Fvp + 1, line search)")


# ----------------------------------------------------------------------------- CPU reference arm
def blas_threads():
    """BLAS threads numpy really uses (threadpoolctl), not the affinity mask."""
    try:
        from threadpoolctl import threadpool_info
        n = [int(i.get("num_threads", 0)) for i in threadpool_info() if i.get("user_api") == "blas"]
        return max(n) if n else None
    except Exception:
        return None


class CpuArm:
    """The oracle port of the reference's CPU path (float32 = the fork's floatX), timed on this box's host cores with
    all BLAS threads: GAE (scipy lfilter per path, as the reference) + one TRPO update (1 gradient, 10 CG
    Fisher-vector products + 1, line search).  The Fvp is the oracle's CLOSED FORM (forward + R-forward + reverse
    sweep), which does less arithmetic than the reverse-over-reverse graph Theano differentiates: the port is a
    conservative (fast) stand-in for the reference."""

    def __init__(self, wl, n_max):
        from modular_rl_b200 import synth
        from oracle import policy_math as pm
        self.wl, self.pm = wl, pm
        self.spec = pm.NetSpec(wl.dims, pm.GAUSS if wl.head == 0 else pm.CAT)

        def fwd(th, ob):
            _, z = pm.forward(th, self.spec, ob, np.float32)
            return z if wl.head == 0 else pm.softmax(z)
        self.data = synth.policy_batch(wl, fwd, N=n_max)
        self.base = np.tanh(self.data["ob"][:, 0]).astype(np.float32)
        self.n_max = n_max

    def step(self, n):
        """one update on the first n timesteps (whole trajectories are not needed by the arithmetic) -> seconds"""
        from oracle import advantage as oadv, natgrad
        d = self.data
        k = int(np.searchsorted(d["offsets"], n, side="right"))
        off = np.concatenate([d["offsets"][:k], [n]]) if d["offsets"][k - 1] != n else d["offsets"][:k]
        term = d["terminated"][:len(off) - 1]
        t0 = time.perf_counter()
        ret, adv = oadv.gae_flat(d["reward"][:n], self.base[:n], off, term, CFG["gamma"], CFG["lam"])
        adv = oadv.standardize(adv).astype(np.float32)
        natgrad.trpo_update(d["theta"], self.spec, d["ob"][:n], d["act"][:n], adv, d["oldprob"][:n],
                            CFG["cg_damping"], CFG["max_kl"], dtype=np.float32)
        return time.perf_counter() - t0


def cpu_update_rate(wl, n_sample, steps, warmup):
    arm = CpuArm(wl, n_sample)
    times = [arm.step(n_sample) for _ in range(warmup + steps)][warmup:]
    return n_sample * len(times) / sum(times), float(np.mean(times))


def run_reference(args, wl, n_total, rank, world):
    if rank != 0:
        return
    arm = CpuArm(wl, n_total)
    threads = blas_threads()
    # sample size: one calibration step, then the largest sample whose K+W steps fit the budget; one step on the FULL
    # batch shows that the rate does not depend on the sample size
    n_cal = min(n_total, 50_000)
    sec_cal = arm.step(n_cal)
    rates = {n_cal: n_cal / sec_cal}
    reps = args.steps + args.warmup
    n_sample = int(min(n_total, max(n_cal, rates[n_cal] * args.ref_budget_s / max(reps, 1))))
    if n_sample < n_total:
        rates[n_total] = n_total / arm.step(n_total)
    times = [arm.step(n_sample) for _ in range(reps)][args.warmup:]
    rate, sec = n_sample * len(times) / sum(times), float(np.mean(times))
    rates[n_sample] = rate
    sample = (f"{n_sample} of {n_total} timesteps per step (sample_fraction {n_sample / n_total:.3f}), oracle port "
              f"(numpy float32, closed-form Fvp, scipy lfilter per path), {threads} BLAS threads on {HOST_CORES} cores; "
              "rate by sample size: " + ", ".join(f"{n}: {r:.0f}/s" for n, r in sorted(rates.items())))
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3 * n_total / n_sample,
            "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_desc(wl, n_total), "timesteps": n_total, "sample_timesteps": n_sample,
                       "sample_fraction": n_sample / n_total, "parallelism": "cpu", **CFG},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads or HOST_CORES, "kind": "port", "sample": sample,
                             "rate_by_sample": {str(k): v for k, v in sorted(rates.items())}},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def nvlink_kib(gpu_index):
    """(tx KiB, rx KiB) summed over the NVLink links of one GPU (nvidia-smi nvlink -gt d), or None."""
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(gpu_index)], capture_output=True, text=True, timeout=20).stdout
        tx = rx = 0
        for ln in out.splitlines():
            f = ln.split()
            if "Tx:" in f:
                tx += int(f[f.index("Tx:") + 1])
            if "Rx:" in f:
                rx += int(f[f.index("Rx:") + 1])
        return (tx, rx) if (tx or rx) else None
    except Exception:
        return None


# ----------------------------------------------------------------------------- B200 arm
def chain_mma_flops_per_timestep(dims):
    """TF32 tensor-core flops the backward chain kernel ISSUES per timestep for an Fvp (3xTF32, widths padded to 8,
    weight-gradient m-tiles padded to 16): chain phase 3 GEMM passes over the (k-step, n-tile) pairs (W and V in the
    R-forward, W^T in the reverse sweep), grad phase one m16n8k8 block per 8 timesteps."""
    nt = [-(-d // 8) for d in dims]
    pairs = sum(nt[l - 1] * nt[l] for l in range(2, len(dims)))
    blocks = sum(-(-dims[l - 1] // 16) * nt[l] for l in range(2, len(dims)))
    return 3 * (3 * pairs) * 2048 / 16 + blocks * 3 * 2048 / 8


def tc_chain_issued_flops_per_timestep(dims):
    """TF32 tensor-core flops the tcgen05 Fisher-vector chain (mlp_fvp_tc.cu) ISSUES per timestep: 3 MMAs per product
    (split precision), K padded to 8, N to 16, the (k) weight-gradient tiles always M = 128 rows."""
    L = len(dims) - 1
    r8 = lambda d: -(-d // 8) * 8
    r16 = lambda d: -(-d // 16) * 16
    macs = 0
    for l in range(2, L + 1):
        macs += 2 * r8(dims[l - 1]) * r16(dims[l])        # Rh.W and h.V
        macs += r8(dims[l]) * r16(dims[l - 1])            # delta.W^T
    l = L                                                   # (k) passes: consecutive layers share a 128-row tile
    while l >= 2:
        rows = cols = 0
        k = l
        while k >= 2 and rows + dims[k - 1] + 1 <= 128 and cols + r16(dims[k]) <= 128:
            rows += dims[k - 1]; cols += r16(dims[k]); k -= 1
        macs += 128 * cols
        l = k
    return 3 * 2 * macs


def algorithmic_flops_per_timestep(dims):
    d0d1 = dims[0] * dims[1]
    S = sum(dims[l - 1] * dims[l] for l in range(2, len(dims)))
    return {"l1_forward": 2 * d0d1, "l1_grad": 2 * d0d1, "mid_forward": 2 * S, "mid_backward_grad": 4 * S,
            "mid_backward_fvp": 8 * S}

# ----------------------------------------------------------------------------- parity on the full batch
def run_parity(args, wl, n_total, rank, world, dist, dev, net, vf, batch, comm, reward_d, theta_d, rows, glob, stats_timed):
    """Outside the timed region: the CUDA path on the FULL bench batch against the float64 oracle (rank 0 holds the
    global host arrays; every rank takes part in the device calls).  Returns the measured relative errors."""
    if args.verify == "none":
        return None
    import torch
    from modular_rl_b200 import synth
    vf.predict_into_baseline(batch)
    ret_d, adv_d = batch.gae(reward_d, None, CFG["gamma"], CFG["lam"], True, comm)
    batch.refresh_advantages()
    net.set_params(theta_d)
    ls = net.losses(batch)
    g, _ = net.policy_gradient(batch)
    v = np.random.default_rng(12345).standard_normal(net.P).astype(np.float32)
    f = net.fvp(batch, v)
    full = None
    if args.verify == "full":
        st, info = net.trpo_step(batch, CFG["cg_damping"], CFG["max_kl"])
        sd, fs, sc = net.trpo_vectors()
        full = (np.array(st), info, sd, fs, net.get_params())
    # replicated parameters must be bit-identical on every rank
    th = torch.from_numpy(net.get_params().view(np.int32).astype(np.int64)).to(dev)
    chk = torch.stack([th.sum(), (th * torch.arange(1, th.numel() + 1, device=dev)).sum()])
    identical = True
    if world > 1:
        allc = [torch.empty_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        identical = all(bool((c == allc[0]).all()) for c in allc)
    if rank != 0:
        return None
    from oracle import advantage as oadv, natgrad, policy_math as pm
    rel = lambda a, b: float(np.linalg.norm(np.asarray(a, np.float64) - b) / max(np.linalg.norm(b), 1e-300))
    t0 = time.perf_counter()
    spec = pm.NetSpec(wl.dims, pm.GAUSS if wl.head == 0 else pm.CAT)
    r0, r1 = rows
    oret, oad = oadv.gae_flat(glob["reward"], glob["base"].astype(np.float64), glob["off"], glob["term"], CFG["gamma"], CFG["lam"])
    oads = oadv.standardize(oad)
    adv32 = oads.astype(np.float32)
    a = (glob["ob"], glob["act"], adv32, glob["oldprob"])
    th = glob["theta"]
    ols = pm.losses(th, spec, *a)
    og = pm.policy_gradient(th, spec, *a)
    of = pm.fisher_vector_product(th, spec, glob["ob"], v)
    og32 = pm.policy_gradient(th, spec, *a, dtype=np.float32)
    of32 = pm.fisher_vector_product(th, spec, glob["ob"], v, dtype=np.float32)
    out = {"timesteps": n_total, "oracle": "float64 numpy restatement (oracle/policy_math.py, oracle/advantage.py) on the full batch",
           "tolerance": 1e-5,
           "losses_rel": [float(abs(x - y) / max(abs(y), 1e-12)) for x, y in zip(ls, ols)],
           "losses_abs": [float(abs(x - y)) for x, y in zip(ls, ols)],
           "grad_rel_l2": rel(g, og), "fvp_rel_l2": rel(f, of),
           "returns_rel_l2": rel(ret_d.cpu().numpy(), oret[r0:r1]),
           "advantages_max_abs": float(np.max(np.abs(adv_d.cpu().numpy() - oads[r0:r1]))),
           "reference_fp32_noise_floor": {"grad_rel_l2": rel(og32, og), "fvp_rel_l2": rel(of32, of),
                                          "what": "the oracle run in float32 (the fork's floatX) against float64"},
           "theta_identical_across_ranks": identical}
    if full is not None:
        st, info, sd, fs, thn = full
        ostats, oinfo = natgrad.trpo_update(th, spec, *a, CFG["cg_damping"], CFG["max_kl"])
        want = np.array([ostats[k] for k in ("surr_before", "surr_after", "kl_before", "kl_after", "ent_before", "ent_after")])
        out.update(stepdir_rel_l2=rel(sd, oinfo["stepdir"]), fullstep_rel_l2=rel(fs, oinfo["fullstep"]),
                   theta_new_rel_l2=rel(thn, oinfo["theta_new"]),
                   stats_rel=[float(abs(x - y) / max(abs(y), 1e-12)) for x, y in zip(st, want)],
                   kl_after_rel=float(abs(st[3] - want[3]) / abs(want[3])),
                   accepted_index=[int(info["accepted_index"]), int(oinfo["accepted_index"])],
                   cg_iters=[int(info["cg_iters_run"]), int(oinfo["cg_iters_run"])])
    # the same global batch at every N: the timed update's statistics against the committed 1-GPU record
    ref_path = os.path.join(ROOT, "profiles", "n1_stats_%s_%d.json" % (wl.name, n_total))
    if world == 1 and os.environ.get("MRL_WRITE_N1_STATS"):
        json.dump({"workload": wl.name, "timesteps": n_total, "cfg": CFG, "stats": [float(x) for x in stats_timed]},
                  open(ref_path, "w"))
    try:
        n1 = json.load(open(ref_path))
        if n1["cfg"] == CFG:
            out["stats_vs_1gpu_record_max_rel"] = float(max(abs(x - y) / max(abs(y), 1e-12) for x, y in zip(stats_timed, n1["stats"])))
    except Exception:
        pass
    out["oracle_seconds"] = time.perf_counter() - t0
    ok = (max(out["grad_rel_l2"], out["fvp_rel_l2"]) < 1e-5 and out["advantages_max_abs"] < 1e-5 and identical and
          all(r < 1e-5 or d < 2e-7 for r, d in zip(out["losses_rel"], out["losses_abs"])))
    out["pass"] = bool(ok)
    return out

# ----------------------------------------------------------------------------- configs[3] and configs[4]
def kernel_table(lib, steps):
    nk = lib.mrl_profile_kinds()
    pms, pcnt = (C.c_double * nk)(), (C.c_longlong * nk)()
    from modular_rl_b200 import _lib as L
    L.check(lib.mrl_profile_read(pms, pcnt))
    lib.mrl_profile_enable(0)
    out = {}
    for k in range(nk):
        if pcnt[k]:
            out[lib.mrl_profile_kind_name(k).decode()] = {"launches_per_step": pcnt[k] / steps, "ms_per_step": pms[k] / steps,
                                                          "avg_ms": pms[k] / pcnt[k]}
    return out


def run_extra(args):
    """`--workload walker_ppo`: PpoLbfgsUpdater penalised-KL update on the 200 k-timestep Walker2d batch (configs[3]);
    `--workload cat_vf`: VF predict + GAE + standardise + NnVf fit on the 4 M-timestep ragged Categorical batch
    (configs[4]).  One GPU.  scipy's L-BFGS-B runs on the host as in the reference (ppo.py:85, core.py:687), every
    loss / gradient evaluation is a device pass over the resident batch."""
    import scipy.optimize
    import torch
    from modular_rl_b200 import _lib as L, synth
    from modular_rl_b200.device import DeviceBatch, DeviceNet
    from oracle import advantage as oadv, policy_math as pm, ppo_penalty, valuefn as vfo
    torch.cuda.set_device(0)
    lib = L.lib()
    ppo = args.workload == "walker_ppo"
    wl = synth.WORKLOADS["walker2d" if ppo else "cat128"]
    N = args.timesteps or wl.N
    rng = np.random.default_rng(wl.seed)
    theta0 = synth.init_params(wl.dims, wl.head, rng)
    ob = synth.make_obs(N, wl.dims[0], rng)
    off, term = synth.make_paths(N, wl.t_max, rng)
    reward = rng.standard_normal(N)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    ob_h, reward_h = pin(ob), pin(reward)
    batch = DeviceBatch(wl.dims[0], True)
    batch.set_obs(ob).set_paths(off, term, float(wl.t_max))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sampler = ClockSampler(0)
    maxiter = 25
    if ppo:
        net = DeviceNet(wl.dims, wl.head)
        net.set_params(theta0)
        out = net.forward(batch)
        d = wl.dims[-1]
        oldprob = np.concatenate([out, np.broadcast_to(np.exp(theta0[-d:])[None], out.shape)], 1).astype(np.float32)
        act = synth.sample_actions(wl.head, oldprob, rng)
        adv = rng.standard_normal(N)
        adv = ((adv - adv.mean()) / adv.std()).astype(np.float32)
        act_h, adv_h, oldprob_h = pin(act), pin(adv), pin(oldprob)
        batch.set_policy_inputs(wl.head, d, act, adv, oldprob)
        theta = synth.perturb(theta0, 0.01, wl.seed + 7)
        kl_coeff, kl_target = 1.0, 0.01
        evals = [0]

        def update(b):
            def lossandgrad(th):
                evals[0] += 1
                net.set_params(th)
                pen, g, _ = net.ppo_lossgrad(b, kl_coeff, 2 * kl_target)
                return pen, g
            net.set_params(theta)
            before = net.ppo_lossgrad(b, kl_coeff, 2 * kl_target, want_grad=False)[2]
            th, _, _ = scipy.optimize.fmin_l_bfgs_b(lossandgrad, theta.astype(np.float64), maxiter=maxiter)
            net.set_params(th)
            after = net.ppo_lossgrad(b, kl_coeff, 2 * kl_target, want_grad=False)[2]
            return before, after

        step_resident = lambda: update(batch)
        batch2 = DeviceBatch(wl.dims[0], True)

        def step_e2e():
            batch2.set_obs(ob_h.numpy()).set_paths(off, term, float(wl.t_max))
            batch2.set_policy_inputs(wl.head, d, act_h.numpy(), adv_h.numpy(), oldprob_h.numpy())
            return update(batch2)
        h2d = ob_h.numel() * 4 + act_h.numel() * 4 + adv_h.numel() * 4 + oldprob_h.numel() * 4 + off.nbytes + term.nbytes
        d2h = 0
        metric, what = "ppo_lbfgs_update_timesteps_per_sec", "PpoLbfgsUpdater update (penalised KL, L-BFGS-B maxiter 25 on the host, ppo.py:59-112)"
    else:
        vdims = (wl.dims[0] + 1, 64, 64, 1)
        vf = DeviceNet(vdims, synth.VALUE)
        vtheta = synth.init_params(vdims, synth.VALUE, np.random.default_rng(wl.seed + 1), last_scale=1.0)
        vf.set_params(vtheta)
        reward_d = reward_h.cuda()
        evals = [0]
        ret_h = torch.empty(N, dtype=torch.float64).pin_memory()
        adv_h = torch.empty(N, dtype=torch.float64).pin_memory()

        def fit(b):
            def lossandgrad(th):
                evals[0] += 1
                vf.set_params(th)
                ls, g = vf.vf_lossgrad(b, 1e-3)
                return ls[0], g
            b.mix_vf_target(0.1)                                # core.py:622-624, mixfrac = 0.1 (agentzoo.py:60)
            th, _, _ = scipy.optimize.fmin_l_bfgs_b(lossandgrad, vtheta.astype(np.float64), maxiter=maxiter)
            vf.set_params(th)
            return vf.vf_lossgrad(b, 1e-3, want_grad=False)[0]

        def step_resident():
            vf.set_params(vtheta)
            vf.predict_into_baseline(batch)
            batch.gae(reward_d, None, CFG["gamma"], CFG["lam"], True, None, want_outputs=False)
            return fit(batch)
        batch2 = DeviceBatch(wl.dims[0], True)

        def step_e2e():
            batch2.set_obs(ob_h.numpy()).set_paths(off, term, float(wl.t_max))
            vf.set_params(vtheta)
            vf.predict_into_baseline(batch2)
            batch2.gae(reward_h.numpy(), None, CFG["gamma"], CFG["lam"], True, None, out=(ret_h.numpy(), adv_h.numpy()))
            return fit(batch2)
        h2d = ob_h.numel() * 4 + reward_h.numel() * 8 + off.nbytes + term.nbytes
        d2h = 2 * N * 8
        metric, what = "gae_vf_fit_timesteps_per_sec", "VF predict + GAE + standardise + NnVf.fit (L-BFGS-B maxiter 25 on the host, core.py:63-105,619-697)"

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if profile:
            lib.mrl_profile_enable(1)
        l0 = lib.mrl_launch_count()
        evals[0] = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), int(lib.mrl_launch_count() - l0), res, evals[0] / steps
    sampler.start()
    ms, launches, res, n_eval = timed(step_resident, args.steps, max(args.warmup, 3))
    if args.dump_outputs:
        if ppo:
            dump_outputs(args.dump_outputs, {"losses_before": res[0], "losses_after": res[1], "theta": net.get_params()})
        else:
            dump_outputs(args.dump_outputs, {"vf_losses": res, "vf_theta": vf.get_params()})
    pms, _, _, _ = timed(step_resident, args.steps, 1, profile=True)
    clocks = sampler.stop()
    kernels = kernel_table(lib, args.steps)
    ems, _, _, _ = timed(step_e2e, args.steps, 3)
    fp32, tc32 = C.c_double(), C.c_double()
    L.check(lib.mrl_measure_fp32_tflops(0, C.byref(fp32)))
    L.check(lib.mrl_measure_tcgen05_tf32_tflops(0, C.byref(tc32)))
    dims = wl.dims if ppo else vdims
    flops = algorithmic_flops_per_timestep((dims[0],) + tuple(dims[1:]))
    for k, v in kernels.items():
        if k in flops:
            v["algo_tflops"] = flops[k] * N / (v["avg_ms"] * 1e-3) / 1e12
    top = max((k for k in kernels if k in flops), key=lambda k: kernels[k]["ms_per_step"])
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    roof = {"kernel": top, "bound": "tensor", "achieved": kernels[top]["algo_tflops"], "peak": peak_tf, "unit": "TFLOP/s",
            "frac": kernels[top]["algo_tflops"] / peak_tf, "traffic": None,
            "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"),
            "flops_counted": "algorithmic FP32 flops; each costs 3 TF32 MMAs", "tcgen05_tf32_peak_tflops": tc32.value,
            "fp32_fma_peak_tflops": fp32.value, "share_of_step": kernels[top]["ms_per_step"] / (pms / args.steps),
            "device_ms_per_step_all_kernels": sum(v["ms_per_step"] for v in kernels.values()),
            "host_ms_per_step": ms / args.steps - sum(v["ms_per_step"] for v in kernels.values())}
    extra_roof = None
    if not ppo and "gae" in kernels:
        gbs = 24.0 * N / (kernels["gae"]["avg_ms"] * 1e-3) / 1e9
        hbm = peaks.get("hbm_gbs") or 6650.0
        extra_roof = {"kernel": "gae", "bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                      "algorithmic_bytes_per_timestep": 24, "real_bytes_per_timestep": 40,
                      "note": "24 B = float32 reward/baseline in, return/advantage out + standardise; the kernel moves float64 reward, baseline, return, advantage"}
    # ---- parity at full size (outside the timed region) and the CPU port on a bounded sample
    if args.verify == "none":
        print(json.dumps({"metric": metric, "value": N * args.steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / args.steps,
                          "kernels": kernels, "note": "--verify none: timing only"}), flush=True)
        return
    rel = lambda a, b: float(np.linalg.norm(np.asarray(a, np.float64) - b) / max(np.linalg.norm(b), 1e-300))
    n_cpu = min(N, 100_000 if ppo else 400_000)
    k = int(np.searchsorted(off, n_cpu, side="right"))
    offc = np.concatenate([off[:k], [n_cpu]]) if off[k - 1] != n_cpu else off[:k]
    termc = term[:len(offc) - 1]
    if ppo:
        spec = pm.NetSpec(wl.dims, pm.GAUSS)
        net.set_params(theta)
        pen, g, ls = net.ppo_lossgrad(batch, kl_coeff, 2 * kl_target)
        open_, og = pm.ppo_lossgrad(theta, spec, ob, act, adv, oldprob, kl_coeff, 2 * kl_target)
        parity = {"timesteps": N, "pensurr_abs": float(abs(pen - open_)), "grad_rel_l2": rel(g, og), "tolerance": 1e-5,
                  "pass": bool(rel(g, og) < 2e-5)}
        t0 = time.perf_counter()
        ppo_penalty.ppo_lbfgs_update(theta, spec, ob[:n_cpu], act[:n_cpu], adv[:n_cpu], oldprob[:n_cpu], kl_coeff, kl_target,
                                     maxiter=maxiter, dtype=np.float32)
        sec = time.perf_counter() - t0
    else:
        spec = pm.NetSpec(vdims, pm.VALUE)
        vf.set_params(vtheta)
        base = vf.forward(batch)[:, 0]
        vf.predict_into_baseline(batch)
        ret, advd = batch.gae(reward, None, CFG["gamma"], CFG["lam"], True)
        oret, oad = oadv.gae_flat(reward, base.astype(np.float64), off, term, CFG["gamma"], CFG["lam"])
        tidx, _ = oadv.time_index(off)
        x = np.empty((N, vdims[0]), np.float64)
        x[:, :-1] = ob
        x[:, -1] = tidx / float(wl.t_max)
        batch.set_vf_target(ret)
        lsd, gd = vf.vf_lossgrad(batch, 1e-3)
        _, og = vfo.vf_lossgrad(vtheta, spec, x, oret.reshape(-1, 1), l2coeff=1e-3)
        parity = {"timesteps": N, "returns_rel_l2": rel(ret, oret), "advantages_max_abs": float(np.max(np.abs(advd - oadv.standardize(oad)))),
                  "vf_grad_rel_l2": rel(gd, og), "time_index_exact": bool(np.array_equal(batch.time_index(), tidx.astype(np.int32))),
                  "tolerance": 1e-5, "pass": bool(rel(gd, og) < 1e-5 and rel(ret, oret) < 1e-12)}
        t0 = time.perf_counter()
        b32 = base[:n_cpu]
        r_, a_ = oadv.gae_flat(reward[:n_cpu], b32, offc, termc, CFG["gamma"], CFG["lam"])
        oadv.standardize(a_)
        vfo.regression_fit(vtheta, spec, x[:n_cpu].astype(np.float32), r_.reshape(-1, 1), mixfrac=0.1, maxiter=maxiter, dtype=np.float32)
        sec = time.perf_counter() - t0
    threads = blas_threads()
    cpu = {"value": n_cpu / sec, "unit": UNIT, "cores": threads or HOST_CORES, "kind": "port",
           "sample": f"one step on {n_cpu} of {N} timesteps ({sec:.1f} s), oracle port in float32 (numpy + scipy L-BFGS-B / lfilter), {threads} BLAS threads"}
    line = {"metric": metric, "value": N * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{wl.name}: obs {wl.dims[0]}, {N} timesteps, {len(term)} trajectories; step = {what}",
                       "timesteps": N, "lossgrad_evals_per_step": n_eval, "maxiter": maxiter,
                       "l2": "inputs larger than L2" if N * wl.dims[0] * 4 > 126e6 else "L2 flushed by the step's own traffic (> 126 MB per step)",
                       **CFG},
            "roofline": roof, "roofline_gae": extra_roof, "cpu_baseline": cpu,
            "e2e": {"value": N * args.steps / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": ems / args.steps},
            "gpu_launches": launches, "clocks": clocks, "kernels": kernels, "parity": parity,
            "result": [float(v) for v in np.ravel(res[1] if ppo else res)]}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    from modular_rl_b200 import synth
    if args.workload in ("walker_ppo", "cat_vf"):
        if args.impl == "reference" or int(os.environ.get("WORLD_SIZE", 1)) > 1:
            raise SystemExit("--workload walker_ppo / cat_vf: one GPU, b200 arm only")
        return run_extra(args)
    wl = synth.WORKLOADS[args.workload]
    n_total = args.timesteps or wl.N
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs: b200 arm only (the reference arm sizes its sample from a timing, so its inputs vary)")
        run_reference(args, wl, n_total, rank, world)
        return

    import torch
    import torch.distributed as dist
    from modular_rl_b200 import _lib as L
    from modular_rl_b200.device import Comm, DeviceBatch, DeviceNet
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cores = 0
    if world > 1 and os.environ.get("MRL_NUMA_BIND", "1") != "0":
        from modular_rl_b200.parallel import bind_to_device_numa
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[local_rank]) if visible and visible.replace(",", "").isdigit() else local_rank
        numa_cores = bind_to_device_numa(phys)     # before any pinned allocation: first touch on the GPU's node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.lib()

    # ---- ONE global synthetic batch for every N (seeded once), sharded by WHOLE trajectories (parallel.shard_bounds):
    # the update statistics of the N = 1, 2, 4, 8 runs are then directly comparable (strong scaling: n_total is fixed)
    from modular_rl_b200.parallel import shard_bounds
    d0, dout = wl.dims[0], wl.dims[-1]
    grng = np.random.default_rng(wl.seed)
    theta = synth.init_params(wl.dims, wl.head, np.random.default_rng(wl.seed))
    vdims = (d0 + 1,) + tuple(wl.dims[1:-1]) + (1,)
    vtheta = synth.init_params(vdims, synth.VALUE, np.random.default_rng(wl.seed + 1), last_scale=1.0)
    ob_g = synth.make_obs(n_total, d0, grng)
    off_g, term_g = synth.make_paths(n_total, wl.t_max, grng)
    reward_g = grng.standard_normal(n_total)
    noise_g = (grng.standard_normal((n_total, dout), dtype=np.float32) if wl.head == synth.GAUSS
               else grng.random((n_total, 1), dtype=np.float32))
    pa, pb = shard_bounds(np.diff(off_g), world)[rank]
    r0, r1 = int(off_g[pa]), int(off_g[pb])
    n_local = r1 - r0
    offsets = (off_g[pa:pb + 1] - off_g[pa]).astype(np.int64)
    terminated = np.ascontiguousarray(term_g[pa:pb])

    net = DeviceNet(wl.dims, wl.head, device=local_rank)
    vf = DeviceNet(vdims, synth.VALUE, device=local_rank)
    net.set_params(theta)
    vf.set_params(vtheta)
    # the policy's own output on the global batch = path["prob"]; every rank computes it so that all N see the same rows
    tmp = DeviceBatch(d0, True, device=local_rank)
    tmp.set_obs(ob_g).set_paths(off_g, term_g, float(wl.t_max))
    out_g = net.forward(tmp)
    base_g = vf.forward(tmp)[:, 0].copy() if (rank == 0 and args.verify != "none") else None
    tmp.close()
    del tmp
    if wl.head == synth.GAUSS:
        oldprob_g = np.concatenate([out_g, np.broadcast_to(np.exp(theta[-dout:])[None], out_g.shape)], 1).astype(np.float32)
        act_g = (noise_g * oldprob_g[:, dout:] + oldprob_g[:, :dout]).astype(np.float32)     # DiagGauss.sample, core.py:432-435
    else:
        oldprob_g = out_g
        act_g = np.argmax(np.cumsum(oldprob_g, axis=1) > noise_g, axis=1).astype(np.int32)   # distributions.py:3-13
    del out_g, noise_g
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    ob_h, reward_h = pin(ob_g[r0:r1]), pin(reward_g[r0:r1])
    act_h, oldprob_h = pin(act_g[r0:r1]), pin(oldprob_g[r0:r1])
    if not (rank == 0 and args.verify != "none"):
        del ob_g, act_g, oldprob_g, reward_g            # only rank 0 keeps the global arrays (oracle legs)

    batch = DeviceBatch(d0, True, device=local_rank)
    comm = None
    if world > 1:
        from modular_rl_b200.parallel import comm_from_torch_distributed
        comm = comm_from_torch_distributed(local_rank, p2p=not args.nccl_only)
        net.set_comm(comm)
    batch.set_obs(ob_h.numpy()).set_paths(offsets, terminated, float(wl.t_max))
    batch.set_global_n(n_total)
    # move the policy slightly off theta_old, as after a few updates, so that ratios/KL are not trivial
    theta_cur = pin(synth.perturb(theta, 0.01, wl.seed + 7))
    reward_d = reward_h.to(dev)
    theta_d = theta_cur.to(dev)
    batch.set_policy_inputs(wl.head, dout, act_h.numpy(), np.zeros(n_local, np.float32), oldprob_h.numpy())

    def step_resident():
        vf.predict_into_baseline(batch)
        batch.gae(reward_d, None, CFG["gamma"], CFG["lam"], True, comm, want_outputs=False)
        batch.refresh_advantages()
        net.set_params(theta_d)
        return net.trpo_step(batch, CFG["cg_damping"], CFG["max_kl"])

    batch2 = DeviceBatch(wl.dims[0], True, device=local_rank)
    ret_h = torch.empty(n_local, dtype=torch.float64).pin_memory()
    adv_h = torch.empty(n_local, dtype=torch.float64).pin_memory()

    def step_e2e():
        batch2.set_obs(ob_h.numpy()).set_paths(offsets, terminated, float(wl.t_max))
        batch2.set_global_n(n_total)
        vf.predict_into_baseline(batch2)
        batch2.gae(reward_h.numpy(), None, CFG["gamma"], CFG["lam"], True, comm, out=(ret_h.numpy(), adv_h.numpy()))
        batch2.set_policy_inputs(wl.head, wl.dims[-1], act_h.numpy(), None, oldprob_h.numpy())
        net.set_params(theta_cur.numpy())
        return net.trpo_step(batch2, CFG["cg_damping"], CFG["max_kl"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        barrier()
        if profile:
            lib.mrl_profile_enable(1)
        l0 = lib.mrl_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), int(lib.mrl_launch_count() - l0), res

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # The timed region proper carries no per-kernel events: an event pair around each of the ~108 launches
    # of a step opens ~4 us of launch gap each (0.43 ms per step, measured; 1 % at 1M timesteps on one
    # GPU but 7 % of the 8-GPU step).  The per-kernel table and the roofline come from a second pass of the
    # same K steps, in this process, with the library's CUDA events on the launching stream.
    nv0 = nvlink_kib(local_rank) if (rank == 0 and world > 1) else None
    ms, launches, (stats, info) = timed(step_resident, args.steps, max(args.warmup, 3))
    nv1 = nvlink_kib(local_rank) if (rank == 0 and world > 1) else None
    if args.dump_outputs and rank == 0:         # the parameters are replicated: rank 0's are everyone's
        dump_outputs(args.dump_outputs, {"trpo_stats": stats, "trpo_info": list(info.values()), "theta": net.get_params()})
    nvlink = None
    if nv0 and nv1:
        nsteps = args.steps + max(args.warmup, 3)
        nvlink = {"tx_kib_per_step": (nv1[0] - nv0[0]) / nsteps, "rx_kib_per_step": (nv1[1] - nv0[1]) / nsteps,
                  "how": "nvidia-smi nvlink -gt d on rank 0's GPU around the warm-up + timed steps",
                  "expected_kib_per_step": 13 * net.P * 8 * (world - 1) / 1024.0,
                  "what": "each of the 13 sums over ranks per update (1 gradient, 11 Fvp, loss triples apart) reads P doubles from every peer"}
    pms_total, _, _ = timed(step_resident, args.steps, 1, profile=True)
    clocks = sampler.stop() if rank == 0 else None
    nk = lib.mrl_profile_kinds()
    pms, pcnt = (C.c_double * nk)(), (C.c_longlong * nk)()
    L.check(lib.mrl_profile_read(pms, pcnt))
    lib.mrl_profile_enable(0)
    value = n_total * args.steps / (ms * 1e-3)
    e2e = None
    if not args.no_e2e:
        ems, _, _ = timed(step_e2e, args.steps, 3)
        h2d = (ob_h.numel() * 4 + act_h.numel() * act_h.element_size() + oldprob_h.numel() * 4 +
               reward_h.numel() * 8 + theta_cur.numel() * 4 + offsets.nbytes + terminated.nbytes) * world
        d2h = (ret_h.numel() * 8 + adv_h.numel() * 8 + 6 * 8 + 4 * 32) * world
        e2e = {"value": n_total * args.steps / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": ems / args.steps}

    parity = run_parity(args, wl, n_total, rank, world, dist if world > 1 else None, dev, net, vf, batch, comm, reward_d, theta_d,
                        (r0, r1), dict(ob=ob_g, act=act_g, oldprob=oldprob_g, reward=reward_g, off=off_g, term=term_g,
                                       base=base_g, theta=theta_cur.numpy()) if (rank == 0 and args.verify != "none") else None,
                        stats)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        fp32, mma32, tc32 = C.c_double(), C.c_double(), C.c_double()
        L.check(lib.mrl_measure_fp32_tflops(local_rank, C.byref(fp32)))
        L.check(lib.mrl_measure_mma_tf32_tflops(local_rank, C.byref(mma32)))
        L.check(lib.mrl_measure_tcgen05_tf32_tflops(local_rank, C.byref(tc32)))
        fvp_on_tc = os.environ.get("MRL_FVP_TC", "1") != "0" and wl.name in ("humanoid", "hopper", "walker2d", "cat128", "cartpole")
        flops = algorithmic_flops_per_timestep(wl.dims)
        kernels = {}
        for k in range(nk):
            name = lib.mrl_profile_kind_name(k).decode()
            if pcnt[k] == 0:
                continue
            avg_ms = pms[k] / pcnt[k]
            ent = {"launches_per_step": pcnt[k] / args.steps, "ms_per_step": pms[k] / args.steps, "avg_ms": avg_ms}
            if name in flops:
                tf = flops[name] * n_local / (avg_ms * 1e-3) / 1e12
                ent.update(algo_tflops=tf, frac_fp32_peak=tf / fp32.value)
            if name == "gae":
                ent.update(algo_gbs=24.0 * n_local / (avg_ms * 1e-3) / 1e9)
            kernels[name] = ent
        top = max((k for k in kernels if k in flops), key=lambda k: kernels[k]["ms_per_step"])
        peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            if tr["workload"] == wl.name and tr["timesteps"] == n_local and top in tr["kernels"]:
                traffic = tr["kernels"][top]["read"] + tr["kernels"][top]["write"]
        except Exception:
            pass
        pipes = {"mid_backward_fvp": ("tcgen05.mma kind::tf32 x3 split precision in TS mode (activations written to TMEM by the epilogue warps, "
                                      "weights streamed through a shared-memory ring), R-forward and delta phases of consecutive tiles overlapped"
                                      if fvp_on_tc else
                                      "per-warp register chain, mma.sync TF32 x3 split precision (FP32-class accuracy) + FP32 epilogues"),
                 "mid_backward_grad": "per-warp register chain, mma.sync TF32 x3 split precision + FP32 heads",
                 "mid_forward": "per-warp register chain, mma.sync TF32 x3 split precision + FP32 heads",
                 "l1_forward": "tcgen05.mma kind::tf32 x3 split precision, TMEM accumulators, raw-fp32 operand split in shared memory",
                 "l1_grad": "tcgen05.mma kind::tf32 x3 split precision, TMEM accumulators, raw-fp32 operand split in shared memory"}
        roof = {"kernel": top, "bound": "tensor", "achieved": kernels[top]["algo_tflops"], "peak": peak_tf,
                "unit": "TFLOP/s", "frac": kernels[top]["algo_tflops"] / peak_tf, "traffic": traffic,
                "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else
                                "fallback 1.4 PFLOP/s sustained (of fallback)"),
                "pipe": pipes.get(top, ""), "flops_counted": "algorithmic FP32 flops; each costs 3 TF32 MMAs",
                "tf32_mma_tflops_issued": (((tc_chain_issued_flops_per_timestep if fvp_on_tc else chain_mma_flops_per_timestep)(wl.dims)
                                            * n_local / (kernels[top]["avg_ms"] * 1e-3) / 1e12)
                                           if top == "mid_backward_fvp" else 3.0 * kernels[top]["algo_tflops"]),
                "mma_sync_tf32_peak_tflops": mma32.value,
                "tcgen05_tf32_peak_tflops": tc32.value,
                "fp32_fma_peak_tflops": fp32.value,
                "frac_of_fp32_fma_peak": kernels[top]["algo_tflops"] / fp32.value,
                "share_of_step": kernels[top]["ms_per_step"] / (pms_total / args.steps),
                "kernel_events": "second pass of the same %d steps with per-kernel CUDA events (%.3f ms per step; "
                                 "the timed region itself has none)" % (args.steps, pms_total / args.steps)}
        on_tc = top in ("l1_forward", "l1_grad") or (top == "mid_backward_fvp" and fvp_on_tc)
        if on_tc:
            roof["frac_of_tcgen05_tf32_peak"] = roof["tf32_mma_tflops_issued"] / tc32.value if tc32.value else None
        else:
            roof["frac_of_mma_sync_tf32_peak"] = roof["tf32_mma_tflops_issued"] / mma32.value if mma32.value else None
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cores = len(os.sched_getaffinity(0))
            n_sample = min(args.cpu_sample, n_total)
            rate, sec = cpu_update_rate(wl, n_sample, 1, 0)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"one update on {n_sample} of {n_total} timesteps ({sec:.1f} s), oracle port "
                             f"(numpy float32 + scipy lfilter), {cores} BLAS threads"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_desc(wl, n_total), "timesteps": n_total,
                           "timesteps_per_gpu": n_local, "parallelism": f"dp{world}",
                           "allreduce": ("none" if world == 1 else ("nvlink peer-memory exchange (publish fused into the slab reduce, "
                                                                    "peer reads fused into the CG step)" if comm.p2p else "nccl")),
                           "host_numa_cores_bound": numa_cores,
                           "l2": "inputs larger than L2 (observations %.2f GB per GPU)" % (n_local * wl.dims[0] * 4 / 1e9),
                           **CFG},
                "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
                "kernels": kernels, "parity": parity, "nvlink": nvlink,
                "update": {"stats": [float(s) for s in stats], "info": info}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        if comm:
            comm.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
