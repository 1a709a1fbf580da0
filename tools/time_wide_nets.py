#!/usr/bin/env python
"""Time updates of nets that run layers >= 2 on the layer-by-layer path (mlp_layers.cu), and one net on the fused
kernels for context.  For each case: the median wall time of one update (TRPO step, or one NnVf.fit), the per-class
kernel times from the library's CUDA-event profiler in a separate profiled run, and the algorithmic TFLOP/s of the
layers >= 2 classes (mid_forward, mid_backward_grad, mid_backward_fvp), computed from the shapes: per timestep and
layer l >= 2 with K = d[l-1], N = d[l], a forward pass is 2KN flops, a gradient pass 4KN (delta and weight
gradient), an Fvp pass 8KN (two R-forward products, delta, weight gradient).  The 3xTF32 split triples the tensor
work actually issued; the rate given is the algorithmic one.  A report, not a check.

  python tools/time_wide_nets.py --out_dir /tmp/wide_nets

Writes one JSON per case with the card name and power limit read in the same run."""
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

CASES = [   # name, kind, dims, timesteps, head (0 DiagGauss, 1 Categorical, 2 value)
    ("trpo_11-256-256-3_50k", "trpo", (11, 256, 256, 3), 50_000, 0),
    ("trpo_11-256-256-3_1m", "trpo", (11, 256, 256, 3), 1_000_000, 0),
    ("trpo_4-128-128-2_50k", "trpo", (4, 128, 128, 2), 50_000, 1),
    ("vffit_12-256-256-1_200k", "vffit", (12, 256, 256, 1), 200_000, 2),
    ("trpo_11-64-64-3_50k_fused", "trpo", (11, 64, 64, 3), 50_000, 0),
]
PASS_FLOPS = {"mid_forward": 2, "mid_backward_grad": 4, "mid_backward_fvp": 8}


def kernel_table(lib, L):
    nk = lib.mrl_profile_kinds()
    pms, pcnt = (C.c_double * nk)(), (C.c_longlong * nk)()
    L.check(lib.mrl_profile_read(pms, pcnt))
    lib.mrl_profile_enable(0)
    return {lib.mrl_profile_kind_name(k).decode(): (pms[k], pcnt[k]) for k in range(nk) if pcnt[k]}


def setup(kind, dims, N, head):
    """-> one update as a callable; it returns after the device has finished (its results come back to the host)"""
    from modular_rl_b200 import core, synth
    from modular_rl_b200.device import DeviceBatch, DeviceNet
    rng = np.random.default_rng(0)
    if kind == "trpo":
        net = DeviceNet(dims, head)
        batch = DeviceBatch(dims[0], with_time_feature=True)

        def forward(theta, ob):        # oldprob from the same net: the batch a TRPO iteration would see
            net.set_params(theta)
            batch.set_obs(ob)
            return net.forward(batch)
        d = synth.policy_batch(synth.Workload("wide", dims, head, N, 1000, 7), forward)
        batch.set_obs(d["ob"]).set_paths(d["offsets"], d["terminated"], 1000.0)
        batch.set_policy_inputs(head, dims[-1], d["act"], d["adv"], d["oldprob"])
        theta0 = synth.perturb(d["theta"], 0.02, 5)

        def update():
            net.set_params(theta0)
            net.trpo_step(batch, cg_damping=0.1, max_kl=0.01)
        return update
    vf = core.NnVf(core.make_value_net(dims[0] - 1, list(dims[1:-1])), 1000, dict(mixfrac=0.1, maxiter=25))
    theta0 = vf.reg.net.get_params()
    ob = synth.make_obs(N, dims[0] - 1, rng)
    off = np.asarray(synth.make_paths(N, 1000, rng)[0], np.int64)
    y = rng.standard_normal(N)
    paths = [{"observation": ob[off[i]:off[i + 1]], "return": y[off[i]:off[i + 1]]} for i in range(len(off) - 1)]

    def update():
        vf.reg.net.set_params(theta0)
        vf.fit(paths)
    return update


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out_dir", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--cases", default=",".join(c[0] for c in CASES))
    args = ap.parse_args()
    from modular_rl_b200 import _lib as L
    from time_dp_training import card
    lib = L.lib()
    name, watts = card()
    os.makedirs(args.out_dir, exist_ok=True)
    want = set(args.cases.split(","))
    for cname, kind, dims, N, head in CASES:
        if cname not in want:
            continue
        update = setup(kind, dims, N, head)
        update()                                   # warm-up: module loads, buffer growth
        secs = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            update()
            secs.append(time.perf_counter() - t0)
        lib.mrl_profile_enable(1)                 # profiled run of its own
        update()
        table = kernel_table(lib, L)
        kn = sum(dims[l - 1] * dims[l] for l in range(2, len(dims)))
        classes = {}
        for k, (ms, cnt) in table.items():
            row = dict(ms_per_update=ms, passes=cnt)
            if k in PASS_FLOPS:
                flops = PASS_FLOPS[k] * kn * N * cnt
                row["algorithmic_tflops"] = flops / (ms * 1e-3) / 1e12 if ms > 0 else None
            classes[k] = row
        rep = dict(case=cname, card=name, power_limit_w=watts, update=kind, dims=list(dims), timesteps=N,
                   path="fused" if cname.endswith("_fused") else "layer-by-layer",
                   median_s_per_update=float(np.median(secs)), spread_s=[float(min(secs)), float(max(secs))],
                   reps=args.reps, kernel_classes=classes)
        print(json.dumps(rep), flush=True)
        with open(os.path.join(args.out_dir, "r05a_%s.json" % cname), "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
