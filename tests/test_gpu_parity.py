"""Parity of the CUDA path (through the C ABI) against the oracle and the golden vectors.

Tolerances (north_star): bit-exact for trajectory indexing / segment boundaries; 1e-5 relative
(L2 over the vector) for fp32 Fvp, gradient, step direction, KL, advantages, against the float64
oracle.  The step direction is tested at cg_damping=0.1 (battery-trpo.yaml:10); with the code
default 1e-3 the CG system is so ill-conditioned that rounding the tangent to float32 - which
the reference itself does, trpo.py:48 - moves the solution by 1e-4 (see test_oracle_golden).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from conftest import relerr  # noqa: E402

TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    from modular_rl_b200 import device
    from modular_rl_b200 import _lib
    _lib.lib()
    return device


def _oracle():
    from oracle import advantage, natgrad, policy_math, ppo_penalty, valuefn, zfilter
    return advantage, natgrad, policy_math, ppo_penalty, valuefn, zfilter


def _bind(dev, spec_dims, head, ob, act, adv, oldprob, theta, with_time=True, activation="tanh"):
    net = dev.DeviceNet(spec_dims, head, activation)
    batch = dev.DeviceBatch(spec_dims[0], with_time_feature=with_time)
    batch.set_obs(ob)
    N = ob.shape[0]
    batch.set_paths(np.array([0, N], np.int64), np.array([1], np.uint8), 1000.0)
    batch.set_policy_inputs(head, spec_dims[-1], act, adv, oldprob)
    net.set_params(theta)
    return net, batch


def _golden_case(golden, tag):
    _, _, pm, *_ = _oracle()
    head = pm.GAUSS if tag == "tg" else pm.CAT
    dims = tuple(int(d) for d in golden[tag + "_dims"])
    act = golden[tag + "_act"]
    if tag == "tc":
        act = act.astype(np.int64)
    return pm.NetSpec(dims, head), (0 if tag == "tg" else 1), golden[tag + "_theta"], golden[tag + "_ob"], act, \
        golden[tag + "_adv"], golden[tag + "_oldprob"]


@pytest.mark.parametrize("tag", ["tg", "tc"])
def test_golden_losses_gradient_fvp(dev, golden, tag):
    spec, head, th, ob, act, adv, oldp = _golden_case(golden, tag)
    net, batch = _bind(dev, spec.dims, head, ob, act, adv, oldp, th)
    assert net.P == th.size
    th32 = th.astype(np.float32)
    assert np.array_equal(net.get_params(), th32)
    _, _, pm, *_ = _oracle()
    # the device holds float32 parameters: compare with the oracle at the same rounded theta
    ls = net.losses(batch)
    ols = pm.losses(th32, spec, ob, act, adv, oldp)
    assert np.allclose(ls, ols, rtol=TOL, atol=1e-7), (ls, ols)
    g, ls2 = net.policy_gradient(batch)
    assert np.allclose(ls2, ls, rtol=1e-12)
    assert relerr(g, pm.policy_gradient(th32, spec, ob, act, adv, oldp)) < TOL
    assert relerr(g, golden[tag + "_pg"]) < 1e-4          # golden is at the un-rounded theta
    f = net.fvp(batch, golden[tag + "_v"])
    assert relerr(f, pm.fisher_vector_product(th32, spec, ob, golden[tag + "_v"])) < TOL
    assert relerr(f, golden[tag + "_fvp"]) < 1e-4
    out = net.forward(batch)
    _, z = pm.forward(th32, spec, ob)
    want = z if head == 0 else pm.softmax(z)
    assert relerr(out, want) < TOL


@pytest.mark.parametrize("tag", ["tg", "tc"])
@pytest.mark.parametrize("cfg", ["d", "b"])
def test_golden_trpo_step(dev, golden, tag, cfg):
    spec, head, th, ob, act, adv, oldp = _golden_case(golden, tag)
    net, batch = _bind(dev, spec.dims, head, ob, act, adv, oldp, th)
    damping, max_kl = golden[f"{tag}_{cfg}_cfg"]
    stats, info = net.trpo_step(batch, cg_damping=damping, max_kl=max_kl)
    key = f"{tag}_{cfg}_"
    _, natgrad, pm, *_ = _oracle()
    _, oinfo = natgrad.trpo_update(th.astype(np.float32), spec, ob, act, adv, oldp, damping, max_kl)
    assert info["success"] == int(golden[key + "success"]) and info["skipped"] == 0
    assert info["cg_iters_run"] == oinfo["cg_iters_run"] and info["n_fvp"] == oinfo["n_fvp"]
    sd, fs, sc = net.trpo_vectors()
    # cfg "d" (cg_damping=1e-3 on a 96-sample batch) is ill-conditioned: the reference's own
    # float32 path differs from float64 by 2.4e-4 (gauss) / 5.4e-3 (categorical) in the step
    # direction and 2 % in kl_after (measured with oracle dtype=float32, see DESIGN.md), so the
    # bound there is that noise floor, not 1e-5.
    tol = 2e-2 if cfg == "d" else 1e-4
    assert relerr(sd, golden[key + "stepdir"]) < tol
    assert relerr(fs, golden[key + "fullstep"]) < tol
    assert relerr(net.get_params(), golden[key + "theta_new"]) < (2e-2 if cfg == "d" else 1e-5)
    assert np.allclose(stats[0::2], golden[key + "before"], rtol=1e-5, atol=1e-7)
    assert np.allclose(stats[1::2], golden[key + "after"], rtol=(5e-2 if cfg == "d" else 1e-4), atol=1e-6)


def test_cg_iteration_kernels_agree(dev, golden, monkeypatch):
    """The CG iteration has two kernels: one thread-block cluster with the vectors in registers (P <= 49 152) and
    the grid-barrier kernel for longer vectors.  MRL_CG_GRID=1 forces the second on a small net: same iteration
    count and the same step to fp64 rounding of the partial-sum grouping."""
    spec, head, th, ob, act, adv, oldp = _golden_case(golden, "tg")
    damping, max_kl = golden["tg_b_cfg"]
    res = []
    for force_grid in (False, True):
        if force_grid:
            monkeypatch.setenv("MRL_CG_GRID", "1")
        net, batch = _bind(dev, spec.dims, head, ob, act, adv, oldp, th)
        for _ in range(2):                      # twice: the barrier words must come back to their rest state
            net.set_params(th)
            stats, info = net.trpo_step(batch, cg_damping=damping, max_kl=max_kl)
        res.append((np.array(stats), info, net.trpo_vectors()[0].copy(), net.get_params().copy()))
    monkeypatch.delenv("MRL_CG_GRID")
    (s0, i0, d0, t0), (s1, i1, d1, t1) = res
    assert i0["cg_iters_run"] == i1["cg_iters_run"] and i0["success"] == i1["success"]
    assert relerr(d1, d0) < 1e-9 and relerr(t1, t0) < 1e-6
    assert np.allclose(s0, s1, rtol=1e-6, atol=1e-9)


SHAPES = {
    "hopper": ((11, 64, 64, 3), 0, 5000),
    "humanoid": ((376, 100, 50, 25, 17), 0, 3001),
    "walker": ((17, 64, 64, 6), 0, 1234),
    "cat128": ((128, 64, 64, 18), 1, 2500),
    "cartpole": ((4, 64, 64, 2), 1, 777),
    "linear": ((6, 4), 0, 100),
    "one_hidden": ((9, 33, 5), 1, 257),
    # first hidden layer wider than 128: single (not double-buffered) TMEM accumulator in the layer-1 forward
    # kernel, wide rows in the layer-1 gradient kernel, generic job-list kernels for the rest
    "wide": ((20, 160, 16, 4), 0, 1500),
    "wide_in": ((300, 136, 24, 5), 1, 900),
    # --activation relu|sigmoid (agentzoo.py:22,37,58): generic job-list kernels
    "relu": ((11, 64, 64, 3), 0, 2000, "relu"),
    "sigmoid": ((17, 32, 16, 5), 1, 1500, "sigmoid"),
    "relu_humanoid": ((376, 100, 50, 25, 17), 0, 1100, "relu"),
}


def _synth_case(name):
    from modular_rl_b200 import synth
    _, _, pm, *_ = _oracle()
    dims, head, N = SHAPES[name][:3]
    act = SHAPES[name][3] if len(SHAPES[name]) > 3 else "tanh"
    wl = synth.Workload(name, dims, head, N, 200, 11)
    spec = pm.NetSpec(dims, pm.GAUSS if head == 0 else pm.CAT, act)

    def fwd(th, ob):
        _, z = pm.forward(th, spec, ob)
        return z if head == 0 else pm.softmax(z)
    data = synth.policy_batch(wl, fwd)
    theta = synth.perturb(data["theta"], 0.02, 5)
    return spec, head, theta, data


MEASURED = {}   # name -> measured relative errors, written to gpurun_out/parity_measured.json at session end


@pytest.fixture(scope="module", autouse=True)
def _dump_measured():
    yield
    import json
    import os
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "parity_measured.json"), "w") as f:
            json.dump(MEASURED, f, indent=1, sort_keys=True)
    except OSError:
        pass


@pytest.mark.parametrize("name", list(SHAPES))
def test_synthetic_shapes(dev, name):
    spec, head, theta, d = _synth_case(name)
    _, natgrad, pm, *_ = _oracle()
    net, batch = _bind(dev, spec.dims, head, d["ob"], d["act"], d["adv"], d["oldprob"], theta,
                       activation=spec.activation)
    args = (d["ob"], d["act"], d["adv"], d["oldprob"])
    ls = net.losses(batch)
    ols = pm.losses(theta, spec, *args)
    assert np.allclose(ls, ols, rtol=TOL, atol=2e-7), (ls, ols)
    g, _ = net.policy_gradient(batch)
    og = pm.policy_gradient(theta, spec, *args)
    assert relerr(g, og) < TOL
    v = np.random.default_rng(3).standard_normal(net.P).astype(np.float32)
    f = net.fvp(batch, v)
    of = pm.fisher_vector_product(theta, spec, d["ob"], v)
    assert relerr(f, of) < TOL
    # a second Fvp reuses the cached activations and must not depend on call history
    assert np.array_equal(net.fvp(batch, v), f)
    stats, info = net.trpo_step(batch, cg_damping=0.1, max_kl=0.01)
    ostats, oinfo = natgrad.trpo_update(theta, spec, *args, 0.1, 0.01)
    assert info["success"] == int(oinfo["success"]) and info["accepted_index"] == oinfo["accepted_index"]
    assert info["cg_iters_run"] == oinfo["cg_iters_run"]
    sd, fs, sc = net.trpo_vectors()
    # Step direction (north_star: 1e-5).  CG amplifies rounding by the conditioning of F + damping*I, so the bar is
    # 1e-5 wherever the REFERENCE's own float32 path (oracle dtype=float32 = the fork's floatX) stays within 1e-5 of
    # float64; elsewhere the CUDA path must be at least as close to float64 as that float32 path is.  Both numbers
    # are recorded (gpurun_out/parity_measured.json).
    _, o32 = natgrad.trpo_update(theta, spec, *args, 0.1, 0.01, dtype=np.float32)
    e_sd, e_fs = relerr(sd, oinfo["stepdir"]), relerr(fs, oinfo["fullstep"])
    floor = relerr(o32["stepdir"], oinfo["stepdir"])
    MEASURED[name] = dict(grad=relerr(g, og), fvp=relerr(f, of), stepdir=e_sd, fullstep=e_fs,
                          stepdir_reference_float32=floor, theta_new=relerr(net.get_params(), oinfo["theta_new"]))
    assert e_sd < max(TOL, 1.5 * floor), (e_sd, floor)
    assert e_fs < max(TOL, 1.5 * floor), (e_fs, floor)
    assert relerr(net.get_params(), oinfo["theta_new"]) < 1e-5
    want = np.array([ostats[k] for k in ("surr_before", "surr_after", "kl_before", "kl_after",
                                         "ent_before", "ent_after")])
    assert np.allclose(stats, want, rtol=1e-4, atol=1e-6), (stats, want)


def test_zero_gradient_is_skipped(dev):
    spec, head, theta, d = _synth_case("linear")
    net, batch = _bind(dev, spec.dims, head, d["ob"], d["act"], np.zeros_like(d["adv"]), d["oldprob"], theta)
    stats, info = net.trpo_step(batch)
    assert info["skipped"] == 1 and info["success"] == 0
    assert np.array_equal(net.get_params(), theta)
    assert stats[0] == stats[1] and stats[2] == stats[3]


def test_linesearch_failure_rolls_back(dev):
    """accept_ratio > 1 can never be met by a concave-improvement step: (False, x) + rollback
    (trpo.py:159,133)."""
    spec, head, theta, d = _synth_case("one_hidden")
    net, batch = _bind(dev, spec.dims, head, d["ob"], d["act"], d["adv"], d["oldprob"], theta)
    stats, info = net.trpo_step(batch, cg_damping=0.1, max_kl=0.01, accept_ratio=5.0)
    assert info["success"] == 0 and info["accepted_index"] == -1 and info["n_loss_passes"] == 11
    assert np.array_equal(net.get_params(), theta)
    assert stats[0] == stats[1]


# ----------------------------------------------------------------------------- GAE / scans
def _ragged(rng, n_paths, tmax):
    lens = rng.integers(1, tmax + 1, n_paths)
    lens[0] = 1
    lens[-1] = 1
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    term = (rng.random(n_paths) < 0.7).astype(np.uint8)
    return off, term


def test_gae_golden(dev, golden):
    lens = golden["adv_lens"]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    ret, adv = dev.gae_flat(golden["adv_reward"], golden["adv_baseline"], off, golden["adv_term"],
                            float(golden["adv_gamma"]), float(golden["adv_lam"]))
    assert np.allclose(ret, golden["adv_return"], rtol=1e-13, atol=1e-13)
    sadv, stats = dev.standardize(adv)
    assert np.allclose(sadv, golden["adv_advantage"], rtol=1e-6, atol=1e-7)
    assert stats[0] == adv.size


@pytest.mark.parametrize("n_paths,tmax", [(1, 1), (3, 5), (40, 300), (700, 3000), (5, 20000)])
def test_gae_ragged_vs_oracle(dev, n_paths, tmax):
    oadv, *_ = _oracle()
    rng = np.random.default_rng(n_paths * 7 + tmax)
    off, term = _ragged(rng, n_paths, tmax)
    N = int(off[-1])
    r = rng.standard_normal(N)
    v = rng.standard_normal(N).astype(np.float32)
    ret, adv = dev.gae_flat(r, v, off, term, 0.995, 0.97)
    oret, oad = oadv.gae_flat(r, v.astype(np.float64), off, term, 0.995, 0.97)
    assert np.allclose(ret, oret, rtol=1e-12, atol=1e-12)
    assert np.allclose(adv, oad, rtol=1e-12, atol=1e-12)
    # boundaries are exact: the last step of a path sees nothing after it
    last = off[1:] - 1
    assert np.array_equal(ret[last], r[last])
    # against the reference's dtype behaviour (float32 baseline, gamma*b1 rounded on open paths)
    _, oad32 = oadv.gae_flat(r, v, off, term, 0.995, 0.97)
    assert relerr(adv, oad32) < TOL


def test_batch_gae_and_time_index(dev):
    oadv, *_ = _oracle()
    rng = np.random.default_rng(5)
    off, term = _ragged(rng, 60, 400)
    N = int(off[-1])
    ob = rng.standard_normal((N, 7)).astype(np.float32)
    r = rng.standard_normal(N)
    v = rng.standard_normal(N).astype(np.float32)
    b = dev.DeviceBatch(7, with_time_feature=True)
    b.set_obs(ob).set_paths(off, term, 400.0)
    t, pid = oadv.time_index(off)
    assert np.array_equal(b.time_index(), t.astype(np.int32))        # bit-exact integer contract
    ret, adv = b.gae(r, v, 0.99, 0.95, standardize=True)
    oret, oad = oadv.gae_flat(r, v.astype(np.float64), off, term, 0.99, 0.95)
    assert np.allclose(ret, oret, rtol=1e-12, atol=1e-12)
    assert np.allclose(adv, oadv.standardize(oad), rtol=1e-10, atol=1e-10)
    assert abs(adv.mean()) < 1e-12 and abs(adv.std() - 1) < 1e-12


def test_zfilter_scan(dev, golden):
    *_, zf = _oracle()
    from modular_rl_b200 import filters
    X = golden["rs_x"]
    y, st = filters.zfilter_scan(X, None, demean=True, destd=True, clip=5.0)
    assert np.allclose(y, golden["zf_ob_y"], rtol=1e-12, atol=1e-12) and np.all(y[0] == 0)
    assert st[0] == len(X) and np.allclose(st[1], golden["rs_mean"][-1], rtol=1e-13)
    r = golden["zf_rew_x"].reshape(-1, 1)
    y, _ = filters.zfilter_scan(r, None, demean=False, destd=True, clip=10.0)
    assert np.allclose(y[:, 0], golden["zf_rew_y"], rtol=1e-12, atol=1e-12)
    rng = np.random.default_rng(9)
    X = (rng.standard_normal((5000, 11)) * rng.uniform(0.1, 30, 11) + rng.uniform(-5, 5, 11))
    state = zf.WelfordState((11,))
    want1 = zf.zfilter_batch(state, X[:1777], clip=5.0)
    y1, st1 = filters.zfilter_scan(X[:1777], None, clip=5.0)
    assert np.allclose(y1, want1, rtol=1e-10, atol=1e-10)
    want2 = zf.zfilter_batch(state, X[1777:], clip=5.0)           # continues from the carried state
    y2, st2 = filters.zfilter_scan(X[1777:], st1, clip=5.0)
    assert np.allclose(y2, want2, rtol=1e-10, atol=1e-10)
    assert st2[0] == 5000 and np.allclose(st2[1], state.M, rtol=1e-12) and np.allclose(st2[2], state.S, rtol=1e-10)


# ----------------------------------------------------------------------------- value function / PPO
def test_vf_lossgrad_golden(dev, golden):
    *_, pm, _, vf, _ = _oracle()
    dims = tuple(int(d) for d in golden["vf_dims"])
    lens = golden["vf_lens"]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    net = dev.DeviceNet(dims, 2)
    b = dev.DeviceBatch(dims[0] - 1, with_time_feature=True)
    b.set_obs(golden["vf_obs"]).set_paths(off, np.ones(len(lens), np.uint8), float(golden["vf_tl"]))
    b.set_vf_target(golden["vf_y"][:, 0])
    th32 = golden["vf_theta"].astype(np.float32)
    net.set_params(th32)
    pred = net.forward(b)
    assert relerr(pred, golden["vf_pred"]) < TOL
    ls, g = net.vf_lossgrad(b, 1e-3)
    assert np.allclose(ls, golden["vf_losses"], rtol=TOL)
    assert relerr(g, golden["vf_grad"]) < TOL


@pytest.mark.parametrize("tag", ["tg", "tc"])
@pytest.mark.parametrize("ptag", ["p0", "p1", "p2"])
def test_ppo_lossgrad_golden(dev, golden, tag, ptag):
    spec, head, th, ob, act, adv, oldp = _golden_case(golden, tag)
    _, _, pm, *_ = _oracle()
    net, batch = _bind(dev, spec.dims, head, ob, act, adv, oldp, th)
    klc, cutoff, rev = golden[f"{tag}_{ptag}_cfg"]
    pen, g, ls = net.ppo_lossgrad(batch, klc, cutoff, bool(rev))
    th32 = th.astype(np.float32)
    open_, og = pm.ppo_lossgrad(th32, spec, ob, act, adv, oldp, klc, cutoff, reverse_kl=bool(rev))
    ols, _, _ = pm.surr_kl_grads(th32, spec, ob, act, adv, oldp, ratio="lik", reverse_kl=bool(rev))
    dpen_dkl = klc + 2000.0 * (ols[1] > cutoff) * (ols[1] - cutoff)
    # the penalty amplifies the KL by up to 2000*(kl-cut): bound pen by 1e-5 relative error IN surr AND kl
    assert abs(pen - open_) < TOL * (abs(ols[0]) + abs(dpen_dkl) * ols[1]) + 1e-7
    assert relerr(g, og) < 2 * TOL
    assert relerr(g, golden[f"{tag}_{ptag}_grad"]) < 1e-4
    assert np.allclose(ls, golden[f"{tag}_{ptag}_losses"], rtol=1e-4, atol=1e-6)


# ----------------------------------------------------------------------------- register-chain kernels at scale
@pytest.mark.parametrize("name,N", [("hopper", 160_001), ("humanoid", 20_000), ("cat128", 9_999),
                                    ("hopper", 7), ("humanoid", 65), ("cartpole", 129)])
def test_chain_kernels_many_slabs(dev, name, N):
    """The chain kernels on batches that need several slabs per CTA (persistent loop, last slab and last chain tile
    partial, N not a multiple of 64): losses and gradient (mlp_chain.cu) and Fvp (the tcgen05 chain, mlp_fvp_tc.cu)
    against the oracle."""
    from modular_rl_b200 import synth
    _, _, pm, *_ = _oracle()
    dims, head, _ = SHAPES[name]
    wl = synth.Workload(name, dims, head, N, min(500, N), 17)   # tiny N: one mostly empty tile
    spec = pm.NetSpec(dims, pm.GAUSS if head == 0 else pm.CAT)

    def fwd(th, ob):
        _, z = pm.forward(th, spec, ob)
        return z if head == 0 else pm.softmax(z)
    d = synth.policy_batch(wl, fwd)
    theta = synth.perturb(d["theta"], 0.02, 9)
    net, batch = _bind(dev, spec.dims, head, d["ob"], d["act"], d["adv"], d["oldprob"], theta)
    args = (d["ob"], d["act"], d["adv"], d["oldprob"])
    assert np.allclose(net.losses(batch), pm.losses(theta, spec, *args), rtol=TOL, atol=2e-7)
    g, _ = net.policy_gradient(batch)
    assert relerr(g, pm.policy_gradient(theta, spec, *args)) < TOL
    v = np.random.default_rng(5).standard_normal(net.P).astype(np.float32)
    assert relerr(net.fvp(batch, v), pm.fisher_vector_product(theta, spec, d["ob"], v)) < TOL


@pytest.mark.parametrize("vdims,N", [((12, 64, 64, 1), 7001), ((30, 100, 50, 25, 1), 5000)])
def test_vf_lossgrad_chain_shapes(dev, vdims, N):
    """NnVf loss / gradient (core.py:613-617) on value nets that take the chain kernels (value head)."""
    from modular_rl_b200 import synth
    *_, pm, _, vf, _ = _oracle()
    rng = np.random.default_rng(3)
    off = np.asarray(synth.make_paths(N, 300, rng)[0], np.int64)
    ob = synth.make_obs(N, vdims[0] - 1, rng)
    y = rng.standard_normal(N)
    theta = synth.init_params(vdims, synth.VALUE, rng, last_scale=1.0)
    net = dev.DeviceNet(vdims, 2)
    b = dev.DeviceBatch(vdims[0] - 1, with_time_feature=True)
    b.set_obs(ob).set_paths(off, np.ones(len(off) - 1, np.uint8), 300.0)
    b.set_vf_target(y)
    net.set_params(theta)
    spec = pm.NetSpec(vdims, pm.VALUE)
    tidx = np.concatenate([np.arange(off[i + 1] - off[i]) for i in range(len(off) - 1)])
    x = np.concatenate([ob.astype(np.float64), (tidx / 300.0)[:, None]], axis=1)
    pred = net.forward(b)
    assert relerr(pred, vf.vf_forward(theta, spec, x)) < TOL
    ls, g = net.vf_lossgrad(b, 1e-3)
    _, og = vf.vf_lossgrad(theta, spec, x, y.reshape(-1, 1), l2coeff=1e-3)
    assert np.allclose(ls, vf.vf_losses(theta, spec, x, y.reshape(-1, 1), l2coeff=1e-3), rtol=TOL)
    assert relerr(g, og) < TOL


@pytest.mark.parametrize("name", ["walker", "cat128"])
@pytest.mark.parametrize("rev", [False, True])
def test_ppo_lossgrad_chain_shapes(dev, name, rev):
    """PpoLbfgsUpdater's penalised surrogate and gradient (ppo.py:35-49) on chain shapes, both KL directions."""
    spec, head, theta, d = _synth_case(name)
    _, _, pm, *_ = _oracle()
    net, batch = _bind(dev, spec.dims, head, d["ob"], d["act"], d["adv"], d["oldprob"], theta)
    args = (d["ob"], d["act"], d["adv"], d["oldprob"])
    klc, cutoff = 0.7, 1e-4
    pen, g, ls = net.ppo_lossgrad(batch, klc, cutoff, rev)
    open_, og = pm.ppo_lossgrad(theta, spec, *args, klc, cutoff, reverse_kl=rev)
    ols, _, _ = pm.surr_kl_grads(theta, spec, *args, ratio="lik", reverse_kl=rev)
    dpen_dkl = klc + 2000.0 * (ols[1] > cutoff) * (ols[1] - cutoff)
    assert abs(pen - open_) < TOL * (abs(ols[0]) + abs(dpen_dkl) * ols[1]) + 1e-7
    assert relerr(g, og) < 2 * TOL
