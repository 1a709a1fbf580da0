"""The delta_1 hand-off to the layer-1 gradient GEMM, checked on every kernel that writes it.

The reverse sweep stores delta_1 (the layer-1 error) in `DG` as raw fp32 in the UMMA K-major order, and
l1_grad_tc_kernel splits it into the (hi, lo) TF32 pair in shared memory.  Four kernels write `DG`:
chain_bwd_kernel (gradient of the instantiated chain shapes, e.g. Humanoid), fvp_tc_kernel (Fisher-vector
product of tanh nets), lw_dg_kernel (nets too wide for the fused kernels, covered by test_gpu_wide_nets.py)
and mid_backward_kernel (everything else).  Each case below routes the gradient and the Fvp to a different
pair of the other three and compares the layer-1 weight and bias blocks with the float64
oracle.  N is not a multiple of 8 or 128, so the last 8-timestep group is partly padding.  The calls are
interleaved (gradient, Fvp, gradient, Fvp): each writer must overwrite everything the other left in the
shared buffer, so the repeated calls have to be bit-identical.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from conftest import relerr  # noqa: E402

TOL = 1e-5   # tests/test_gpu_parity.py

CASES = {
    # gradient: chain_bwd_kernel (104-56-32-24 chain shape), Fvp: fvp_tc_kernel
    "humanoid": ((376, 100, 50, 25, 17), "tanh", 2021),
    # gradient: mid_backward_kernel (no chain shape with two hidden layers this wide), Fvp: fvp_tc_kernel
    "two_hidden": ((376, 100, 50, 17), "tanh", 1237),
    # gradient and Fvp: mid_backward_kernel (the chain and the tcgen05 Fvp are tanh only)
    "relu_humanoid": ((376, 100, 50, 25, 17), "relu", 1509),
}


def _case(name):
    from modular_rl_b200 import synth
    from oracle import policy_math as pm
    dims, act, N = CASES[name]
    wl = synth.Workload(name, dims, synth.GAUSS, N, 200, 17)
    spec = pm.NetSpec(dims, pm.GAUSS, act)
    data = synth.policy_batch(wl, lambda th, ob: pm.forward(th, spec, ob)[1])
    return spec, synth.perturb(data["theta"], 0.02, 9), data


def _layer1(spec, x):
    from oracle import policy_math as pm
    sl = {name: (a, b) for name, _, a, b in pm.param_slices(spec)}
    return x[slice(*sl["W1"])], x[slice(*sl["b1"])]


@pytest.mark.parametrize("name", list(CASES))
def test_layer1_gradient_and_fvp(name):
    from modular_rl_b200 import _lib
    from modular_rl_b200.device import DeviceBatch, DeviceNet
    from oracle import policy_math as pm
    _lib.lib()
    spec, theta, d = _case(name)
    N = d["ob"].shape[0]
    assert N % 8 != 0
    net = DeviceNet(spec.dims, 0, spec.activation)
    batch = DeviceBatch(spec.dims[0], with_time_feature=True)
    batch.set_obs(d["ob"])
    batch.set_paths(np.array([0, N], np.int64), np.array([1], np.uint8), 1000.0)
    batch.set_policy_inputs(0, spec.dims[-1], d["act"], d["adv"], d["oldprob"])
    net.set_params(theta)
    v = np.random.default_rng(4).standard_normal(net.P).astype(np.float32)

    g1, _ = net.policy_gradient(batch)
    f1 = net.fvp(batch, v)
    g2, _ = net.policy_gradient(batch)
    f2 = net.fvp(batch, v)
    assert np.array_equal(g1, g2)
    assert np.array_equal(f1, f2)

    og = pm.policy_gradient(theta, spec, d["ob"], d["act"], d["adv"], d["oldprob"])
    of = pm.fisher_vector_product(theta, spec, d["ob"], v)
    for got, want in ((g1, og), (f1, of)):
        (gW, gb), (wW, wb) = _layer1(spec, got), _layer1(spec, want)
        assert relerr(gW, wW) < TOL, relerr(gW, wW)
        assert relerr(gb, wb) < TOL, relerr(gb, wb)
        assert relerr(got, want) < TOL
