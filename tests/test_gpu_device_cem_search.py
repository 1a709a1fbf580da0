"""The cross-entropy method's search on the device (cem_search.cu, mrl_cem_search_*, device.DeviceSearch,
cem._DeviceGaussianSearch, run_cem.py --device_search): draws against oracle/cem_search.py, determinism, the refit
and its elite rule on device-scored and crafted populations, and whole runs of run_cem_algorithm and run_cem.py."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

DIMS = [4, 64, 64, 2]
P = sum(DIMS[i] * DIMS[i + 1] + DIMS[i + 1] for i in range(len(DIMS) - 1))      # 4610


def _rows(search):
    import torch
    return torch.as_tensor(search.rows, device="cuda").cpu().numpy()


def _search(M, P=P, seed=0):
    from modular_rl_b200.device import DeviceSearch
    rng = np.random.default_rng(seed)
    s = DeviceSearch(P, M)
    mean, var = rng.standard_normal(P) * 0.5 + 0.25, rng.random(P) * 0.8 + 0.05
    s.set_mean(mean)
    s.set_var(var)
    return s, mean, var


def _ulp_distance(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


def test_draw_against_oracle():
    from oracle import cem_search as ocs
    M, seed = 4096, 20261022
    s, mean, var = _search(M)
    assert s.ld == 4612 and s.rows.shape == (M, 4612)
    dev = s.draw(seed, 0.09, 0.75)
    rows64, odev = ocs.draw(mean, var, 0.09, 0.75, seed, M)
    np.testing.assert_array_equal(dev, odev)                                       # bit-equal
    got = _rows(s)
    assert np.all(got[:, P:] == 0.0)                                               # padding columns
    d = _ulp_distance(got[:, :P], rows64.astype(np.float32))
    assert d.max() <= 2, (int(d.max()), float(np.mean(d > 0)))
    # odd P, one member: the last pair writes only its first column
    s1, m1, v1 = _search(1, P=7, seed=2)
    dev1 = s1.draw(5, 0.0, 0)
    r1, od1 = ocs.draw(m1, v1, 0.0, 0, 5, 1)
    np.testing.assert_array_equal(dev1, od1)
    g1 = _rows(s1)
    assert g1.shape == (1, 8) and g1[0, 7] == 0.0
    assert _ulp_distance(g1[:, :7], r1.astype(np.float32)).max() <= 2


def test_same_seed_same_bits():
    s, mean, var = _search(512)
    s.draw(7, 0.0, 1.0)
    a = _rows(s)
    s.draw(7, 0.0, 1.0)
    b = _rows(s)
    s.draw(8, 0.0, 1.0)
    c = _rows(s)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.mean(a[:, :P] == c[:, :P]) < 1e-3
    # the next generation draws from the refitted distribution with the next seed: different rows
    s.refit(np.arange(512, dtype=np.float64), 100)
    s.draw(8, 0.0, 1.0)
    assert np.mean(_rows(s)[:, :P] == c[:, :P]) < 1e-3


def _check_refit(s, mean, dev, seed, scores, keep):
    """Within 1e-12 of the oracle relative to each column's scale: |mean| + dev for the mean, var + dev^2 for the
    variance (a mean that happens to lie near 0 still carries the rounding of values of size dev)."""
    from oracle import cem_search as ocs
    scores = np.asarray(scores, np.float64)
    s.refit(scores, keep)
    want_mean, want_var = ocs.refit(mean, dev, seed, scores, keep)
    got_mean, got_var = s.get_mean(), s.get_var()
    err_mean = np.abs(got_mean - want_mean) / (np.abs(want_mean) + dev)
    err_var = np.abs(got_var - want_var) / (want_var + dev * dev)
    assert err_mean.max() <= 1e-12 and err_var.max() <= 1e-12, (err_mean.max(), err_var.max())
    return got_mean, got_var


def test_refit_on_device_scored_population():
    """Candidates scored by a CartPole population round reading the rows in place; integer scores with many ties."""
    from modular_rl_b200.device import DeviceRollouts
    M, seed = 1000, 31
    s, mean, var = _search(M, seed=4)
    dev = s.draw(seed, 0.0, 0)
    ro = DeviceRollouts("CartPole-v0", M, 200)
    out = ro.run_population(DIMS, "tanh", s.rows, seed)
    scores = out["returns"]
    assert len(np.unique(scores)) < M // 2                                     # ties are the normal case
    host = ro.run_population(DIMS, "tanh", _rows(s), seed)                    # the same rows read from the host
    assert np.array_equal(host["returns"], scores)
    _check_refit(s, mean, dev, seed, scores, int(round(M * 0.2)))


@pytest.mark.parametrize("keep", [1, 50, 200, 0, 4096, 5000])
def test_refit_crafted_scores(keep):
    from oracle import cem_search as ocs
    M, seed = 4096, 77
    s, mean, var = _search(M, seed=keep + 1)
    dev = s.draw(seed, 0.01, 0.5)
    rng = np.random.default_rng(keep)
    scores = rng.integers(0, 40, M).astype(np.float64)
    scores[rng.integers(0, M, 3)] = np.nan
    scores[rng.integers(0, M, 5)] = -0.0
    scores[rng.integers(0, M, 5)] = 0.0
    got_mean, got_var = _check_refit(s, mean, dev, seed, scores, keep)
    # a wrong elite set misses by far more than the tolerance: shifting the elite by one member shows it
    n = M if keep in (0,) or keep > M else keep
    if n < M:
        wrong = ocs.elite(scores, n + 1)[:-1]
        best = ocs.candidates(mean, dev, seed, wrong)
        assert np.max(np.abs(best.mean(axis=0) - got_mean) / np.abs(got_mean)) > 1e-9


def test_rejections():
    from modular_rl_b200 import _lib as L
    from modular_rl_b200.device import DeviceSearch
    lib = L.lib()
    h = C.c_void_p()
    with pytest.raises(RuntimeError, match="M = 4097; a generation is one rollout round of 1..4096 members"):
        L.check(lib.mrl_cem_search_create(C.byref(h), 0, 10, 4097, 12))
    with pytest.raises(RuntimeError, match="M = 0"):
        L.check(lib.mrl_cem_search_create(C.byref(h), 0, 10, 0, 12))
    with pytest.raises(RuntimeError, match="ld = 10; rows need ld >= P = 10 and a multiple of 4"):
        L.check(lib.mrl_cem_search_create(C.byref(h), 0, 10, 8, 10))
    with pytest.raises(RuntimeError, match="ld = 8; rows need ld >= P = 10"):
        L.check(lib.mrl_cem_search_create(C.byref(h), 0, 10, 8, 8))
    with pytest.raises(RuntimeError, match="P = 0"):
        L.check(lib.mrl_cem_search_create(C.byref(h), 0, 0, 8, 4))
    s = DeviceSearch(10, 8)
    sc = np.zeros(8)
    with pytest.raises(RuntimeError, match="no generation has been drawn"):
        s.refit(sc, 2)
    s.set_mean(np.zeros(10))
    s.set_var(np.ones(10))
    s.draw(1, 0.0, 0)
    with pytest.raises(RuntimeError, match="keep = -1 is negative"):
        s.refit(sc, -1)
    with pytest.raises(RuntimeError, match="loc = 2 \\(MRL_HOST or MRL_DEVICE\\)"):
        L.check(lib.mrl_cem_search_refit(s._h, L.ptr(sc), 2, 2, None))
    with pytest.raises(RuntimeError, match="loc = MRL_DEVICE but scores is not device memory of device 0"):
        L.check(lib.mrl_cem_search_refit(s._h, L.ptr(sc), L.DEVICE, 2, None))
    out = np.zeros(10)
    with pytest.raises(RuntimeError, match="loc = MRL_DEVICE but mean is not device memory of device 0"):
        L.check(lib.mrl_cem_search_get_mean(s._h, L.ptr(out), L.DEVICE, None))
    with pytest.raises(ValueError, match="scores must be float64 \\[8\\]"):
        s.refit(np.zeros(7), 2)
    with pytest.raises(ValueError, match="need float64 \\[10\\]"):
        s.set_mean(np.zeros(9))


def test_device_scores_and_setters():
    """Scores, mean and var handed over as CUDA tensors give what the host arrays give."""
    import torch
    s, mean, var = _search(300, P=50, seed=9)
    t, _, _ = _search(300, P=50, seed=9)
    scores = np.random.default_rng(3).integers(0, 9, 300).astype(np.float64)
    for x in (s, t):
        x.draw(5, 0.0, 0)
    s.refit(scores, 60)
    t.refit(torch.from_numpy(scores).cuda(), 60)
    assert np.array_equal(s.get_mean(), t.get_mean()) and np.array_equal(s.get_var(), t.get_var())
    t.set_mean(torch.from_numpy(mean).cuda())
    t.set_var(torch.from_numpy(var).cuda())
    assert np.array_equal(t.get_mean(), mean) and np.array_equal(t.get_var(), var)


def test_run_cem_algorithm_device_search(monkeypatch):
    from modular_rl_b200 import _lib as L, agentzoo, cem, device, envs
    monkeypatch.setattr(cem, "DEVICE_ENVS", True)
    monkeypatch.setattr(cem, "DEVICE_SEARCH", True)
    lib = L.lib()
    thetas, stamps, launches = [], [], []

    def counted(name, fn):
        def call(*a, **k):
            n0 = lib.mrl_launch_count()
            out = fn(*a, **k)
            launches.append((name, lib.mrl_launch_count() - n0))
            return out
        return call
    monkeypatch.setattr(cem._DeviceGaussianSearch, "draw", counted("draw", cem._DeviceGaussianSearch.draw))
    monkeypatch.setattr(cem._DeviceGaussianSearch, "refit", counted("refit", cem._DeviceGaussianSearch.refit))
    monkeypatch.setattr(cem, "evaluate_population_device", counted("round", cem.evaluate_population_device))
    orig_run = device.DeviceRollouts.run_population

    def run_population(self, dims, activation, ths, *a, **k):
        thetas.append(type(ths))
        return orig_run(self, dims, activation, ths, *a, **k)
    monkeypatch.setattr(device.DeviceRollouts, "run_population", run_population)
    env = envs.CartPoleEnv()
    np.random.seed(0)
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[64, 64]))
    state = np.random.get_state()
    infos = []
    stamps.append(lib.mrl_launch_count())

    def callback(info):
        infos.append(info)
        stamps.append(lib.mrl_launch_count())
    cem.run_cem_algorithm(env, agent, dict(batch_size=64, n_iter=6, timestep_limit=200, seed=0), callback=callback)
    assert len(infos) == 6
    assert launches == [("draw", 1), ("round", 1), ("refit", 2)] * 6       # draw, the round, rank + refit
    per_generation = np.diff(stamps)[1:]                  # + the agent's set_from_flat between generations
    assert len(set(per_generation.tolist())) == 1 and per_generation[0] <= 8, per_generation
    assert thetas == [device.DeviceRows] * 6
    after = np.random.get_state()
    assert after[0] == state[0] and np.array_equal(after[1], state[1]) and after[2:] == state[2:]
    for info in infos:
        assert info["ys"].dtype == info["th"].dtype == info["std"].dtype == np.float64
        assert info["th"].shape == info["std"].shape == (P,) and info["ys"].shape == (64,)
    assert max(info["ymean"] for info in infos[1:]) > infos[0]["ymean"]
    np.testing.assert_array_equal(agent.get_flat(), infos[-1]["th"].astype(np.float32))


def test_pendulum_device_search(monkeypatch):
    from modular_rl_b200 import agentzoo, cem, envs
    monkeypatch.setattr(cem, "DEVICE_ENVS", True)
    monkeypatch.setattr(cem, "DEVICE_SEARCH", True)
    env = envs.PendulumEnv()
    agent = agentzoo.DeterministicAgent(env.observation_space, env.action_space, dict(hid_sizes=[16]))
    infos = []
    cem.run_cem_algorithm(env, agent, dict(batch_size=33, n_iter=3, timestep_limit=50, extra_std=0.1),
                          callback=infos.append)
    assert len(infos) == 3 and all(np.all(np.isfinite(i["ys"])) and np.all(np.isfinite(i["th"])) for i in infos)


def test_run_cem_cli_device_search(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "run_cem.py"), "--env", "CartPole-v0", "--agent",
                          "modular_rl.agentzoo.DeterministicAgent", "--device_envs", "--device_search", "--n_iter", "2",
                          "--batch_size", "40", "--snapshot_every", "2", "--outfile", str(tmp_path / "c.h5")],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "device_search: candidates drawn and refitted on the device" in out.stdout
    assert os.listdir(str(tmp_path / "c.h5.dir"))
