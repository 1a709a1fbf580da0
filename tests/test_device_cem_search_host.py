"""Host side of the cross-entropy method's device search (oracle/cem_search.py, cem._DeviceGaussianSearch,
cem.DEVICE_SEARCH, run_cem.py --device_search, the mrl_cem_search_* symbols): the oracle's elite rule, refit and
normals, the command-line and configuration rejections, and the seed each generation's draw and round share.  No
device is used."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SYMBOLS = ["mrl_cem_search_create", "mrl_cem_search_destroy", "mrl_cem_search_set_mean", "mrl_cem_search_set_var",
           "mrl_cem_search_get_mean", "mrl_cem_search_get_var", "mrl_cem_search_draw", "mrl_cem_search_rows",
           "mrl_cem_search_refit"]


def test_elite_rule_is_numpy_stable_argsort():
    from oracle import cem_search as ocs
    rng = np.random.default_rng(0)
    cases = [rng.integers(0, 5, 40).astype(np.float64),                         # many ties
             np.where(rng.random(50) < 0.1, np.nan, rng.integers(0, 3, 50)),      # ties and NaN
             np.array([0.0, -0.0, 1.0, -0.0, 0.0, np.nan, np.nan, -np.inf, np.inf]),
             rng.standard_normal(33)]
    for sc in cases:
        M = sc.size
        for keep in (0, 1, 2, 7, M - 1, M, M + 5):
            want = np.argsort(sc, kind="stable")[-keep:]
            np.testing.assert_array_equal(ocs.elite(sc, keep), want, err_msg="keep %d" % keep)
    assert ocs.elite(np.array([3.0, 3.0, 3.0]), 1).tolist() == [2]             # a tie goes to the higher index
    assert ocs.elite(np.array([np.nan, 5.0, np.nan]), 2).tolist() == [0, 2]     # NaN sorts last, in index order
    with pytest.raises(ValueError, match="keep = -1 is negative"):
        ocs.elite(np.zeros(4), -1)


def test_oracle_refit_equals_host_search_on_tie_free_scores():
    from modular_rl_b200.cem import _GaussianSearch
    from oracle import cem_search as ocs
    rng = np.random.default_rng(1)
    P, M, seed = 37, 60, 99
    host = _GaussianSearch(rng.standard_normal(P), 0.7, 0.3, 10.0)
    host.var = rng.random(P) + 0.1
    host.generation = 4
    dev = ocs.deviation(host.var, host.extra_var, host.noise_left())
    rows, dev2 = ocs.draw(host.mean, host.var, host.extra_var, host.noise_left(), seed, M)
    np.testing.assert_array_equal(dev, dev2)
    np.testing.assert_array_equal(dev, np.sqrt(host.var + host.extra_var * host.noise_left()))
    scores = rng.permutation(M).astype(np.float64) * 1.5
    for keep in (12, 1, M):
        mean, var = ocs.refit(host.mean, dev, seed, scores, keep)
        h = _GaussianSearch(host.mean, 1.0, 0.0, 1.0)
        h.refit(rows, scores, keep)
        np.testing.assert_array_equal(mean, h.mean)
        np.testing.assert_array_equal(var, h.var)


def test_normals_moments_and_stream():
    from oracle import cem_search as ocs
    z = ocs.normals(5, np.arange(2048), 64)
    assert z.shape == (2048, 64)
    n = z.size
    assert abs(z.mean()) < 4 / np.sqrt(n)
    assert abs(z.var() - 1.0) < 4 * np.sqrt(2.0 / n)
    assert abs((z ** 3).mean()) < 4 * np.sqrt(15.0 / n)
    assert abs((z ** 4).mean() - 3.0) < 4 * np.sqrt(96.0 / n)
    c = np.corrcoef(z[:, 0], z[:, 1])[0, 1]                  # the cos / sin halves of one pair are uncorrelated
    assert abs(c) < 4 / np.sqrt(2048)
    # a member's row does not depend on which other members are drawn; seeds and members give distinct streams
    np.testing.assert_array_equal(ocs.normals(5, [7, 3], 64), z[[7, 3]])
    assert not np.array_equal(ocs.normals(6, [7], 64), z[[7]])
    # odd P: the last pair's sine is dropped
    np.testing.assert_array_equal(ocs.normals(5, [1], 63), z[[1], :63])


def _parse(capsys, *args):
    import run_cem
    with pytest.raises(SystemExit) as e:
        run_cem.parse_cli(["--env", "CartPole-v0", "--agent", "modular_rl.agentzoo.DeterministicAgent"] + list(args))
    return e.value.code, capsys.readouterr().err


def test_parse_cli_rejections(capsys):
    code, err = _parse(capsys, "--device_search")
    assert code == 2 and "--device_search needs --device_envs" in err
    code, err = _parse(capsys, "--device_envs", "--device_search", "--elite_frac", "-0.2")
    assert code == 2 and "--elite_frac is -0.2" in err
    code, err = _parse(capsys, "--device_envs", "--device_search", "--parallel", "1")
    assert code == 2 and "--device_envs and --parallel 1" in err
    code, err = _parse(capsys, "--device_envs", "--device_search", "--batch_size", "4097")
    assert code == 2 and "at most 4096 environments" in err
    import run_cem
    args, _ = run_cem.parse_cli(["--env", "CartPole-v0", "--agent", "modular_rl.agentzoo.DeterministicAgent",
                                 "--device_envs", "--device_search"])
    assert args.device_search and args.device_envs


def test_help_names_the_flag():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "run_cem.py"), "--env", "CartPole-v0", "--agent",
                          "modular_rl.agentzoo.DeterministicAgent", "--help"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode == 0 and "--device_search" in out.stdout and "Philox" in out.stdout


def test_abi_symbols_exported():
    from modular_rl_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.lib()
    for name in SYMBOLS:
        assert hasattr(lib, name), name
        assert name in _lib.exported_symbols(), name
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], check=True, capture_output=True,
                         text=True).stdout
    exported = {f[-1] for f in (line.split() for line in out.splitlines()) if f}
    assert set(SYMBOLS) <= exported


class _FlatAgent(object):
    class policy:
        class net:
            device = 0

    def __init__(self, dim):
        self.th = np.zeros(dim)

    def get_flat(self):
        return self.th

    def set_from_flat(self, th):
        self.th = np.array(th)


def test_configuration_rejections(monkeypatch):
    from modular_rl_b200 import cem
    monkeypatch.setattr(cem, "DEVICE_SEARCH", True)
    with pytest.raises(ValueError, match="set both"):
        cem.run_cem_algorithm("env", _FlatAgent(3), dict(batch_size=4, n_iter=1))
    monkeypatch.setattr(cem, "DEVICE_ENVS", True)
    with pytest.raises(ValueError, match="elite_frac = -0.5 is negative"):
        cem.run_cem_algorithm("env", _FlatAgent(3), dict(batch_size=4, n_iter=1, elite_frac=-0.5))


def test_draw_and_round_share_the_generation_seed(monkeypatch):
    """A stand-in for the device search: generation g draws with seed + g, its round gets the same seed, numpy's
    generator is untouched, and the info dict carries host float64 th and std."""
    from modular_rl_b200 import cem, device
    draws, rounds = [], []

    class FakeSearch(object):
        def __init__(self, P, M, device=None):
            self.P, self.M, self.rows = P, M, "rows"
            self.mean = None

        def set_mean(self, m):
            self.mean = np.array(m, np.float64)

        def set_var(self, v):
            self.var = np.array(v, np.float64)

        def draw(self, seed, extra_var, noise_left):
            draws.append((seed, noise_left))
            return np.sqrt(self.var + extra_var * noise_left)

        def refit(self, scores, keep):
            assert scores.dtype == np.float64 and scores.shape == (self.M,) and keep == 4
            self.mean = self.mean + 1.0

        def get_mean(self):
            return self.mean.copy()

    def fake_round(env, agent, ths, timestep_limit, seed):
        assert ths == "rows"
        rounds.append(seed)
        return np.arange(20, dtype=np.float64)
    monkeypatch.setattr(device, "DeviceSearch", FakeSearch)
    monkeypatch.setattr(cem, "DEVICE_ENVS", True)
    monkeypatch.setattr(cem, "DEVICE_SEARCH", True)
    monkeypatch.setattr(cem, "evaluate_population_device", fake_round)
    np.random.seed(3)
    state = np.random.get_state()[1].copy()
    agent = _FlatAgent(6)
    infos = []
    cem.run_cem_algorithm("env", agent, dict(batch_size=20, n_iter=3, timestep_limit=30, seed=11, extra_std=0.5,
                                             std_decay_time=2.0), callback=infos.append)
    assert [s for s, _ in draws] == rounds == [11, 12, 13]
    assert [n for _, n in draws] == [1.0, 0.5, 0]
    assert np.array_equal(np.random.get_state()[1], state)
    for g, info in enumerate(infos):
        assert info["th"].dtype == np.float64 and info["std"].dtype == np.float64 and info["ys"].dtype == np.float64
        np.testing.assert_array_equal(info["th"], np.full(6, g + 1.0))
    np.testing.assert_array_equal(agent.get_flat(), infos[-1]["th"])
