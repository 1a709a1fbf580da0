"""Thin object wrappers over the C ABI: a flattened batch of trajectories and an MLP resident
on one B200.  All arithmetic happens in libmrl_b200.so; arrays passed in may be numpy arrays
(host memory) or torch CUDA tensors (device memory, borrowed for the call)."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib as L
from . import parallel

_F = (np.dtype(np.float32), np.dtype(np.float64))


def _is_torch_cuda(x) -> bool:
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda") and x.is_cuda


def _arg(x, dtypes=None):
    """-> (keepalive, pointer, dtype_code, loc, shape)"""
    if x is None:
        return None, None, 0, L.HOST, ()
    if _is_torch_cuda(x):
        import torch
        codes = {torch.float32: L.F32, torch.float64: L.F64, torch.int32: L.I32, torch.int64: L.I64}
        x = x.contiguous()
        return x, C.c_void_p(x.data_ptr()), codes[x.dtype], L.DEVICE, tuple(x.shape)
    a = L.as_c(x, dtypes)
    return a, L.ptr(a), L.dtype_code(a), L.HOST, a.shape


def current_stream():
    """Raw cudaStream_t of torch's current stream if torch+CUDA is live, else the default stream."""
    try:
        import torch
        if torch.cuda.is_available() and torch.cuda.is_initialized():
            return C.c_void_p(torch.cuda.current_stream().cuda_stream)
    except Exception:
        pass
    return None


class Comm:
    """NCCL communicator owned by the library (one per process/GPU)."""

    def __init__(self, unique_id: bytes, rank: int, world: int, device: int):
        self._h = C.c_void_p()
        buf = C.create_string_buffer(unique_id, 128)
        L.check(L.lib().mrl_comm_create(C.byref(self._h), buf, rank, world, device))
        self.rank, self.world = rank, world
        self.p2p = False

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        L.check(L.lib().mrl_comm_unique_id(buf))
        return buf.raw

    def p2p_export(self, max_doubles: int) -> bytes:
        """Allocate this rank's NVLink receive buffer; returns its 64-byte CUDA IPC handle."""
        buf = C.create_string_buffer(64)
        L.check(L.lib().mrl_comm_p2p_export(self._h, int(max_doubles), buf))
        return buf.raw

    def p2p_connect(self, handles) -> None:
        """handles: the 64-byte handles of all ranks, in rank order (this rank's own included)."""
        blob = b"".join(handles)
        assert len(blob) == 64 * self.world
        L.check(L.lib().mrl_comm_p2p_connect(self._h, C.create_string_buffer(blob, len(blob))))

    def p2p_enable(self, on: bool = True) -> None:
        L.check(L.lib().mrl_comm_p2p_enable(self._h, int(on)))
        self.p2p = bool(on)

    def close(self):
        if self._h:
            L.lib().mrl_comm_destroy(self._h)
            self._h = C.c_void_p()


def _snapshot_device(stored: int) -> int:
    """Device a snapshot is rebuilt on: the loading rank's in data-parallel training, else the stored one."""
    return parallel.current_device() if parallel.context() is not None else stored


class DeviceBatch:
    def __init__(self, ob_dim: int, with_time_feature: bool = True, device: Optional[int] = None):
        """device None: this process's device (parallel.current_device(), GPU 0 in a single-process run)."""
        if device is None:
            device = parallel.current_device()
        self._h = C.c_void_p()
        L.check(L.lib().mrl_batch_create(C.byref(self._h), device, int(ob_dim), int(with_time_feature)))
        self.ob_dim, self.device, self.with_time = int(ob_dim), device, bool(with_time_feature)
        self.N = 0

    def __getstate__(self):
        # snapshots (run_pg.py:141-142) carry no batch data: an empty batch of the same shape comes back
        return dict(ob_dim=self.ob_dim, with_time=self.with_time, device=self.device)

    def __setstate__(self, d):
        self.__init__(d["ob_dim"], d["with_time"], _snapshot_device(d["device"]))

    def close(self):
        if getattr(self, "_h", None):
            L.lib().mrl_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_obs(self, ob, stream=None):
        keep, p, dt, loc, shape = _arg(ob, _F)
        assert len(shape) == 2 and shape[1] == self.ob_dim, shape
        L.check(L.lib().mrl_batch_set_obs(self._h, p, dt, shape[1], shape[0], loc, stream))
        self.N = int(shape[0])
        return self

    def set_paths(self, offsets, terminated, timestep_limit: float = 1.0, stream=None):
        off = np.ascontiguousarray(offsets, np.int64)
        term = np.ascontiguousarray(terminated, np.uint8)
        assert off.ndim == 1 and term.shape == (off.size - 1,)
        L.check(L.lib().mrl_batch_set_paths(self._h, L.ptr(off), L.ptr(term), int(term.size),
                                            float(timestep_limit), L.HOST, stream))
        self.n_paths = int(term.size)
        return self

    def set_policy_inputs(self, head: int, dout: int, act, adv, oldprob, stream=None):
        ka, pa, da, la, _ = _arg(act)
        kv, pv, dv, lv, _ = _arg(adv, _F)
        kp, pp, dp, lp, _ = _arg(oldprob, _F)
        locs = {l for l, x in ((la, act), (lv, adv), (lp, oldprob)) if x is not None}
        assert len(locs) == 1, "act/adv/oldprob must all be host or all device arrays"
        L.check(L.lib().mrl_batch_set_policy_inputs(self._h, head, dout, pa, da, pv, dv, pp, dp, locs.pop(),
                                                    stream))
        return self

    def set_vf_target(self, y, stream=None):
        k, p, dt, loc, _ = _arg(y, _F)
        L.check(L.lib().mrl_batch_set_vf_target(self._h, p, dt, loc, stream))
        return self

    def mix_vf_target(self, mixfrac: float, stream=None):
        L.check(L.lib().mrl_batch_mix_vf_target(self._h, float(mixfrac), stream))
        return self

    def set_global_n(self, n: int):
        L.check(L.lib().mrl_batch_set_global_n(self._h, int(n)))

    def time_index(self) -> np.ndarray:
        out = np.empty(self.N, np.int32)
        L.check(L.lib().mrl_batch_get_time_index(self._h, L.ptr(out), L.HOST, None))
        return out

    def gae(self, reward, baseline, gamma, lam, standardize=True, comm: Optional[Comm] = None,
            want_outputs=True, out=None, stream=None):
        """compute_advantage on the device.  reward/baseline: host arrays or CUDA tensors (both in the same
        place); baseline=None uses what predict_into_baseline left.  Returns (returns, advantages) as
        float64 arrays living where the inputs live (or (None, None) when want_outputs is False and no
        `out=(ret, adv)` buffers are given)."""
        kr, pr, dr, lr, _ = _arg(reward, _F)
        kb, pb, db, lb, _ = _arg(baseline, _F)
        assert baseline is None or lb == lr, "reward and baseline must live in the same place"
        ret = adv = None
        pret = padv = None
        if out is not None:
            ret, adv = out
        elif want_outputs:
            if lr == L.HOST:
                ret, adv = np.empty(self.N, np.float64), np.empty(self.N, np.float64)
            else:
                import torch
                ret = torch.empty(self.N, dtype=torch.float64, device=reward.device)
                adv = torch.empty_like(ret)
        if ret is not None:
            _, pret, _, lo, _ = _arg(ret)
            _, padv, _, _, _ = _arg(adv)
            assert lo == lr, "output buffers must live where the inputs live"
        L.check(L.lib().mrl_batch_gae(self._h, pr, dr, pb, db, float(gamma), float(lam), int(standardize),
                                      comm._h if comm else None, pret, padv, lr, stream))
        return ret, adv

    def gather_from(self, src: "DeviceBatch", idx, stream=None):
        """This batch <- rows idx of `src` (observations + policy side inputs), gathered on the device."""
        if _is_torch_cuda(idx):
            import torch
            assert idx.dtype == torch.int32
            idx = idx.contiguous()
            n, p, loc, keep = int(idx.numel()), C.c_void_p(idx.data_ptr()), L.DEVICE, idx
        else:
            keep = np.ascontiguousarray(idx, np.int32)
            n, p, loc = int(keep.size), L.ptr(keep), L.HOST
        L.check(L.lib().mrl_batch_gather(self._h, src._h, p, n, loc, stream))
        self.N = n
        return self

    def refresh_advantages(self, stream=None):
        L.check(L.lib().mrl_batch_refresh_advantages(self._h, stream))
        return self


class DeviceNet:
    def __init__(self, dims: Sequence[int], head: int, activation: str = "tanh", device: Optional[int] = None):
        if device is None:
            device = parallel.current_device()
        if activation not in L.ACTIVATIONS:
            raise ValueError(f"activation {activation!r} not supported (tanh, relu, sigmoid)")
        self.dims = [int(d) for d in dims]
        arr = (C.c_int * len(self.dims))(*self.dims)
        self._h = C.c_void_p()
        L.check(L.lib().mrl_net_create(C.byref(self._h), device, len(self.dims) - 1, arr, head,
                                       L.ACTIVATIONS[activation]))
        self.head, self.device, self.activation = head, device, activation
        self.P = int(L.lib().mrl_net_num_params(self._h))
        self.dout = self.dims[-1]
        self.theta_version = 0           # bumped by every call that can change the device parameters

    def __getstate__(self):
        # the device handle is rebuilt on load; theta travels as the flat float32 vector of SURVEY A.1.
        # A communicator is not part of a snapshot: re-attach it with set_comm after loading.
        return dict(dims=self.dims, head=self.head, activation=self.activation, device=self.device,
                    theta=self.get_params())

    def __setstate__(self, d):
        self.__init__(d["dims"], d["head"], d["activation"], _snapshot_device(d["device"]))
        self.set_params(d["theta"])

    def close(self):
        if getattr(self, "_h", None):
            L.lib().mrl_net_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_comm(self, comm: Optional[Comm]):
        L.check(L.lib().mrl_net_set_comm(self._h, comm._h if comm else None))

    def set_params(self, theta, stream=None):
        k, p, dt, loc, shape = _arg(theta, _F)
        assert int(np.prod(shape)) == self.P, (shape, self.P)
        self.theta_version += 1
        L.check(L.lib().mrl_net_set_params(self._h, p, dt, loc, stream))

    def get_params(self) -> np.ndarray:
        out = np.empty(self.P, np.float32)
        L.check(L.lib().mrl_net_get_params(self._h, L.ptr(out), L.HOST, None))
        return out

    def forward(self, batch: DeviceBatch, stream=None) -> np.ndarray:
        out = np.empty((batch.N, self.dout), np.float32)
        L.check(L.lib().mrl_net_forward(self._h, batch._h, L.ptr(out), L.HOST, stream))
        return out

    def predict_into_baseline(self, batch: DeviceBatch, stream=None):
        L.check(L.lib().mrl_net_predict_into_baseline(self._h, batch._h, stream))

    def losses(self, batch: DeviceBatch, stream=None) -> np.ndarray:
        out = np.zeros(3, np.float64)
        L.check(L.lib().mrl_net_losses(self._h, batch._h, L.ptr(out), stream))
        return out

    def policy_gradient(self, batch: DeviceBatch, stream=None):
        g = np.empty(self.P, np.float32)
        ls = np.zeros(3, np.float64)
        L.check(L.lib().mrl_net_policy_gradient(self._h, batch._h, L.ptr(g), L.HOST, L.ptr(ls), stream))
        return g, ls

    def fvp(self, batch: DeviceBatch, v, stream=None) -> np.ndarray:
        v = np.ascontiguousarray(v, np.float32)
        out = np.empty(self.P, np.float32)
        L.check(L.lib().mrl_net_fvp(self._h, batch._h, L.ptr(v), L.ptr(out), L.HOST, stream))
        return out

    def ppo_lossgrad(self, batch: DeviceBatch, kl_coeff, kl_cutoff, reverse_kl=False, want_grad=True,
                     stream=None):
        pen = C.c_double()
        g = np.empty(self.P, np.float64) if want_grad else None
        ls = np.zeros(3, np.float64)
        L.check(L.lib().mrl_net_ppo_lossgrad(self._h, batch._h, float(kl_coeff), float(kl_cutoff),
                                             int(bool(reverse_kl)), C.byref(pen), L.ptr(g), L.ptr(ls), stream))
        return pen.value, g, ls

    def ppo_sgd_step(self, minibatch: DeviceBatch, kl_coeff, kl_cutoff, stepsize, reverse_kl=False, beta1=0.9,
                     beta2=0.999, epsilon=1e-8, stream=None):
        """One PpoSgd `train` call on the device: loss + gradient on the minibatch, Adam step, no host sync."""
        self.theta_version += 1
        L.check(L.lib().mrl_net_ppo_sgd_step(self._h, minibatch._h, float(kl_coeff), float(kl_cutoff), int(bool(reverse_kl)),
                                             float(stepsize), float(beta1), float(beta2), float(epsilon), stream))

    def ppo_sgd_read(self, stream=None):
        """-> (mean [surr, kl, ent] of the minibatch losses since the last read, number of minibatches)"""
        ls = np.zeros(3, np.float64)
        cnt = C.c_longlong()
        L.check(L.lib().mrl_net_ppo_sgd_read(self._h, L.ptr(ls), C.byref(cnt), stream))
        return ls, int(cnt.value)

    def adam_reset(self, stream=None):
        L.check(L.lib().mrl_net_adam_reset(self._h, stream))

    def ppo_clip_lossgrad(self, batch: DeviceBatch, clip_eps, want_grad=True, stream=None):
        """PPO clipped surrogate on the whole batch -> (gradient float64 [P] or None, [surr, kl, ent, clipfrac])."""
        g = np.empty(self.P, np.float64) if want_grad else None
        ls = np.zeros(4, np.float64)
        L.check(L.lib().mrl_net_ppo_clip_lossgrad(self._h, batch._h, float(clip_eps), L.ptr(g), L.ptr(ls), stream))
        return g, ls

    def ppo_clip_sgd_step(self, minibatch: DeviceBatch, clip_eps, stepsize, beta1=0.9, beta2=0.999, epsilon=1e-8,
                          stream=None):
        """One PPO-clip minibatch step on the device: clipped gradient, Adam step (the moments of ppo_sgd_step),
        no host sync."""
        self.theta_version += 1
        L.check(L.lib().mrl_net_ppo_clip_sgd_step(self._h, minibatch._h, float(clip_eps), float(stepsize), float(beta1),
                                                  float(beta2), float(epsilon), stream))

    def vf_lossgrad(self, batch: DeviceBatch, l2coeff=1e-3, want_grad=True, stream=None):
        ls = np.zeros(3, np.float64)
        g = np.empty(self.P, np.float64) if want_grad else None
        L.check(L.lib().mrl_net_vf_lossgrad(self._h, batch._h, float(l2coeff), L.ptr(ls), L.ptr(g), stream))
        return ls, g

    def trpo_step(self, batch: DeviceBatch, cg_damping=1e-3, max_kl=1e-2, cg_iters=10, residual_tol=1e-10,
                  max_backtracks=10, accept_ratio=0.1, stream=None):
        cfg = L.TrpoCfg(cg_damping, max_kl, residual_tol, accept_ratio, cg_iters, max_backtracks)
        stats = np.zeros(6, np.float64)
        info = np.zeros(6, np.int32)
        self.theta_version += 1
        L.check(L.lib().mrl_net_trpo_step(self._h, batch._h, C.byref(cfg), L.ptr(stats), L.ptr(info), stream))
        keys = ("skipped", "success", "accepted_index", "cg_iters_run", "n_fvp", "n_loss_passes")
        return stats, dict(zip(keys, (int(v) for v in info)))

    def trpo_vectors(self):
        sd, fs, sc = np.empty(self.P), np.empty(self.P), np.zeros(4)
        L.check(L.lib().mrl_net_get_trpo_vectors(self._h, L.ptr(sd), L.ptr(fs), L.ptr(sc)))
        return sd, fs, dict(shs=sc[0], lm=sc[1], expected_improve_rate=sc[2], cg_rdotr=sc[3])


_user_env_ids = {}           # envs.DeviceEnv (bound to its shapes) -> library id


def rollout_env_id(kind) -> int:
    """The library's id of an envs.device_kind: a built-in's MRL_ENV_* code, or for a user environment (a bound
    envs.DeviceEnv) the id of its kernels, compiled with NVRTC on first use in the process."""
    if isinstance(kind, str):
        return L.DEVICE_ENVS[kind]
    if kind not in _user_env_ids:
        env = C.c_int()
        L.check(L.lib().mrl_rollout_env_compile(str(kind.name).encode(), kind.source.encode(), kind.ob_dim,
                                                kind.state_dim, L.CATEGORICAL if kind.categorical else L.GAUSS,
                                                kind.n_out, C.byref(env)))
        _user_env_ids[kind] = env.value
    return _user_env_ids[kind]


def rollout_env_log(kind) -> str:
    """The compiler's report (ptxas registers and spills of the six kernel instances) of a user environment."""
    buf = C.create_string_buffer(1 << 16)
    L.check(L.lib().mrl_rollout_env_log(rollout_env_id(kind), buf, len(buf)))
    return buf.value.decode(errors="replace")


def rollout_env_info(kind) -> dict:
    """mrl_rollout_env_info for an envs.py device kind: ob_dim, state_dim, categorical, n_out (the policy's outputs:
    K classes or the DiagGauss dimension d), act_dim (1 for Categorical, else d) and prob_dim (K, or 2d for
    [mean, std])."""
    ob, st, head, n_out = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    L.check(L.lib().mrl_rollout_env_info(rollout_env_id(kind), C.byref(ob), C.byref(st), C.byref(head), C.byref(n_out)))
    cat = head.value == L.CATEGORICAL
    return dict(ob_dim=ob.value, state_dim=st.value, categorical=cat, n_out=n_out.value,
                act_dim=1 if cat else n_out.value, prob_dim=n_out.value if cat else 2 * n_out.value)


class DeviceRollouts:
    """mrl_rollout_*: rounds of n_envs lockstep rollouts of a built-in environment, each round one kernel launch on
    the device (the policy forward, the action draws, the dynamics and both ZFilters included).  `env`: a built-in
    environment's id ("CartPole-v0", "Pendulum-v0", "Acrobot-v1", "MountainCar-v0", "MountainCarContinuous-v0") or
    instance, or a user environment with an envs.DeviceEnv (its id or instance)."""

    def __init__(self, env, n_envs: int, timestep_limit: int, device: Optional[int] = None):
        from .envs import device_kind
        kind = device_kind(env)
        if device is None:
            device = parallel.current_device()
        self._h = C.c_void_p()
        L.check(L.lib().mrl_rollout_create(C.byref(self._h), device, rollout_env_id(kind), int(n_envs), int(timestep_limit)))
        self.kind, self.n_envs, self.timestep_limit, self.device = kind, int(n_envs), int(timestep_limit), device
        info = rollout_env_info(kind)
        self.ob_dim, self.state_dim, self.categorical = info["ob_dim"], info["state_dim"], info["categorical"]
        self.act_dim, self.prob_dim = info["act_dim"], info["prob_dim"]

    @staticmethod
    def max_envs() -> int:
        return int(L.lib().mrl_rollout_max_envs())

    def close(self):
        if getattr(self, "_h", None):
            L.lib().mrl_rollout_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _filter_in(filt, size):
        """filt: None (identity) or (state (n, M, S), demean, destd, clip) -> (cfg, state in/out, pushed out)."""
        if filt is None:
            return None, None, None
        (n, M, S), demean, destd, clip = filt
        state = np.concatenate([[float(n)], np.asarray(M, np.float64).ravel(), np.asarray(S, np.float64).ravel()])
        assert state.size == 1 + 2 * size, (state.size, size)
        cfg = L.ZFilterCfg(1, int(bool(demean)), int(bool(destd)), float(clip or 0.0))
        return cfg, state, np.zeros_like(state)

    @staticmethod
    def _state_out(state, size):
        return None if state is None else (float(state[0]), state[1:1 + size].copy(), state[1 + size:].copy())

    def run(self, net: DeviceNet, seed: int, stochastic: bool = True, obfilter=None, rewfilter=None,
            want_states: bool = False, stream=None) -> dict:
        """One round.  obfilter / rewfilter: None (identity) or ((n, M, S), demean, destd, clip).  Returns the
        compacted path-major arrays and the filter states after the round plus those of this round's samples alone
        (ob_state, ob_pushed, rew_state, rew_pushed; None for an identity filter).  The arrays: lengths int32 and
        terminated uint8 per environment; per timestep observation float64 [T, ob_dim] (filtered), action (int32 [T]
        for a Categorical head, float32 [T, d] for DiagGauss), prob float32 [T, prob_dim] (the K probabilities, or
        [mean, std]), reward float64 [T] (raw) and with want_states the raw states float64 [T, state_dim]."""
        d = self.ob_dim
        ocfg, ost, opu = self._filter_in(obfilter, d)
        rcfg, rst, rpu = self._filter_in(rewfilter, 1)
        n = C.c_longlong()
        L.check(L.lib().mrl_rollout_run(self._h, net._h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(bool(stochastic)),
                                        C.byref(ocfg) if ocfg else None, L.ptr(ost), L.ptr(opu),
                                        C.byref(rcfg) if rcfg else None, L.ptr(rst), L.ptr(rpu),
                                        int(bool(want_states)), C.byref(n), stream))
        return self._read(self.n_envs, int(n.value), True, want_states, ost, opu, rst, rpu)

    def run_population(self, dims: Sequence[int], activation: str, thetas, seed: int, obfilter=None, rewfilter=None,
                       want_rows: bool = False, want_states: bool = False, stream=None) -> dict:
        """One round in which environment m acts deterministically with its own parameters thetas[m] (the
        cross-entropy method's population).  thetas: [M, ld] float32, numpy (host), a torch CUDA tensor or the
        DeviceRows of a DeviceSearch draw (both read in place); each row holds the Dense kernels and biases of the net `dims` in the reference's flat order (no logstd
        block), ld >= their count, M <= n_envs.  Filters as `run`.  Returns `returns` (float64 [M], the sum of each
        episode's raw rewards), lengths, terminated, the four filter states, and with want_rows the row arrays of `run`
        (prob: the K raw outputs of a Categorical head, [mean, 1] for DiagGauss).  Members act on the argmax of their
        raw outputs (first maximum) or on the raw output itself, which the environment clips."""
        dims = [int(x) for x in dims]
        if isinstance(thetas, DeviceRows):
            keep, th_ptr, loc = thetas, thetas.ptr, L.DEVICE
        elif _is_torch_cuda(thetas):
            import torch
            keep = thetas.to(torch.float32).contiguous()
            th_ptr, loc = C.c_void_p(keep.data_ptr()), L.DEVICE
        else:
            keep = np.ascontiguousarray(thetas, np.float32)
            th_ptr, loc = L.ptr(keep), L.HOST
        if keep.ndim != 2:
            raise ValueError("thetas must be [members, ld_theta], got shape %s" % (tuple(keep.shape),))
        M, ld = int(keep.shape[0]), int(keep.shape[1])
        ocfg, ost, opu = self._filter_in(obfilter, self.ob_dim)
        rcfg, rst, rpu = self._filter_in(rewfilter, 1)
        returns = np.empty(M, np.float64)
        n = C.c_longlong()
        arr = (C.c_int * len(dims))(*dims)
        L.check(L.lib().mrl_rollout_run_population(
            self._h, len(dims) - 1, arr, L.ACTIVATIONS[activation], th_ptr, ld, loc, M,
            int(seed) & 0xFFFFFFFFFFFFFFFF, C.byref(ocfg) if ocfg else None, L.ptr(ost), L.ptr(opu),
            C.byref(rcfg) if rcfg else None, L.ptr(rst), L.ptr(rpu), L.ptr(returns), int(bool(want_rows)),
            int(bool(want_states)), C.byref(n), stream))
        out = self._read(M, int(n.value), want_rows, want_states, ost, opu, rst, rpu)
        out["returns"] = returns
        return out

    def _read(self, n_envs, T, want_rows, want_states, ost, opu, rst, rpu) -> dict:
        d = self.ob_dim
        out = dict(lengths=np.empty(n_envs, np.int32), terminated=np.empty(n_envs, np.uint8))
        if want_rows:
            out.update(observation=np.empty((T, d), np.float64),
                       action=np.empty(T, np.int32) if self.categorical else np.empty((T, self.act_dim), np.float32),
                       prob=np.empty((T, self.prob_dim), np.float32),
                       reward=np.empty(T, np.float64))
        states = np.empty((T, self.state_dim), np.float64) if want_states else None
        L.check(L.lib().mrl_rollout_read(self._h, L.ptr(out["lengths"]), L.ptr(out["terminated"]),
                                         L.ptr(out.get("observation")), L.ptr(out.get("action")),
                                         L.ptr(out.get("prob")), L.ptr(out.get("reward")), L.ptr(states)))
        if want_states:
            out["states"] = states
        out["ob_state"], out["ob_pushed"] = self._state_out(ost, d), self._state_out(opu, d)
        out["rew_state"], out["rew_pushed"] = self._state_out(rst, 1), self._state_out(rpu, 1)
        return out


class DeviceRows:
    """The float32 candidate rows [M, ld] of a DeviceSearch, in the library's device memory (valid while the search
    lives).  `__cuda_array_interface__` lets torch read them in place: torch.as_tensor(rows, device="cuda")."""

    def __init__(self, owner, ptr: C.c_void_p, shape, device: int):
        self._owner, self.ptr, self.shape, self.ndim, self.device = owner, ptr, tuple(shape), 2, device

    @property
    def __cuda_array_interface__(self):
        return dict(shape=self.shape, typestr="<f4", data=(self.ptr.value, False), version=2, strides=None)


class DeviceSearch:
    """mrl_cem_search_*: the cross-entropy method's diagonal-Gaussian search distribution on the device.  P parameters,
    M candidates per generation (at most DeviceRollouts.max_envs()); rows padded to a multiple of 4 floats.  Mean and
    var are float64 [P]; `draw` writes the candidate rows and returns dev (host float64), `refit` takes the M scores
    (host array or CUDA tensor) and the elite count."""

    def __init__(self, P: int, M: int, device: Optional[int] = None):
        if device is None:
            device = parallel.current_device()
        self.P, self.M, self.device = int(P), int(M), device
        self.ld = (self.P + 3) // 4 * 4
        self._h = C.c_void_p()
        L.check(L.lib().mrl_cem_search_create(C.byref(self._h), device, self.P, self.M, self.ld))
        p, ld = C.c_void_p(), C.c_longlong()
        L.check(L.lib().mrl_cem_search_rows(self._h, C.byref(p), C.byref(ld)))
        self.rows = DeviceRows(self, p, (self.M, int(ld.value)), device)

    def close(self):
        if getattr(self, "_h", None):
            L.lib().mrl_cem_search_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _set(self, fn, x, stream):
        k, p, dt, loc, shape = _arg(x, (np.dtype(np.float64),))
        if dt != L.F64 or int(np.prod(shape)) != self.P:
            raise ValueError("need float64 [%d], got %s %s" % (self.P, tuple(shape), dt))
        L.check(fn(self._h, p, loc, stream))

    def set_mean(self, mean, stream=None):
        self._set(L.lib().mrl_cem_search_set_mean, mean, stream)

    def set_var(self, var, stream=None):
        self._set(L.lib().mrl_cem_search_set_var, var, stream)

    def get_mean(self, stream=None) -> np.ndarray:
        out = np.empty(self.P)
        L.check(L.lib().mrl_cem_search_get_mean(self._h, L.ptr(out), L.HOST, stream))
        return out

    def get_var(self, stream=None) -> np.ndarray:
        out = np.empty(self.P)
        L.check(L.lib().mrl_cem_search_get_var(self._h, L.ptr(out), L.HOST, stream))
        return out

    def draw(self, seed: int, extra_var: float, noise_left: float, stream=None) -> np.ndarray:
        """Rows of one generation into self.rows; returns dev = sqrt(var + extra_var * noise_left)."""
        dev = np.empty(self.P)
        L.check(L.lib().mrl_cem_search_draw(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF, float(extra_var),
                                            float(noise_left), L.ptr(dev), L.HOST, stream))
        return dev

    def refit(self, scores, keep: int, stream=None):
        k, p, dt, loc, shape = _arg(scores, (np.dtype(np.float64),))
        if dt != L.F64 or tuple(shape) != (self.M,):
            raise ValueError("scores must be float64 [%d], got %s" % (self.M, tuple(shape)))
        L.check(L.lib().mrl_cem_search_refit(self._h, p, loc, int(keep), stream))


def population_forward(dims: Sequence[int], activation: str, thetas, obs, device: int = 0) -> np.ndarray:
    """mrl_population_forward: out[m] = MLP_{thetas[m]}(obs[m]) for all members in one launch (linear last layer).
    thetas [M, P] holds Dense kernels and biases in the reference's flat order (no logstd block)."""
    th = np.ascontiguousarray(thetas, np.float32)
    ob = np.ascontiguousarray(obs, np.float32)
    dims = [int(d) for d in dims]
    M = th.shape[0]
    assert ob.shape == (M, dims[0]), (ob.shape, M, dims[0])
    out = np.empty((M, dims[-1]), np.float32)
    arr = (C.c_int * len(dims))(*dims)
    L.check(L.lib().mrl_population_forward(device, len(dims) - 1, arr, L.ACTIVATIONS[activation], L.ptr(th), th.shape[1],
                                           L.ptr(ob), M, L.ptr(out), L.HOST, None))
    return out


def gae_flat(reward, baseline, offsets, terminated, gamma, lam):
    """mrl_gae on host arrays -> (returns, advantages) float64."""
    r = L.as_c(reward, _F)
    b = L.as_c(baseline, _F)
    off = np.ascontiguousarray(offsets, np.int64)
    term = np.ascontiguousarray(terminated, np.uint8)
    N = r.shape[0]
    ret, adv = np.empty(N), np.empty(N)
    L.check(L.lib().mrl_gae(L.ptr(r), L.dtype_code(r), L.ptr(b), L.dtype_code(b), L.ptr(off), L.ptr(term),
                            int(term.size), N, float(gamma), float(lam), L.ptr(ret), L.ptr(adv), L.HOST, None))
    return ret, adv


def standardize(x):
    x = np.array(x, np.float64, copy=True)
    stats = np.zeros(3)
    L.check(L.lib().mrl_standardize(L.ptr(x), x.size, L.ptr(stats), L.HOST, None))
    return x, stats
