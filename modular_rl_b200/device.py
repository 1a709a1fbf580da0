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
