"""Observation / reward filters with the reference's interface (filters.py).

``ZFilter.__call__`` keeps the reference's per-sample semantics on the host (one call per
environment step).  ``ZFilter.filter_batch`` / ``zfilter_scan`` run the same recurrence for a
block of consecutive samples on the device: sample t is normalised with statistics that include
samples 0..t and everything pushed before (SURVEY 3.6).
"""
import ctypes as C

import numpy as np

from . import _lib as L
from .running_stat import RunningStat


def zfilter_scan(X, state=None, demean=True, destd=True, clip=10.0, out_dtype=np.float64):
    """Device scan.  X [N, d]; state = (n, M[d], S[d]) or None -> (Y [N, d], new_state)."""
    X = L.as_c(X, (np.dtype(np.float64), np.dtype(np.float32)))
    assert X.ndim == 2
    N, d = X.shape
    if state is None:
        n, M, S = 0.0, np.zeros(d), np.zeros(d)
    else:
        n, M, S = float(state[0]), np.array(state[1], np.float64).reshape(d), np.array(state[2], np.float64).reshape(d)
    Y = np.empty((N, d), out_dtype)
    n_c = C.c_double(n)
    L.check(L.lib().mrl_zfilter_scan(L.ptr(X), L.dtype_code(X), N, d, C.byref(n_c), L.ptr(M), L.ptr(S),
                                     int(bool(demean)), int(bool(destd)), float(clip or 0.0), L.ptr(Y),
                                     L.dtype_code(Y), L.HOST, None))
    return Y, (n_c.value, M, S)


class ZFilter(object):
    """y = (x-mean)/std using running estimates of mean,std (filters.py:17-40)."""

    pushed = None       # RunningStat of the samples pushed since start_round() (data-parallel training), else None

    def __init__(self, shape, demean=True, destd=True, clip=10.0):
        self.demean = demean
        self.destd = destd
        self.clip = clip
        self.rs = RunningStat(shape)

    def __call__(self, x, update=True):
        if update:
            self.rs.push(x)
            if self.pushed is not None:
                self.pushed.push(x)
        if self.demean:
            x = x - self.rs.mean
        if self.destd:
            x = x / (self.rs.std + 1e-8)
        if self.clip:
            x = np.clip(x, -self.clip, self.clip)
        return x

    def filter_batch(self, X):
        """N consecutive __call__(x, update=True) on the device; the running state advances."""
        X = np.asarray(X)
        shp = self.rs.shape
        Y, st = zfilter_scan(X.reshape(X.shape[0], -1), self.rs.state(), self.demean, self.destd, self.clip)
        self.rs.set_state(*st)
        if self.pushed is not None:
            _, st = zfilter_scan(X.reshape(X.shape[0], -1), self.pushed.state(), False, False, 0.0)
            self.pushed.set_state(*st)
        return Y.reshape((X.shape[0],) + tuple(shp))

    def start_round(self):
        """Also record the samples pushed from now on in `pushed`, a state of their own: data-parallel training
        merges every rank's samples of an iteration into one state (parallel.sync_rollouts)."""
        self.pushed = RunningStat(self.rs.shape)

    def output_shape(self, input_space):
        return input_space.shape


class Composition(object):
    def __init__(self, fs):
        self.fs = fs

    def __call__(self, x, update=True):
        for f in self.fs:
            x = f(x)
        return x

    def output_shape(self, input_space):
        out = input_space.shape
        for f in self.fs:
            out = f.output_shape(out)
        return out


class Flatten(object):
    def __call__(self, x, update=True):
        return x.ravel()

    def output_shape(self, input_space):
        return (int(np.prod(input_space.shape)),)


class Ind2OneHot(object):
    def __init__(self, n):
        self.n = n

    def __call__(self, x, update=True):
        out = np.zeros(self.n)
        out[x] = 1
        return out

    def output_shape(self, input_space):
        return (input_space.n,)
