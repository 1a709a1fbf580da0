#!/usr/bin/env python
"""Per-kernel timing of a few Fisher-vector products on a Humanoid-shaped batch (experiment helper)."""
import ctypes as C, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from modular_rl_b200 import _lib as L, synth
from modular_rl_b200.device import DeviceBatch, DeviceNet

N = int(sys.argv[1]) if len(sys.argv) > 1 else 262144
dims = (376, 100, 50, 25, 17)
rng = np.random.default_rng(0)
ob = synth.make_obs(N, dims[0], rng)
theta = synth.init_params(dims, synth.GAUSS, rng)
net = DeviceNet(dims, synth.GAUSS)
batch = DeviceBatch(dims[0], with_time_feature=False)
batch.set_obs(ob)
net.set_params(theta)
v = rng.standard_normal(net.P).astype(np.float32)
for _ in range(2):
    net.fvp(batch, v)
lib = L.lib()
lib.mrl_profile_enable(1)
for _ in range(5):
    f = net.fvp(batch, v)
nk = lib.mrl_profile_kinds()
ms = (C.c_double * nk)(); cnt = (C.c_longlong * nk)()
lib.mrl_profile_read(ms, cnt)
lib.mrl_profile_kind_name.restype = C.c_char_p
print("N=%d |" % N,
      "  ".join("%s %.4f" % (lib.mrl_profile_kind_name(k).decode(), ms[k] / cnt[k]) for k in range(nk) if cnt[k]),
      "| |fvp| %.6e" % float(np.linalg.norm(f)))
