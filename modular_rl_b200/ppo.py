"""PPO with a penalised KL and L-BFGS (ppo.py:3-112) on the B200 path.

pensurr = surr + kl_coeff*kl + 1000*(kl > 2*kl_target)*(kl - 2*kl_target)^2 with
surr = -(1/N) sum (p/oldp)*adv (likelihood ratio, ppo.py:35-36,47).  L-BFGS-B stays scipy's routine
on the host - the one the reference calls (ppo.py:85) - and each of its evaluations is one
set_params + fused forward / reverse sweep on the device (mrl_net_ppo_lossgrad), where the chain-rule
coefficient of the KL term is computed from the batch-wide KL without a host round trip.

PpoSgdUpdater (ppo.py:115-258, SURVEY 8f rank 2) reuses the same device loss/gradient entry point on
minibatches of 128 gathered rows; Adam (adam_updates, ppo.py:231-258) runs on the host in float32 like the
reference's floatX shared variables.
"""
from collections import OrderedDict

import numpy as np
import scipy.optimize

from . import _lib as L
from . import parallel
from .core import EzFlat, concat
from .device import DeviceBatch
from .misc_utils import EzPickle, update_default_config, zipsame


class PpoLbfgsUpdater(EzFlat, EzPickle):
    options = [
        ("kl_target", float, 1e-2, "Desired KL divergence between old and new policy"),
        ("maxiter", int, 25, "Maximum number of iterations"),
        ("reverse_kl", int, 0, "kl[new, old] instead of kl[old, new]"),
        ("do_split", int, 0, "Do train/test split on batches"),
    ]

    def __init__(self, stochpol, usercfg):
        EzPickle.__init__(self, stochpol, usercfg)
        cfg = update_default_config(self.options, usercfg)
        print("PPOUpdater", cfg)
        self.stochpol = stochpol
        self.cfg = cfg
        self.kl_coeff = 1.0
        EzFlat.__init__(self, stochpol.net)
        self.loss_names = ["surr", "kl", "ent"]
        self._train = DeviceBatch(stochpol.dims[0], with_time_feature=True)
        self._test = DeviceBatch(stochpol.dims[0], with_time_feature=True)

    def _bind(self, batch, ob, act, adv, prob):
        batch.set_obs(np.asarray(ob).reshape(len(ob), -1))
        batch.set_policy_inputs(self.stochpol.probtype.head, self.stochpol.dims[-1], act, adv, prob)
        return batch

    def _losses(self, batch):
        """[surr, kl, ent] with the configured KL direction (ppo.py:39-43,57)."""
        _, _, ls = self.stochpol.net.ppo_lossgrad(batch, 0.0, 1e300, self.cfg["reverse_kl"], want_grad=False)
        return ls

    def __call__(self, paths):
        cfg = self.cfg
        net = self.stochpol.net
        prob_np = concat([path["prob"] for path in paths])
        ob_no = concat([path["observation"] for path in paths])
        action_na = concat([path["action"] for path in paths])
        advantage_n = concat([path["advantage"] for path in paths])

        N = ob_no.shape[0]
        train_stop = int(0.75 * N) if cfg["do_split"] else N
        tr, te = slice(0, train_stop), slice(train_stop, None)
        train = self._bind(self._train, ob_no[tr], action_na[tr], advantage_n[tr], prob_np[tr])
        n_total = parallel.global_timesteps(paths)
        if n_total is not None and not cfg["do_split"]:
            train.set_global_n(n_total)          # this rank's shard of the batch of all ranks
        kl_cutoff = cfg["kl_target"] * 2.0

        thprev = self.get_params_flat().astype(np.float64)

        def lossandgrad(th):
            self.set_params_flat(th)
            l, g, _ = net.ppo_lossgrad(train, self.kl_coeff, kl_cutoff, cfg["reverse_kl"])
            return (l, g)

        train_losses_before = self._losses(train)
        if cfg["do_split"]:
            test = self._bind(self._test, ob_no[te], action_na[te], advantage_n[te], prob_np[te])
            test_losses_before = self._losses(test)

        theta, _, opt_info = scipy.optimize.fmin_l_bfgs_b(lossandgrad, thprev, maxiter=cfg["maxiter"])
        del opt_info['grad']
        print(opt_info)
        self.set_params_flat(theta)
        train_losses_after = self._losses(train)
        if cfg["do_split"]:
            test_losses_after = self._losses(test)
        klafter = train_losses_after[self.loss_names.index("kl")]
        if klafter > 1.3 * cfg["kl_target"]:
            self.kl_coeff *= 1.5
            print("Got KL=%.3f (target %.3f). Increasing penalty coeff => %.3f." % (klafter, cfg["kl_target"], self.kl_coeff))
        elif klafter < 0.7 * cfg["kl_target"]:
            self.kl_coeff /= 1.5
            print("Got KL=%.3f (target %.3f). Decreasing penalty coeff => %.3f." % (klafter, cfg["kl_target"], self.kl_coeff))
        else:
            print("KL=%.3f is close enough to target %.3f." % (klafter, cfg["kl_target"]))
        info = OrderedDict()
        for (name, lossbefore, lossafter) in zipsame(self.loss_names, train_losses_before, train_losses_after):
            info[name + "_before"] = lossbefore
            info[name + "_after"] = lossafter
            info[name + "_change"] = lossafter - lossbefore
        if cfg["do_split"]:
            for (name, lossbefore, lossafter) in zipsame(self.loss_names, test_losses_before, test_losses_after):
                info["test_" + name + "_before"] = lossbefore
                info["test_" + name + "_after"] = lossafter
                info["test_" + name + "_change"] = lossafter - lossbefore
        return info


class PpoSgdUpdater(EzFlat, EzPickle):
    """ppo.py:115-228.  Differences from PpoLbfgsUpdater that matter: the old policy's probabilities are a
    forward pass at the parameters the call starts from (not path["prob"]), KL is always kl[old, new], each
    minibatch's `train` returns the losses BEFORE its Adam step, and kl_coeff adapts on the last epoch's mean
    minibatch KL."""

    options = [
        ("kl_target", float, 1e-2, ""),
        ("epochs", int, 10, ""),
        ("stepsize", float, 1e-3, ""),
        ("do_split", int, 0, "do train/test split"),
        ("kl_cutoff_coeff", float, 1000.0, ""),
    ]
    batchsize = 128

    def __init__(self, stochpol, usercfg):
        EzPickle.__init__(self, stochpol, usercfg)
        cfg = update_default_config(self.options, usercfg)
        print("PPOUpdater", cfg)
        if cfg["kl_cutoff_coeff"] != 1000.0:
            raise NotImplementedError("the device penalty kernel fixes kl_cutoff_coeff at 1000 (ppo.py:20)")
        self.stochpol = stochpol
        self.cfg = cfg
        self.kl_coeff = 1.0
        EzFlat.__init__(self, stochpol.net)
        self.loss_names = ["surr", "kl", "ent"]
        self._full = DeviceBatch(stochpol.dims[0], with_time_feature=True)
        self._mb = DeviceBatch(stochpol.dims[0], with_time_feature=True)
        self._sl = DeviceBatch(stochpol.dims[0], with_time_feature=True)
        stochpol.net.adam_reset()                     # adam_updates' moments and shared step counter live on the device

    def __call__(self, paths):
        """ppo.py:170-228.  The whole batch is bound ONCE; every minibatch of 128 is an index gather from the resident
        batch (mrl_batch_gather), its loss / gradient / Adam step one call without a host synchronisation
        (mrl_net_ppo_sgd_step); the host only draws the permutations (numpy's global generator, as the reference) and
        reads the mean losses once per epoch."""
        cfg = self.cfg
        net = self.stochpol.net
        ob_no = concat([path["observation"] for path in paths])
        action_na = concat([path["action"] for path in paths])
        advantage_n = concat([path["advantage"] for path in paths])
        ob_no = np.asarray(ob_no).reshape(len(ob_no), -1)
        N = ob_no.shape[0]
        bs = self.batchsize
        kl_cutoff = cfg["kl_target"] * 2.0
        head, dout = self.stochpol.probtype.head, self.stochpol.dims[-1]

        # update_old_net (ppo.py:174): the old policy is the current one; one forward pass gives its rows
        self._full.set_obs(ob_no)
        oldprob_np = self.stochpol.output_from_head(net.forward(self._full))
        self._full.set_policy_inputs(head, dout, action_na, advantage_n, oldprob_np)

        def losses_of(lo, hi):
            b = self._full if (lo == 0 and hi == N) else self._sl.gather_from(self._full, np.arange(lo, hi, dtype=np.int32))
            return net.ppo_lossgrad(b, 0.0, 1e300, False, want_grad=False)[2]

        if cfg["do_split"]:
            train_stop = (int(.75 * N) // bs) * bs
            test_losses_before = losses_of(train_stop, N)
        else:
            train_stop = N
        train_losses_before = losses_of(0, train_stop)

        train_losses = train_losses_before
        net.ppo_sgd_read() if getattr(self, "_ran", False) else None      # drop a stale running sum
        self._ran = True
        for _ in range(cfg["epochs"]):
            sortinds = np.random.permutation(train_stop).astype(np.int32)
            for istart in range(0, train_stop, bs):
                mb = self._mb.gather_from(self._full, sortinds[istart:istart + bs])
                net.ppo_sgd_step(mb, self.kl_coeff, kl_cutoff, cfg["stepsize"])
            train_losses, _ = net.ppo_sgd_read()
            if cfg["do_split"]:
                test_losses = losses_of(train_stop, N)

        klafter = train_losses[self.loss_names.index("kl")]
        if klafter > 1.3 * cfg["kl_target"]:
            self.kl_coeff *= 1.5
            print("Got KL=%.3f (target %.3f). Increasing penalty coeff => %.3f." % (klafter, cfg["kl_target"], self.kl_coeff))
        elif klafter < 0.7 * cfg["kl_target"]:
            self.kl_coeff /= 1.5
            print("Got KL=%.3f (target %.3f). Decreasing penalty coeff => %.3f." % (klafter, cfg["kl_target"], self.kl_coeff))
        else:
            print("KL=%.3f is close enough to target %.3f." % (klafter, cfg["kl_target"]))
        info = OrderedDict()
        for (name, lossbefore, lossafter) in zipsame(self.loss_names, train_losses_before, train_losses):
            info[name + "_before"] = lossbefore
            info[name + "_after"] = lossafter
            info[name + "_change"] = lossafter - lossbefore
        if cfg["do_split"]:
            for (name, lossbefore, lossafter) in zipsame(self.loss_names, test_losses_before, test_losses):
                info["test_" + name + "_before"] = lossbefore
                info["test_" + name + "_after"] = lossafter
                info["test_" + name + "_change"] = lossafter - lossbefore
        return info
