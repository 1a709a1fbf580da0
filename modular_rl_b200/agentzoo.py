"""Agents = containers with policy, value function, filters and updater - the reference's
agentzoo.py API unchanged (TrpoAgent, PpoLbfgsAgent, the option tables and therefore the run_pg.py
flags), built on device-resident networks instead of Keras models."""
from . import _lib as L
from . import parallel
from .core import (Categorical, DiagGauss, NnVf, PG_OPTIONS, StochPolicyMLP, make_value_net)
from .filters import ZFilter
from .misc_utils import IDENTITY, comma_sep_ints, update_default_config
from .ppo import PpoLbfgsUpdater, PpoSgdUpdater
from .spaces import is_box, is_discrete
from .trpo import TrpoUpdater

MLP_OPTIONS = [
    ("hid_sizes", comma_sep_ints, [64, 64], "Sizes of hidden layers of MLP"),
    ("activation", str, "tanh", "nonlinearity"),
]


def make_mlps(ob_space, ac_space, cfg):
    """(policy, baseline) as agentzoo.py:25-61: Dense(h, act) per hidden size; Box actions ->
    Dense(d) with kernel*0.1 + state-independent logstd, Discrete -> Dense(K, softmax) with
    kernel*0.1; value net on [ob, t/timestep_limit] -> Dense(1); NnVf(mixfrac=0.1)."""
    assert is_box(ob_space)
    hid_sizes = list(cfg["hid_sizes"])
    if is_box(ac_space):
        probtype = DiagGauss(ac_space.shape[0])
    elif is_discrete(ac_space):
        probtype = Categorical(ac_space.n)
    else:
        raise NotImplementedError("action space %r" % (ac_space,))
    policy = StochPolicyMLP(ob_space.shape[0], hid_sizes, probtype, cfg["activation"])
    vfnet = make_value_net(ob_space.shape[0], hid_sizes, cfg["activation"])
    baseline = NnVf(vfnet, cfg["timestep_limit"], dict(mixfrac=0.1))
    return policy, baseline


class DeterministicPolicy(StochPolicyMLP):
    """The net of make_deterministic_mlp (agentzoo.py:63-81): Dense(h, tanh) per hidden size, then a linear
    Dense(outdim) with kernel*0.1, acted on through probtype.maxprob - the output itself for Box actions, the
    argmax for Discrete ones (softmax is monotone, so the argmax of the probabilities is the argmax of the
    reference's logits; the "prob" row holds probabilities here, logits there, and nothing reads it).
    The flat parameter vector is the Dense kernels and biases only: the device net of the Box case carries a
    logstd block (pinned to 0, never used by maxprob) that get/set_params_flat hide, so the search space of
    the cross-entropy method has the reference's dimension."""

    def __init__(self, ob_dim, hid_sizes, probtype, activation="tanh", theta=None):
        self._nlogstd = probtype.d if isinstance(probtype, DiagGauss) else 0
        StochPolicyMLP.__init__(self, ob_dim, hid_sizes, probtype, activation, theta)

    def set_params_flat(self, theta):
        import numpy as np
        theta = np.asarray(theta)
        if theta.size == self.net.P - self._nlogstd:
            theta = np.concatenate([theta.ravel(), np.zeros(self._nlogstd, theta.dtype)])
        StochPolicyMLP.set_params_flat(self, theta)

    def get_params_flat(self):
        th = StochPolicyMLP.get_params_flat(self)
        return th[:th.size - self._nlogstd] if self._nlogstd else th

    def output_from_head(self, out):
        return out          # the reference's prob row here is the bare net output (no ConcatFixedStd layer)

    def act(self, ob, stochastic=False):
        if stochastic:
            raise ValueError("DeterministicPolicy has no sampling distribution; use set_stochastic(False)")
        return StochPolicyMLP.act(self, ob, stochastic=False)

    def act_batch(self, ob_no, stochastic=False):
        if stochastic:
            raise ValueError("DeterministicPolicy has no sampling distribution; use set_stochastic(False)")
        return StochPolicyMLP.act_batch(self, ob_no, stochastic=False)


def make_deterministic_mlp(ob_space, ac_space, cfg):
    """agentzoo.py:63-81 (hidden activation is tanh there regardless of --activation)."""
    assert is_box(ob_space)
    if is_box(ac_space):
        probtype = DiagGauss(ac_space.shape[0])
    elif is_discrete(ac_space):
        probtype = Categorical(ac_space.n)
    else:
        raise NotImplementedError("action space %r" % (ac_space,))
    return DeterministicPolicy(ob_space.shape[0], list(cfg["hid_sizes"]), probtype, "tanh")


FILTER_OPTIONS = [
    ("filter", int, 1, "Whether to do a running average filter of the incoming observations and rewards"),
]


def make_filters(cfg, ob_space):
    if cfg["filter"]:
        obfilter = ZFilter(ob_space.shape, clip=5)
        rewfilter = ZFilter((), demean=False, clip=10)
    else:
        obfilter = IDENTITY
        rewfilter = IDENTITY
    return obfilter, rewfilter


class AgentWithPolicy(object):
    def __init__(self, policy, obfilter, rewfilter):
        self.policy = policy
        self.obfilter = obfilter
        self.rewfilter = rewfilter
        self.stochastic = True

    def set_stochastic(self, stochastic):
        self.stochastic = stochastic

    def act(self, ob_no):
        return self.policy.act(ob_no, stochastic=self.stochastic)

    def get_flat(self):
        return self.policy.get_flat()

    def set_from_flat(self, th):
        return self.policy.set_from_flat(th)

    def obfilt(self, ob):
        return self.obfilter(ob)

    def rewfilt(self, rew):
        return self.rewfilter(rew)


class DeterministicAgent(AgentWithPolicy):
    options = MLP_OPTIONS + FILTER_OPTIONS

    def __init__(self, ob_space, ac_space, usercfg):
        cfg = update_default_config(self.options, usercfg)
        policy = make_deterministic_mlp(ob_space, ac_space, cfg)
        obfilter, rewfilter = make_filters(cfg, ob_space)
        AgentWithPolicy.__init__(self, policy, obfilter, rewfilter)
        self.set_stochastic(False)


class TrpoAgent(AgentWithPolicy):
    options = MLP_OPTIONS + PG_OPTIONS + TrpoUpdater.options + FILTER_OPTIONS

    def __init__(self, ob_space, ac_space, usercfg):
        cfg = update_default_config(self.options, usercfg)
        policy, self.baseline = make_mlps(ob_space, ac_space, cfg)
        obfilter, rewfilter = make_filters(cfg, ob_space)
        self.updater = TrpoUpdater(policy, cfg)
        AgentWithPolicy.__init__(self, policy, obfilter, rewfilter)


class PpoLbfgsAgent(AgentWithPolicy):
    options = MLP_OPTIONS + PG_OPTIONS + PpoLbfgsUpdater.options + FILTER_OPTIONS

    def __init__(self, ob_space, ac_space, usercfg):
        cfg = update_default_config(self.options, usercfg)
        if cfg["do_split"]:
            parallel.reject_data_parallel("PpoLbfgsAgent with do_split=1")
        policy, self.baseline = make_mlps(ob_space, ac_space, cfg)
        obfilter, rewfilter = make_filters(cfg, ob_space)
        self.updater = PpoLbfgsUpdater(policy, cfg)
        AgentWithPolicy.__init__(self, policy, obfilter, rewfilter)


class PpoSgdAgent(AgentWithPolicy):
    options = MLP_OPTIONS + PG_OPTIONS + PpoSgdUpdater.options + FILTER_OPTIONS

    def __init__(self, ob_space, ac_space, usercfg):
        parallel.reject_data_parallel("PpoSgdAgent")
        cfg = update_default_config(self.options, usercfg)
        policy, self.baseline = make_mlps(ob_space, ac_space, cfg)
        obfilter, rewfilter = make_filters(cfg, ob_space)
        self.updater = PpoSgdUpdater(policy, cfg)
        AgentWithPolicy.__init__(self, policy, obfilter, rewfilter)
