"""Data-parallel driver logic: one process per GPU, the timestep batch sharded by WHOLE
trajectories (so GAE and the within-path time index need no halo), partial sums combined by an
all-reduce of the parameter-sized vector, CG / line search / L-BFGS replicated on identical bits.

The reference has no parallel path (core.py:123-124 raises NotImplementedError); this module is the
host-side half of DESIGN.md "Multi-GPU".  Everything here is plain Python/numpy so that it can be
tested on CPU with the gloo backend; the device-side sums run in libmrl_b200.so over NCCL.

Data-parallel training (run_pg.py under torchrun, WORLD_SIZE > 1): `init_data_parallel` records the
process's (rank, world, device, comm) once; core / agentzoo / ppo read it through `context()`.  Each rank
collects its own quota of trajectories; the few KB that must agree across ranks after the rollouts (filter
states, episode rewards and lengths, the rank's timestep count) travel in ONE host all-gather over a gloo group
(`sync_rollouts`), so a rank whose rollouts run long makes the others wait on the host.  Every per-timestep sum
after that runs in the library over `comm`.
"""
from __future__ import annotations

import itertools
import os
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np


def bind_to_device_numa(device_index: int) -> int:
    """Restrict this process to the CPU cores closest to GPU `device_index` (NVML's ideal affinity mask, intersected
    with the cores the process may use) so that the pinned host buffers it allocates afterwards are first-touched on
    the GPU's own NUMA node.  With 8 ranks on a two-socket host the uploads otherwise share one socket's memory and
    inter-socket links (measured 22 GB/s per GPU at N = 8 against 54 GB/s at N = 2).  Returns the number of cores
    bound to, 0 when NVML or the affinity call is unavailable (nothing changed)."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        ideal = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cores = ideal & set(os.sched_getaffinity(0))
        if not cores:
            return 0
        os.sched_setaffinity(0, cores)
        return len(cores)
    except Exception:
        return 0


def shard_bounds(lengths: Sequence[int], world: int) -> List[Tuple[int, int]]:
    """Contiguous blocks of whole trajectories, balanced by timestep count.

    Path p goes to the rank whose ideal span [r*N/world, (r+1)*N/world) contains the path's FIRST
    timestep.  Returns [(first_path, end_path)] per rank; blocks are disjoint, ordered and cover every
    path; a rank may be empty when there are fewer paths than ranks."""
    lengths = np.asarray(lengths, np.int64)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]) if len(lengths) else np.zeros(0, np.int64)
    N = int(lengths.sum())
    out = []
    for r in range(world):
        lo_t = (N * r) // world
        hi_t = (N * (r + 1)) // world
        a = int(np.searchsorted(starts, lo_t, side="left"))
        b = int(np.searchsorted(starts, hi_t, side="left")) if r < world - 1 else len(lengths)
        out.append((a, b))
    return out


def shard_paths(paths: list, rank: int, world: int) -> list:
    a, b = shard_bounds([len(p["reward"]) for p in paths], world)[rank]
    return paths[a:b]


def merge_moments(triples: Sequence[Tuple[float, float, float]]) -> Tuple[float, float, float]:
    """Chan merge of (n, mean, M2) in the given (rank) order - the same arithmetic, in the same order,
    as merge_moments_kernel, so every rank derives bit-identical mean/std for the advantage
    standardisation (core.py:100-105)."""
    n, mean, m2 = 0.0, 0.0, 0.0
    for bn, bm, b2 in triples:
        if bn == 0:
            continue
        if n == 0:
            n, mean, m2 = float(bn), float(bm), float(b2)
            continue
        tot = n + bn
        d = bm - mean
        mean = mean + d * (bn / tot)
        m2 = m2 + b2 + d * d * (n * bn / tot)
        n = tot
    return n, mean, m2


def zfilter_prefix(states: Sequence[Tuple[float, np.ndarray, np.ndarray]], rank: int):
    """Exclusive prefix of Welford states over ranks: the state a rank's ZFilter scan must start from
    when consecutive sample blocks live on consecutive ranks (running_stat.py semantics)."""
    n, M, S = 0.0, None, None
    for bn, bM, bS in states[:rank]:
        bM, bS = np.asarray(bM, np.float64), np.asarray(bS, np.float64)
        if bn == 0:
            continue
        if n == 0:
            n, M, S = float(bn), bM.copy(), bS.copy()
            continue
        tot = n + bn
        d = bM - M
        M = M + d * (bn / tot)
        S = S + bS + d * d * (n * bn / tot)
        n = tot
    return n, M, S


P2P_MAX_DOUBLES = 1 << 17     # receive-slot size: covers parameter vectors up to 131 072 entries


def comm_from_torch_distributed(device: int, p2p: bool = True):
    """Build the library's communicator inside an initialised torch.distributed job: rank 0 creates the
    NCCL unique id, torch broadcasts it (plumbing only).  With p2p (default) the ranks then exchange the
    CUDA IPC handles of their NVLink receive buffers, so that parameter-sized sums bypass NCCL; if any rank
    cannot map a peer (no peer access between the GPUs) every rank stays on NCCL."""
    import torch.distributed as dist
    from .device import Comm
    rank, world = dist.get_rank(), dist.get_world_size()
    box = [Comm.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    comm = Comm(box[0], rank, world, device)
    if p2p and 1 < world <= 8:
        enable_p2p(comm)
    return comm


def enable_p2p(comm, max_doubles: int = P2P_MAX_DOUBLES) -> bool:
    """All ranks must call this together.  Returns True when the peer-memory transport is active."""
    import torch.distributed as dist
    try:
        handle, err = comm.p2p_export(max_doubles), None
    except RuntimeError as e:                       # every rank must still take part in the all-gather
        handle, err = b"", str(e)
    handles = [None] * comm.world
    dist.all_gather_object(handles, (handle, err))
    if any(e is not None for _, e in handles):
        return False
    ok = True
    try:
        comm.p2p_connect([h for h, _ in handles])
    except RuntimeError:
        ok = False
    flags = [None] * comm.world
    dist.all_gather_object(flags, ok)
    if not all(flags):
        return False
    comm.p2p_enable(True)
    return True


# ================================================================ data-parallel training (run_pg.py under torchrun)

class DataParallel(NamedTuple):
    rank: int
    world: int
    device: int          # CUDA device of this rank: every DeviceNet / DeviceBatch the agent creates lives here
    comm: object         # the library communicator shared by the policy net and the value net
    group: object        # gloo process group for the host-side collectives (filter states, statistics)


_context: Optional[DataParallel] = None
_batch_paths, _batch_total = None, 0


def context() -> Optional[DataParallel]:
    """The data-parallel context of this process, None in a single-process run."""
    return _context


def current_device() -> int:
    return _context.device if _context is not None else 0


def is_root() -> bool:
    return _context is None or _context.rank == 0


def launched_data_parallel() -> bool:
    """True under a launcher that starts several processes (torchrun sets WORLD_SIZE)."""
    return int(os.environ.get("WORLD_SIZE", "1") or 1) > 1


def reject_data_parallel(what: str) -> None:
    """Raise for a configuration that data-parallel training does not cover."""
    if launched_data_parallel():
        raise NotImplementedError("%s is not supported in data-parallel training (WORLD_SIZE=%s); run it in one process"
                                  % (what, os.environ.get("WORLD_SIZE")))


def init_data_parallel(p2p: Optional[bool] = None) -> DataParallel:
    """Set up this rank of a torchrun job: pin it to the cores next to GPU LOCAL_RANK, make that GPU current,
    initialise the NCCL process group, build the library communicator (NVLink peer-memory transport unless
    p2p=False or MRL_NCCL_ONLY=1) and a gloo group for the host collectives.  Records and returns the context."""
    global _context
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    bind_to_device_numa(local)
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if p2p is None:
        p2p = os.environ.get("MRL_NCCL_ONLY") != "1"
    comm = comm_from_torch_distributed(local, p2p=p2p)
    group = dist.new_group(backend="gloo")
    _context = DataParallel(rank, world, local, comm, group)
    return _context


def shutdown_data_parallel() -> None:
    """Every rank calls this once its last update is done: closes the communicator and the process group."""
    global _context, _batch_paths
    import torch.distributed as dist
    if _context is None:
        return
    dist.barrier(group=_context.group)
    _context.comm.close()
    _context, _batch_paths = None, None
    dist.destroy_process_group()


def all_gather(obj) -> list:
    """`obj` of every rank in rank order, over the host group ([obj] without torch.distributed)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return [obj]
    group = _context.group if _context is not None else None
    out = [None] * dist.get_world_size(group)
    dist.all_gather_object(out, obj, group=group)
    return out


def barrier() -> None:
    if _context is not None:
        import torch.distributed as dist
        dist.barrier(group=_context.group)


def rank_quota(n_timesteps: int, world: int) -> int:
    """Timesteps one rank collects before it stops (ceil(n / world); each rank stops strictly above it)."""
    return -(-int(n_timesteps) // int(world))


def seed_stream(rank: Optional[int] = None, world: Optional[int] = None):
    """Rollout seeds of one rank: rank, rank + world, ... (itertools.count() in one process), so no seed repeats
    across ranks."""
    if rank is None:
        rank, world = (_context.rank, _context.world) if _context is not None else (0, 1)
    return itertools.count(rank, world)


def check_replicated(arrays) -> None:
    """All ranks must hold bit-identical `arrays` (name -> array); raises RuntimeError naming the ones that differ."""
    import hashlib
    mine = {k: hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest() for k, v in arrays.items()}
    ranks = all_gather(mine)
    bad = sorted(k for k in mine if any(r[k] != ranks[0][k] for r in ranks))
    if bad:
        raise RuntimeError("data-parallel ranks start from different %s; every rank must call np.random.seed(seed) "
                           "with the same seed before it builds the agent (or load the same snapshot)" % ", ".join(bad))


def attach_agent(agent) -> None:
    """Give the agent's policy net and value net the communicator, then check that every rank starts from the same
    parameters (the updates are replicated, so they must)."""
    nets = {"policy parameters": agent.policy.net}
    reg = getattr(agent.baseline, "reg", None)
    if reg is not None:
        nets["value-function parameters"] = reg.net
    for net in nets.values():
        net.set_comm(_context.comm)
    check_replicated({k: net.get_params() for k, net in nets.items()})


def _zfilters(agent):
    from .filters import ZFilter
    return [f for f in (agent.obfilter, agent.rewfilter) if isinstance(f, ZFilter)]


def begin_rollouts(agent) -> list:
    """Before a rank's rollouts: -> the filter states the iteration starts from (identical on every rank); each
    ZFilter also records the samples it pushes from now on in a state of their own."""
    starts = []
    for f in _zfilters(agent):
        starts.append(f.rs.state())
        f.start_round()
    return starts


def merge_filter_states(start, pushed):
    """Chan merge of `start` and the states of the samples rank 0, 1, ... pushed, in that order -> (n, M, S)."""
    n, M, S = zfilter_prefix([start] + list(pushed), len(pushed) + 1)
    return start if M is None else (n, M, S)


def global_timesteps(paths) -> Optional[int]:
    """Timesteps of all ranks when `paths` is this rank's batch of the running iteration, else None."""
    return _batch_total if (_context is not None and paths is _batch_paths) else None


def sync_rollouts(agent, paths, starts) -> dict:
    """After a rank's rollouts: ONE host all-gather of (pushed filter states, episode rewards and lengths).  Every
    rank's ZFilters become the merge of `starts` and all ranks' pushed states (bit-identical everywhere), and
    `paths` is registered as this rank's shard of a batch of n_total timesteps (see global_timesteps).
    -> dict(rewards, lengths) of every episode of the iteration in rank order, n_total."""
    global _batch_paths, _batch_total
    from .core import episode_arrays
    filts = _zfilters(agent)
    rewards, lengths = episode_arrays(paths)
    mine = dict(filters=[f.pushed.state() for f in filts], rewards=rewards, lengths=lengths)
    ranks = all_gather(mine)
    for i, (f, start) in enumerate(zip(filts, starts)):
        f.rs.set_state(*merge_filter_states(start, [r["filters"][i] for r in ranks]))
        f.pushed = None
    lengths = np.concatenate([r["lengths"] for r in ranks])
    _batch_paths, _batch_total = paths, int(lengths.sum())
    return dict(rewards=np.concatenate([r["rewards"] for r in ranks]), lengths=lengths, n_total=_batch_total)


def _moments(x):
    x = np.asarray(x, np.float64).ravel()
    m = float(x.mean()) if x.size else 0.0
    return float(x.size), m, float(np.square(x - m).sum())


def regression_stats(ypredold_ny, yprednew_ny, ytarg_ny):
    """NnRegression's statistics (PredStdevBefore/After, TargStdev, EV_before/after or EV_avg) of the batch of all
    ranks: per-rank (n, mean, M2) of each quantity, merged in rank order, same formulas as the single-process fit
    (population std; explained variance 1 - Var[y - ypred] / Var[y])."""
    cols = (ypredold_ny, yprednew_ny, ytarg_ny, ytarg_ny - ypredold_ny, ytarg_ny - yprednew_ny)
    ranks = all_gather([_moments(c) for c in cols])
    var = []
    for j in range(len(cols)):
        n, _, m2 = merge_moments([r[j] for r in ranks])
        var.append(m2 / n)
    pold, pnew, targ, rold, rnew = var
    out = dict(PredStdevBefore=np.sqrt(pold), PredStdevAfter=np.sqrt(pnew), TargStdev=np.sqrt(targ))
    if np.shape(ytarg_ny)[1] == 1:
        out["EV_before"] = 0.0 if targ < 1e-10 else 1 - rold / targ
        out["EV_after"] = 0.0 if targ < 1e-10 else 1 - rnew / targ
    else:
        out["EV_avg"] = np.nan if targ == 0 else 1 - rnew / targ
    return out
