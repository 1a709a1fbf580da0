"""Data-parallel training: tests/dp_training_check.py under torchrun (bit-identical replicas, agreement with a
one-process replay of the last update) on 2 GPUs over both transports, and run_pg.py itself under torchrun.  The
2-rank tests skip on a machine with fewer than two GPUs.  A 1-rank run of the same check still drives every
data-parallel code path (context, communicator, filter merge, global batch size, merged statistics) on one GPU.  The
host-side exchange is covered on CPU by test_data_parallel_training.py."""
import os
import signal
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _need_gpus(n):
    import torch
    if torch.cuda.device_count() < n:
        pytest.skip("needs %d GPUs" % n)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _torchrun(args, env=None, timeout=600, ranks=2):
    """torchrun in a session of its own, so that a timeout takes the ranks down with the launcher."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ranks),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port())] + args
    p = subprocess.Popen(cmd, cwd=ROOT, env=dict(os.environ, **(env or {})), stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, start_new_session=True)
    try:
        out, _ = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        out, _ = p.communicate()
        pytest.fail("timed out after %d s:\n%s" % (timeout, out[-4000:]))
    return p.returncode, out


@pytest.mark.gpu
@pytest.mark.parametrize("ranks,transport", [(2, "p2p"), (2, "nccl"), (1, "nccl")])
def test_dp_training_matches_one_process_replay(ranks, transport):
    _need_gpus(ranks)
    rc, out = _torchrun([os.path.join(ROOT, "tests", "dp_training_check.py")], ranks=ranks,
                        env={"MRL_NCCL_ONLY": "1" if transport == "nccl" else "0"})
    assert rc == 0 and "DP_TRAINING_CHECK_OK" in out, out[-4000:]
    assert ("transport: nccl" in out) == (transport == "nccl"), out[-4000:]


@pytest.mark.gpu
def test_run_pg_under_torchrun(tmp_path):
    """run_pg.py's own flags under torchrun: rank 0 alone prints and writes the snapshot, --load_snapshot resumes on
    every rank."""
    _need_gpus(2)
    out_file = str(tmp_path / "dp.h5")
    base = [os.path.join(ROOT, "run_pg.py"), "--env", "CartPole-v0", "--agent", "modular_rl.agentzoo.TrpoAgent",
            "--timesteps_per_batch", "2000", "--cg_damping", "0.1", "--vec_envs", "4"]
    rc, out = _torchrun(base + ["--n_iter", "2", "--snapshot_every", "2", "--outfile", out_file])
    assert rc == 0, out[-4000:]
    assert out.count("*********** Iteration 2 ") == 1 and out.count("policy gradient config") == 1, out[-4000:]
    snap = os.path.join(out_file + ".dir", "agent_snapshots", "0002.pkl")
    assert os.path.exists(snap)
    rc, out = _torchrun(base + ["--n_iter", "1", "--load_snapshot", snap, "--outfile", str(tmp_path / "resumed.h5")])
    assert rc == 0 and out.count("*********** Iteration 1 ") == 1, out[-4000:]
