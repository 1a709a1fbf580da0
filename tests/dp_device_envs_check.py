#!/usr/bin/env python
"""dp_training_check.py with the rollouts on the device (core.DEVICE_ENVS, run_pg.py --device_envs), run under
torchrun with one rank per GPU:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
      --master-port 29522 tests/dp_device_envs_check.py

After every iteration the parameters and both filter states must be bit-identical on every rank, and the last update
must match a one-process replay on the paths of all ranks (run_case of dp_training_check.py)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from dp_training_check import run_case  # noqa: E402


def main():
    from modular_rl_b200 import core, parallel
    ctx = parallel.init_data_parallel()
    failures = []
    core.DEVICE_ENVS = 16
    try:
        run_case("TrpoAgent", "CartPole-v0", dict(cg_damping=0.1), 0, failures)
        run_case("PpoLbfgsAgent", "Pendulum-v0", {}, 0, failures)
    finally:
        core.DEVICE_ENVS = 0
    failures = [f for r in parallel.all_gather(failures) for f in r]
    parallel.shutdown_data_parallel()
    if failures:
        print("FAIL", failures, flush=True)
        sys.exit(1)
    if ctx.rank == 0:
        print("DP_DEVICE_ENVS_CHECK_OK", flush=True)


if __name__ == "__main__":
    main()
