"""One tile's prior extraction over two GPUs (skipped on a box with fewer): ShardedPriorExtractor against a single-GPU
PriorExtractor on all the rays, for even, uneven and one-sided splits, several exchange rounds and a spatially skewed
tile.  Worker: tests/sharded_extract_worker.py, one torchrun launch for all the cases."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs on the box")]
HERE = os.path.dirname(os.path.abspath(__file__))
CASES = ["c2", "presight16", "uneven", "idle", "rounds", "skewed"]


@pytest.fixture(scope="module")
def worker_output():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29547", os.path.join(HERE, "sharded_extract_worker.py"),
           ",".join(CASES)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    return r.returncode, r.stdout + r.stderr


@pytest.mark.parametrize("case", CASES)
def test_sharded_finalize_matches_one_gpu(worker_output, case):
    rc, out = worker_output
    lines = [l for l in out.splitlines() if l.startswith(f"SHARDED {case} ")]
    print("\n".join(lines))
    assert rc == 0, out[-3000:]
    assert lines and all(" ok:" in l for l in lines), "\n".join(lines) or out[-3000:]
