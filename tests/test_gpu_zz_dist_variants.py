"""The distributed CholInv schedule under every knob set of tests/dist_cases.py, with all ranks of a 2x1x1, 1x2x2 or 2x2x2 grid sharing
cuda:0 (CUDA IPC between processes on one device: the same peer memory, flags and fused exchanges as on separate GPUs).

The lowered thresholds put the small sizes through every deferred class and through column-chunked, pushed (and optionally
pipelined) products; the ragged sizes split on odd rows at every level, so the products of the chain and of the deferred streams copy
their misaligned operands into their streams' alignment scratch at the same time.  Each case is checked against the numpy oracle, against
the default knob set bit for bit, across the depth replicas bit for bit, and on a second call (tests/dist_variants_worker.py)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_schedule_knob_sets_match_oracle_and_default_bit_for_bit(nproc):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(29611 + nproc), os.path.join(ROOT, "tests", "dist_variants_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    print(r.stdout[-3000:])
    assert r.returncode == 0 and "DV_OK" in r.stdout, r.stdout[-4000:] + r.stderr[-3000:]
