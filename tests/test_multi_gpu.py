"""Two ranks on two GPUs (skipped when the box has fewer): the row-owned, chunk-sharded solve of SURVEY.md 8(e) —
tools/mgpu_check.py under torchrun — must reproduce the oracle: the block rows of H each rank owns (1e-7), the damped step
(1e-6), the LM traces of both paths (final costs 1e-6, same iteration counts) on a 500-pose problem (BASELINE configs[1]).
The data flow itself (owned rows only, one all-gather, replicated top tree) is checked without GPUs in
tests/test_nd_solver_emu.py::test_rank_sharded_solve_matches_dense and, between two processes over gloo, in
tests/test_rank_flow_gloo.py."""
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.mark.gpu
def test_two_rank_sharded_run_matches_the_oracle():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = 29600 + os.getpid() % 1000
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(ROOT / "tools" / "mgpu_check.py"), "B"]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=str(ROOT), timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MGPU_CHECK PASS world 2" in r.stdout, r.stdout[-3000:]
    assert "sharded=True" in r.stdout, r.stdout[-3000:]
