"""Row-partitioned eliminated solve of R / A / E netlists (nodal_b200/dist_sources.py):
tests/dist_sources_check.py under torchrun, on one process and, when the box has two GPUs, on two."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("nproc", [1, 2])
def test_dist_sources_check(nproc):
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPU(s)")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
           "--master-addr", "127.0.0.1", "--master-port", str(29540 + nproc),
           os.path.join(ROOT, "tests", "dist_sources_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert out.returncode == 0 and "DIST_SOURCES_CHECK PASS" in out.stdout, out.stdout[-4000:] + out.stderr[-4000:]
