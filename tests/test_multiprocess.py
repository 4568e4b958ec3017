"""world_size > 1: row-range partitioning + partial-aggregate merge.  gloo on CPU (always), NCCL on
two B200s when present."""
import os
import subprocess
import sys

import numpy as np
import pytest

from datafusion_archive_b200 import parallel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def launch(mode, nproc, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mp_worker.py"), mode]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    if p.returncode != 0:  # keep the workers' own tracebacks (pytest truncates long assertion messages)
        try:
            os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
            with open(os.path.join(ROOT, "gpurun_out", "mp_worker_%s.log" % mode), "w") as f:
                f.write(p.stdout + "\n---- stderr ----\n" + p.stderr)
        except OSError:
            pass
    return p


def test_row_ranges_cover_exactly():
    for n in [0, 1, 7, 8, 9, 1000, 100_000_001]:
        for w in [1, 2, 3, 4, 8]:
            r = [parallel.row_range(g, w, n) for g in range(w)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(r[i][1] == r[i + 1][0] for i in range(w - 1))
            assert all(hi - lo <= -(-n // w) for lo, hi in r)


def test_gloo_world2_partition_and_merge():
    p = launch("gloo", 2, 29631)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    assert "MP_OK mode=gloo world=2" in p.stdout


@pytest.mark.gpu
def test_nccl_world2_partial_aggregate_merge():
    from datafusion_archive_b200 import engine
    if engine.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    p = launch("nccl", 2, 29632)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    assert "MP_OK mode=nccl world=2" in p.stdout
