"""bench.py on a B200 at a reduced size: --steps sets the number of steps of every timed loop, and
--dump-outputs writes what the last timed step returned, the same from run to run and equal to numpy's
answer on the same seeded rows."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from datafusion_archive_b200 import workloads

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS = 10_000_000  # C2 keeps ~5e6 rows: more than the 4 Mi rows bench.py dumps, so the dump is a sample
SAMPLE = 1 << 22


def run_bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(ROWS), "--steps", str(steps), "--warmup", "1",
                        "--no-cpu", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_steps_and_dumped_outputs(tmp_path):
    j3, j4 = run_bench(tmp_path / "a", 3), run_bench(tmp_path / "b", 4)
    for j, k in ((j3, 3), (j4, 4)):
        assert j["steps"] == k and j["e2e"]["steps"] == k and j["c4"]["steps"] == k and j["e2e_c4"]["steps"] == k
        assert "sustained" not in j
    assert j3["gpu_launches"] > 0 and j3["gpu_launches"] * 4 == j4["gpu_launches"] * 3  # launches of the C2 window scale with K

    d3, d4 = load(tmp_path / "a"), load(tmp_path / "b")
    assert sorted(d3) == ["c2_a", "c4_count", "c4_key_hi", "c4_key_lo", "c4_sum"] and sorted(d4) == sorted(d3)
    assert all(x.dtype == np.float64 for x in d3.values()) and sum(x.nbytes for x in d3.values()) <= 64 << 20

    # C2: the seeded sample of SELECT a FROM t WHERE a > 0.5, bit-exact, and identical in both runs
    a = workloads.c2(ROWS, seed=42)[0][0]
    sel = a[a > 0.5]
    pos = np.sort(np.random.default_rng(0).choice(len(sel), SAMPLE, replace=False))
    assert np.array_equal(d3["c2_a"], sel[pos]) and np.array_equal(d4["c2_a"], d3["c2_a"])

    # C4: rows sorted by key; keys and counts exact, sums within 1e-9
    (_, v), _, _, k_raw = workloads.c4(ROWS, seed=46)
    cnt = np.bincount(k_raw, minlength=100_000)
    present = np.nonzero(cnt)[0]
    keys = workloads.mix_keys(present.astype(np.int64))
    order = np.argsort(keys)
    for d in (d3, d4):
        k = (d["c4_key_hi"].astype(np.int64) << 32) | d["c4_key_lo"].astype(np.int64)
        assert np.array_equal(k, keys[order])
        assert np.array_equal(d["c4_count"], cnt[present][order].astype(np.float64))
        np.testing.assert_allclose(d["c4_sum"], np.bincount(k_raw, weights=v, minlength=100_000)[present][order], rtol=1e-9, atol=0)
