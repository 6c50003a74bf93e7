"""-m gpu: bench.py end to end at a reduced size -- `--steps` sets the number of timed steps, and `--dump-outputs` writes
the product of the last timed step, the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import generators as G
from helpers import HBSM

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(steps, out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--n", "8192",
           "--no-check", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_bench_steps_and_dumped_outputs(tmp_path):
    d2, d3 = _bench(2, tmp_path / "s2"), _bench(3, tmp_path / "s3")
    assert (d2["steps"], d3["steps"]) == (2, 3)
    assert d2["gpu_launches"] * 3 == d3["gpu_launches"] * 2, "launches of the timed region do not scale with --steps"
    names = sorted(os.listdir(tmp_path / "s2"))
    assert names and names == sorted(os.listdir(tmp_path / "s3"))
    assert sum(os.path.getsize(tmp_path / "s2" / x) for x in names) <= 64 << 20
    got = {x[:-4]: np.load(tmp_path / "s2" / x) for x in names}
    for x in names:
        assert np.array_equal(got[x[:-4]], np.load(tmp_path / "s3" / x)), x
    # the dump is the product the timed path computes
    n, b, lam, tau = 8192, 64, 0.01, 1e-6
    hb.init(0)
    W = G.decay_width(lam, 1e-12)
    A = HBSM(np.float64, b); A.generate_decay(n, lam, W, 1); A.update_internal_info()
    B = HBSM(np.float64, b); B.generate_decay(n, lam, W, 2); B.update_internal_info()
    C = HBSM(np.float64)
    nm, nr = HBSM.spamm(A, 0, B, 0, C, tau, True)
    assert got["counts"].tolist() == [nm, nr] == [d2["products_per_multiply"], d2["c_tiles"]]
    assert len(got["c_tiles_row"]) == nr
    assert len(got["c_sample_tiles"]) > 0
    for i, j, t in zip(got["c_sample_row"], got["c_sample_col"], got["c_sample_tiles"]):
        assert np.array_equal(t, C.get_tile(int(i), int(j)))
