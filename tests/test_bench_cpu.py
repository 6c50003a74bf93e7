"""CPU: bench.py's reference arm prints exactly one JSON line on stdout with the contract's keys (tiny sample here)."""
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line(oracle_built):
    env = dict(os.environ, HBSM_CPU_SAMPLE_N="1024", OMP_NUM_THREADS="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["unit"] == "TFLOP/s" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"].startswith("fp64 SpAMM")
    # the arm runs a bounded sample: the line must say which n was really timed, and of what
    assert d["config"]["n"] == 1024 and d["config"]["sample_of"] == 65536
    assert "1024x1024" in d["config"]["workload"] and "1024x1024" in d["cpu_baseline"]["sample"]


def test_native_arm_fails_loudly_without_gpu():
    """No CUDA device here: the product path must refuse to run (no CPU fallback), not print a number."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is visible")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_config_cases_cover_the_baseline_configs():
    """bench.py --config 1..5 = BASELINE.json configs[0..4]; the first case of each is the one `value` is quoted on."""
    sys.path.insert(0, ROOT)
    import bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5
    head = bench.config_cases("headline")[0]
    assert (head["n"], head["b"], head["tau"], head["op"], head["dtype"]) == (65536, 64, 1e-6, "spamm", "f64")
    c1 = bench.config_cases("1")[0]; assert (c1["op"], c1["n"], c1["b"], c1["dtype"]) == ("multiply", 1024, 32, "f64")
    c2 = bench.config_cases("2"); assert all((c["n"], c["b"], c["tau"]) == (16384, 64, 1e-6) for c in c2)
    c3 = bench.config_cases("3"); assert {c["tau"] for c in c3 if c["op"] == "symm_square_spamm"} == {1e-4, 1e-6, 1e-8, 1e-10}
    assert any(c["op"] == "symm_square" for c in c3) and all(c["n"] == 65536 and c.get("symmetric") for c in c3)
    c4 = bench.config_cases("4")[0]; assert (c4["n"], c4["b"]) == (262144, 128)
    c5 = bench.config_cases("5")
    assert {c["b"] for c in c5} == {32, 64, 128, 256} and all(c["dtype"] == "f32" and c["n"] == 65536 for c in c5)
    assert {(c["tA"], c["tB"]) for c in c5 if c["op"] == "spamm"} == {(1, 0), (0, 1)} and any(c["op"] == "add" for c in c5)
    for cfg in ("headline", "1", "2", "3", "4", "5"):
        for c in bench.config_cases(cfg):
            txt = bench.case_config(c, 1, cfg)
            assert txt["n"] == c["n"] and txt["leaf"] == c["b"] and "workload" in txt
            assert bench.metric_of(c)[1] in ("TFLOP/s", "GB/s")
    # the committed single-GPU values every world size is checked against
    exp = bench.expected_results()
    assert bench.expected_key(head) in exp and exp[bench.expected_key(head)]["products"] == 2255020


class _FakeResult:
    """Stands in for a product result: export_leaves / get_params as the engine's matrix answers them."""

    def __init__(self, bi, bj, tiles, b):
        self.bi, self.bj, self.tiles, self.b = bi, bj, tiles, b

    def export_leaves(self, tiles=True, norms=True):
        return self.bi, self.bj, None, self.tiles

    def get_params(self):
        return types.SimpleNamespace(blocksize=self.b)


def test_dump_outputs_writes_sorted_float_tables_and_a_seeded_tile_sample(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    b, n = 4, 300
    rng = np.random.default_rng(1)
    keys = rng.choice(64 * 64, n, replace=False)                 # distinct tiles, exported in no particular order
    bi, bj = keys // 64, keys % 64
    tiles = rng.standard_normal((n, b * b))
    monkeypatch.setattr(bench, "DUMP_TABLE_MAX", 200)
    monkeypatch.setattr(bench, "DUMP_TILE_BYTES", 50 * b * b * 8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _FakeResult(bi, bj, tiles, b), 1234, n)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and all(x.endswith(".npy") for x in names)
    got = {x[:-4]: np.load(tmp_path / "a" / x) for x in names}
    for x in names:      # same inputs, same files
        assert np.array_equal(got[x[:-4]], np.load(tmp_path / "b" / x))
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["counts"].tolist() == [1234.0, n]
    r, c = got["c_tiles_row"], got["c_tiles_col"]
    assert len(r) == 200 and np.all(np.diff(r * 64 + c) > 0)    # a sample, in (row, col) order
    dense = {(int(i), int(j)): t.reshape(b, b).T for i, j, t in zip(bi, bj, tiles)}
    assert np.allclose(got["c_tiles_frob_sq"], [np.sum(dense[(int(i), int(j))] ** 2) for i, j in zip(r, c)])
    assert got["c_sample_tiles"].shape == (50, b, b)
    for i, j, t in zip(got["c_sample_row"], got["c_sample_col"], got["c_sample_tiles"]):
        assert np.array_equal(t, dense[(int(i), int(j))])


def test_peaks_name_their_source():
    sys.path.insert(0, ROOT)
    import bench
    for fn in (bench.fp64_peak, bench.tf32_peak, bench.hbm_peak):
        v, src = fn()
        assert v > 0 and ("measured" in src or "MEASURED" in src or "FALLBACK" in src)
