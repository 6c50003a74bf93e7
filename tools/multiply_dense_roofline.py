#!/usr/bin/env python
"""Roofline of Y = op(A) * X (hbsm_multiply_dense_device) on the bench workload's law: N = 65536, b = 64, lambda = 0.01
decay generated on the device, fp64 and fp32, m in {1, 8, 32} x {N, T, SYM_UPPER} (SYM_UPPER on the upper triangle of the
symmetric law).  Each case: the first call alone (for m = 1, the first case of each operand and op, it also builds the line index the op
walks), then >= 10 timed calls, CUDA events on the
torch stream the call is ordered on, the GPU kept busy while the call is enqueued.  Algorithmic bytes
ceil(m/MC) * L_read * b^2 * s + (K + M * (1 + [beta != 0])) * m * s with L_read = L (N, T) or 2 L_off + L_diag (SYM_UPPER),
flops 2 b^2 m per tile application.  Then the time and iterations of spectral_norm_estimate on the same matrices.
Writes one JSON object per line to --out (default profiles/r03_multiply_dense.jsonl)."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import hierarchical_block_sparse_lib_b200 as hb  # noqa: E402
from hierarchical_block_sparse_lib_b200 import generators as G  # noqa: E402

H = hb.HierarchicalBlockSparseMatrix


def hbm_peak():   # the denominator bench.py uses
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), \
            "MEASURED_PEAKS.json hbm_gbs (driver-written copy bandwidth)"
    except Exception:
        return 6650.0, "FALLBACK: B200_PROFILING.md copy bandwidth (of fallback)"


def fp64_peak():
    for nm in ("r02_peak_fp64.json", "r01_peak_fp64.json"):
        p = os.path.join(ROOT, "profiles", nm)
        if os.path.exists(p):
            return float(json.load(open(p))["dmma884_sustained_tflops"]), "measured: tools/peak_fp64.cu, profiles/%s" % nm
    return 37.2, "FALLBACK (no probe file): 148 SM x 128 FP64 flop/clk x 1.965 GHz"


def device_context():
    ctx = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        ctx["power_limit_w"] = float(q[0])
        ctx["sm_max_mhz"] = float(q[1])
    except Exception as e:   # reported, not guessed
        ctx["power_limit_w"] = "unavailable: %s" % e
    return ctx


def mc_of(m):   # the column chunk the kernel runs (csrc/dense.cu launch_dense)
    return 8 if m <= 8 else (16 if m <= 16 else 32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--b", type=int, default=64)
    ap.add_argument("--lam", type=float, default=0.01)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_multiply_dense.jsonl"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs the GPU (no CPU timing is reported)"
    hb.init(0)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    peak, peak_src = hbm_peak()
    dpeak, dpeak_src = fp64_peak()
    emit({"context": device_context(), "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "fp64_dmma_peak_tflops": dpeak,
          "fp64_dmma_peak_source": dpeak_src, "n": a.n, "b": a.b, "lambda": a.lam, "beta": 0.0,
          "inputs": "A (about 2.9 GB in fp64) exceeds the 126 MB L2 and streams from HBM on every call; X (at most 16 MB) "
                    "stays in L2 between calls"})
    n, b = a.n, a.b
    W = G.decay_width(a.lam)
    s = torch.cuda.Stream()
    for dtype in (np.float64, np.float32):
        es = np.dtype(dtype).itemsize
        tdt = torch.float64 if dtype == np.float64 else torch.float32
        A = H(dtype, b)
        A.generate_decay(n, a.lam, W, 1)
        S = H(dtype, b)
        S.generate_decay(n, a.lam, W, 2, symmetric=True)
        U = H(dtype, b)
        S.get_upper_triangle(U)
        del S
        L, LU = A.get_n_blocks(), U.get_n_blocks()
        bi, bj, _, _ = U.export_leaves(tiles=False, norms=False)
        L_diag = int(np.sum(bi == bj))
        for op, M in (("N", A), ("T", A), ("SYM_UPPER", U)):
            L_read = L if op != "SYM_UPPER" else 2 * (LU - L_diag) + L_diag
            for m in (1, 8, 32):
                with torch.cuda.stream(s):
                    X = torch.randn((m, n), dtype=tdt, device="cuda").t()   # column-major, ld = n
                    Y = torch.zeros((m, n), dtype=tdt, device="cuda").t()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    e0.record(s); M.multiply_dense(X, op=op, Y=Y); e1.record(s)
                    torch.cuda.synchronize()
                    first = e0.elapsed_time(e1)
                    ts = []
                    for _ in range(a.reps):
                        torch.cuda._sleep(2_000_000)   # keeps the GPU busy while the call below is enqueued
                        e0.record(s); M.multiply_dense(X, op=op, Y=Y); e1.record(s)
                        torch.cuda.synchronize()
                        ts.append(e0.elapsed_time(e1))
                MC = mc_of(m)
                nbytes = math.ceil(m / MC) * L_read * b * b * es + (n + n) * m * es
                flops = 2.0 * b * b * m * L_read
                best, med = min(ts), float(np.median(ts))
                d = {"dtype": np.dtype(dtype).name, "op": op, "m": m, "MC": MC, "tiles": L if op != "SYM_UPPER" else LU,
                     "L_read": L_read, "first_call_ms": first, "first_call_builds_line_index": m == 1, "best_ms": best, "median_ms": med, "runs": len(ts),
                     "algorithmic_bytes": nbytes, "GBps_best": nbytes / best / 1e6, "frac_hbm_best": nbytes / best / 1e6 / peak,
                     "GBps_median": nbytes / med / 1e6, "frac_hbm_median": nbytes / med / 1e6 / peak,
                     "flops": flops, "TFps_best": flops / best / 1e9}
                if dtype == np.float64:
                    d["frac_dmma_peak_best"] = flops / best / 1e9 / dpeak
                emit(d)
                del X, Y
        for name, M, sym in (("A^T A", A, False), ("triu(S)+striu(S)^T", U, True)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nrm, lo, hi, it = M.spectral_norm_estimate(symmetric_upper=sym, max_iter=200, rel_tol=1e-8)
            ms = (time.perf_counter() - t0) * 1e3
            emit({"dtype": np.dtype(dtype).name, "spectral_norm_on": name, "max_iter": 200, "rel_tol": 1e-8, "ms": ms,
                  "n_iter": it, "ms_per_iter": ms / max(it, 1), "norm": nrm, "lambda_min": lo, "lambda_max": hi})
        del A, U
    out.close()


if __name__ == "__main__":
    main()
