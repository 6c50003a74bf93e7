#!/usr/bin/env python
"""The accumulating product (hbsm_multiply_accumulate) against the four-call composition it replaces, on the bench
workload's law: N = 65536, b = 64, lambda = 0.01 decay generated on the device, fp64 and fp32.

Workloads:
  purify        X <- 2X - X*X in place (C is A is B), multiply
  purify_spamm  the same step with SpAMM at two tau (tau^2 = the 50th / 90th percentile of the leaf ||.||_F^2 of X, times
                the median: a part of the products is skipped)
  gemm_acc      C <- A*B + C with C_old on A's pattern (C a copy of A)
Per workload and dtype: the fused call (CUDA events on the engine stream around the call, which ends in a host
synchronisation) with its GEMM stage time (hbsm_stage_times_last), the composition multiply / rescale / rescale / add
(each call synchronises the host), and a plain multiply / spamm on the same operands: fused minus plain is the cost of
reading C_old and scaling in the epilogue.  Peak device memory is the high-water mark of the engine's stream-ordered pool
(the device's default pool, CU_MEMPOOL_ATTR_USED_MEM_HIGH), reset before each measured call after the engine's cache of
large blocks is returned to the pool; reported as the peak above what was in use at the reset.  During the measured call
that cache (BlockCache, blocks of 64 MiB and more kept for exact-size reuse) holds freed large temporaries, and the pool
counts them as used: the peak is live plus cached memory, which inflates the composition's figure (its freed P and scaled
copies) more than the fused call's.  Byte model of the C-side
traffic (the leaf GEMMs' operand reads are the same in all three): fused reads C_old and writes the union once,
(L_old + L_out) b^2 s; the composition writes P, reads and writes it in rescale, reads and writes C_old in rescale, and
reads both scaled copies and writes the result in add, (4 L_P + 3 L_old + L_out) b^2 s.
Writes one JSON object per line to --out (default profiles/r05_multiply_accumulate.jsonl)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import hierarchical_block_sparse_lib_b200 as hb  # noqa: E402
from hierarchical_block_sparse_lib_b200 import _capi  # noqa: E402
from hierarchical_block_sparse_lib_b200 import generators as G  # noqa: E402

H = hb.HierarchicalBlockSparseMatrix
CU_MEMPOOL_ATTR_USED_MEM_CURRENT, CU_MEMPOOL_ATTR_USED_MEM_HIGH = 7, 8


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


class Pool:
    """the device's default memory pool (the one the engine allocates from), through the driver API"""
    def __init__(self):
        self.cu = C.CDLL("libcuda.so.1")
        dev = C.c_int(0)
        assert self.cu.cuDeviceGet(C.byref(dev), 0) == 0
        self.pool = C.c_void_p()
        assert self.cu.cuDeviceGetDefaultMemPool(C.byref(self.pool), dev) == 0

    def get(self, attr):
        v = C.c_uint64(0)
        assert self.cu.cuMemPoolGetAttribute(self.pool, attr, C.byref(v)) == 0
        return v.value

    def reset(self):
        """returns the bytes in use; the high-water mark restarts there"""
        _capi.check(_capi.lib().hbsm_finalize())   # synchronises and hands the engine's cached large blocks back to the pool
        z = C.c_uint64(0)
        assert self.cu.cuMemPoolSetAttribute(self.pool, CU_MEMPOOL_ATTR_USED_MEM_HIGH, C.byref(z)) == 0
        return self.get(CU_MEMPOOL_ATTR_USED_MEM_CURRENT)

    def peak_above(self, base):
        return self.get(CU_MEMPOOL_ATTR_USED_MEM_HIGH) - base


def timed(fn, stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    r = fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return r, e0.elapsed_time(e1)


def copy_of(X):
    Y = H(X.dtype, X.get_params().blocksize)
    Y.copy(X)
    return Y


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--b", type=int, default=64)
    ap.add_argument("--lam", type=float, default=0.01)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_multiply_accumulate.jsonl"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs the GPU (no CPU timing is reported)"
    hb.init(0)
    stream = torch.cuda.ExternalStream(_capi.lib().hbsm_stream())
    pool = Pool()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    emit({"context": device_context(), "n": a.n, "b": a.b, "lambda": a.lam, "reps": a.reps,
          "timing": "best and median of reps after one warm-up run of each variant; operands exceed the 126 MB L2"})
    n, b = a.n, a.b
    W = G.decay_width(a.lam)
    for dtype in (np.float64, np.float32):
        s = np.dtype(dtype).itemsize
        tb = b * b * s
        X0 = H(dtype, b)
        X0.generate_decay(n, a.lam, W, 1)
        B0 = H(dtype, b)
        B0.generate_decay(n, a.lam, W, 2)
        X0.update_internal_info()
        nsq = X0.export_leaves(tiles=False)[2].astype(np.float64)
        med = float(np.median(nsq))
        taus = [float(np.sqrt(np.quantile(nsq, q) * med)) for q in (0.5, 0.9)]
        work = [("purify", None), ("purify_spamm", taus[0]), ("purify_spamm", taus[1]), ("gemm_acc", None)]
        for name, tau in work:
            if name == "gemm_acc":
                A, B, alpha, beta = X0, B0, 1.0, 1.0
            else:
                A, B, alpha, beta = X0, X0, -1.0, 2.0

            def fused():
                Cm = copy_of(A)   # C_old: X itself (purify: C is A is B), or a copy of A (gemm_acc)
                Aop = Cm if name != "gemm_acc" else A
                Bop = Cm if name != "gemm_acc" else B
                Cm.update_internal_info()   # the cached leaf norms SpAMM tests, as X0's
                base = pool.reset()
                if tau is None:
                    (nm, nr), ms = timed(lambda: H.multiply_accumulate(Aop, 0, Bop, 0, Cm, alpha, beta), stream)
                else:
                    (nm, nr), ms = timed(lambda: H.spamm_accumulate(Aop, 0, Bop, 0, Cm, alpha, beta, tau), stream)
                st = hb.stage_times()
                return {"ms": ms, "gemm_ms": st["gemm_ms"], "peak_bytes": pool.peak_above(base), "n_mults": nm,
                        "tiles_out": nr, "kernel": st["gemm_kernel"]}, Cm

            def composition():
                Cold = copy_of(A)
                base = pool.reset()

                def run():
                    P = H(dtype, b)
                    if tau is None:
                        H.multiply(A, 0, B, 0, P)
                    else:
                        H.spamm(A, 0, B, 0, P, tau)
                    P1 = H(dtype, b)
                    P1.rescale(P, alpha)
                    del P
                    C1 = H(dtype, b)
                    C1.rescale(Cold, beta)
                    R = H(dtype, b)
                    H.add(P1, C1, R)
                    return R
                R, ms = timed(run, stream)
                return {"ms": ms, "peak_bytes": pool.peak_above(base)}, R, Cold

            def plain():
                P = H(dtype, b)
                base = pool.reset()
                if tau is None:
                    _, ms = timed(lambda: H.multiply(A, 0, B, 0, P), stream)
                else:
                    _, ms = timed(lambda: H.spamm(A, 0, B, 0, P, tau), stream)
                st = hb.stage_times()
                return {"ms": ms, "gemm_ms": st["gemm_ms"], "peak_bytes": pool.peak_above(base), "tiles": P.get_n_blocks()}

            runs = {"fused": [], "composition": [], "plain": []}
            check = None
            for rep in range(a.reps + 1):   # rep 0 warms every variant
                f, Cm = fused()
                c, R, Cold = composition()
                p = plain()
                if rep == 0:
                    fb, rb = Cm.export_leaves(norms=False), R.export_leaves(norms=False)
                    it = np.uint64 if dtype == np.float64 else np.uint32
                    check = all(np.array_equal(x.view(it) if x.dtype.kind == "f" else x, y.view(it) if y.dtype.kind == "f" else y)
                                for x, y in zip((fb[0], fb[1], fb[3]), (rb[0], rb[1], rb[3])))
                    L_old, L_out, L_P = Cold.get_n_blocks(), Cm.get_n_blocks(), p["tiles"]
                    continue
                runs["fused"].append(f)
                runs["composition"].append(c)
                runs["plain"].append(p)
                del Cm, R, Cold

            def summ(rs, key):
                v = sorted(r[key] for r in rs)
                return {"best": v[0], "median": v[len(v) // 2]}

            d = {"dtype": np.dtype(dtype).name, "workload": name, "tau": tau, "alpha": alpha, "beta": beta,
                 "bitwise_equal_to_composition": bool(check), "n_mults": runs["fused"][0]["n_mults"],
                 "gemm_kernel": runs["fused"][0]["kernel"], "tiles_old": L_old, "tiles_P": L_P, "tiles_out": L_out,
                 "fused_ms": summ(runs["fused"], "ms"), "fused_gemm_ms": summ(runs["fused"], "gemm_ms"),
                 "fused_peak_bytes": max(r["peak_bytes"] for r in runs["fused"]),
                 "composition_ms": summ(runs["composition"], "ms"),
                 "composition_peak_bytes": max(r["peak_bytes"] for r in runs["composition"]),
                 "plain_ms": summ(runs["plain"], "ms"), "plain_gemm_ms": summ(runs["plain"], "gemm_ms"),
                 "plain_peak_bytes": max(r["peak_bytes"] for r in runs["plain"]),
                 "model_c_bytes_fused": (L_old + L_out) * tb,
                 "model_c_bytes_composition": (4 * L_P + 3 * L_old + L_out) * tb}
            d["speedup_vs_composition"] = d["composition_ms"]["best"] / d["fused_ms"]["best"]
            d["epilogue_cost_ms"] = d["fused_gemm_ms"]["best"] - d["plain_gemm_ms"]["best"]
            emit(d)
        del X0, B0
    out.close()


if __name__ == "__main__":
    main()
