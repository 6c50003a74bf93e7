#!/usr/bin/env python
"""Cost and payoff of spectral_block_trunc on the bench workload's law: N = 65536, b = 64, lambda = 0.01 decay generated
on the device, fp64 and fp32; the general operator on the decay matrix A, the symmetric-upper operator on the upper triangle
U of the symmetric law; eps = rel * ||op||_2 for rel in {1e-4, 1e-6, 1e-8} (||op||_2 from spectral_norm_estimate).

Per call: the wall time (CUDA events on the engine stream around the whole call, which ends in a host synchronisation),
n_decisions and Lanczos steps, n_dropped against n_frob (the leaves the Frobenius bound alone drops), and the bytes of the
chosen error matrix E_v with the time of one Lanczos step on it (truncation_spectral_errors on E_v for a fixed number of
steps; DESIGN section 9's byte model: (2 L_off + L_diag) b^2 s for the symmetric operator, 2 L b^2 s for E^T E (one N and
one T product), plus 3 vector passes).  The payoff: the time of symm_square_spamm(tau = 0) (symmetric) or multiply
(general) on the spectrally truncated C against the Frobenius-truncated C at the same eps.
Writes one JSON object per line to --out (default profiles/r04_spectral_trunc.jsonl)."""
import argparse
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


def timed(fn, stream):
    """(result, ms) of fn() between two CUDA events on the engine stream"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    r = fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return r, e0.elapsed_time(e1)


def leaf_norms(A):
    import ctypes as C
    n = C.c_size_t(0)
    _capi.check(_capi.lib().hbsm_leaf_norms(A._h, 0, None, C.byref(n)))
    out = np.zeros(n.value, A.dtype)
    _capi.check(_capi.lib().hbsm_leaf_norms(A._h, n.value, out.ctypes.data_as(C.c_void_p), C.byref(n)))
    return out


def frob_tau(nsq, w, eps):
    """tau whose frob_block_trunc drops exactly the leaves of the largest level whose Frobenius bound w * sum <= eps^2"""
    lv, inv = np.unique(nsq, return_inverse=True)
    cnt = np.bincount(inv)
    cum = np.cumsum(w * lv.astype(np.float64) * cnt)
    k = int(np.searchsorted(cum, eps * eps, side="right")) - 1
    lo = float(lv[k]) if k >= 0 else 0.0
    hi = float(lv[k + 1]) if k + 1 < len(lv) else 2 * lo + 1.0
    return float(np.sqrt((lo + hi) / 2)) if k >= 0 else float(np.sqrt(float(lv[0]) / 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--b", type=int, default=64)
    ap.add_argument("--lam", type=float, default=0.01)
    ap.add_argument("--max-iter", type=int, default=100)
    ap.add_argument("--step-iters", type=int, default=30)
    ap.add_argument("--rels", default="1e-4,1e-6,1e-8")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_spectral_trunc.jsonl"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs the GPU (no CPU timing is reported)"
    hb.init(0)
    stream = torch.cuda.ExternalStream(_capi.lib().hbsm_stream())
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    emit({"context": device_context(), "n": a.n, "b": a.b, "lambda": a.lam, "max_iter": a.max_iter,
          "inputs": "A and U exceed the 126 MB L2; E_v's tiles may not"})
    n, b = a.n, a.b
    W = G.decay_width(a.lam)
    for dtype in (np.float64, np.float32):
        es = np.dtype(dtype).itemsize
        A = H(dtype, b)
        A.generate_decay(n, a.lam, W, 1)
        S = H(dtype, b)
        S.generate_decay(n, a.lam, W, 2, symmetric=True)
        U = H(dtype, b)
        S.get_upper_triangle(U)
        del S
        for sym, M in ((True, U), (False, A)):
            nrm = M.spectral_norm_estimate(symmetric_upper=sym, max_iter=200, rel_tol=1e-8)[0]
            nsq = leaf_norms(M)
            bi, bj, _, _ = M.export_leaves(tiles=False, norms=False)
            for rel in (float(x) for x in a.rels.split(",")):
                eps = rel * nrm
                Cs = H(dtype)
                info, ms = timed(lambda: M.spectral_block_trunc(Cs, eps, symmetric_upper=sym, max_iter=a.max_iter), stream)
                Cs2 = H(dtype)
                info2, ms2 = timed(lambda: M.spectral_block_trunc(Cs2, eps, symmetric_upper=sym, max_iter=a.max_iter), stream)
                assert info2 == info
                del Cs2
                drop = nsq <= info["drop_nsq"]
                diag = bi == bj
                L_E = int(drop.sum())
                L_read = (2 * int((drop & ~diag).sum()) + int((drop & diag).sum())) if sym else 2 * L_E
                step_bytes = L_read * b * b * es + 3 * n * es
                step_ms = None
                if L_E:
                    nxt = nsq[nsq > info["drop_nsq"]]
                    tau = float(np.sqrt((info["drop_nsq"] + (nxt.min() if len(nxt) else 2 * info["drop_nsq"] + 1)) / 2))
                    M.truncation_spectral_errors([tau], symmetric_upper=sym, max_iter=2, rel_tol=1e-300)   # warm
                    (_, its), tms = timed(lambda: M.truncation_spectral_errors([tau], symmetric_upper=sym, max_iter=a.step_iters,
                                                                                rel_tol=1e-300), stream)
                    step_ms = tms / max(int(its[0]), 1)
                Cf = H(dtype)
                tf = frob_tau(nsq, 2.0 if sym else 1.0, eps)
                M.frob_block_trunc(Cf, tf)
                prod = {}
                for name, X in (("spectral", Cs), ("frobenius", Cf)):
                    ts = []
                    for _ in range(3):
                        P = H(dtype)
                        if sym:
                            _, t = timed(lambda: H.symm_square_spamm(X, P, 0.0), stream)
                        else:
                            _, t = timed(lambda: H.multiply(X, False, X, False, P), stream)
                        ts.append(t)
                        del P
                    prod[name] = {"tiles": X.get_n_blocks(), "first_ms": ts[0], "best_ms": min(ts[1:])}
                d = {"dtype": np.dtype(dtype).name, "operator": "triu(U)+striu(U)^T" if sym else "A (E^T E)", "rel": rel,
                     "eps": eps, "op_norm": nrm, "tiles": len(nsq), "call_ms": ms, "call_ms_repeat": ms2,
                     "n_dropped": info["n_dropped"], "n_frob": info["n_frob"], "drop_nsq": info["drop_nsq"],
                     "err_bound": info["err_bound"], "certified_by_lanczos": info["certified_by_lanczos"],
                     "n_decisions": info["n_decisions"], "lanczos_steps": info["lanczos_steps"],
                     "E_tiles": L_E, "E_bytes": L_E * b * b * es, "step_bytes": step_bytes, "step_ms": step_ms,
                     "step_GBps": (step_bytes / step_ms / 1e6) if step_ms else None,
                     "product": "symm_square_spamm(tau=0)" if sym else "multiply(C, C)",
                     "frob_tau": tf, "payoff": prod,
                     "product_speedup": prod["frobenius"]["best_ms"] / prod["spectral"]["best_ms"]}
                emit(d)
                del Cs, Cf
        del A, U
    out.close()


if __name__ == "__main__":
    main()
