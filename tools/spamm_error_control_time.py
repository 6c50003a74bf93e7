#!/usr/bin/env python
"""Cost and tightness of SpAMM error control on the bench workload's law: N = 65536, b = 64, lambda = 0.01 decay generated on
the device, fp64 and fp32; the general product A*A, and symm_square on the upper triangle U of the symmetric law.
eps = rel * ||A||_F^2 (||U's full symmetric matrix||_F^2 for symm_square) for rel in {1e-4, 1e-6, 1e-8, 1e-10}.

Per (dtype, product): the time of spamm_error_bounds for 16 taus and of hbsm_spamm_errors (the a-priori host estimator) for
the same 16 taus.  Per eps: the time of spamm_tau_for_error, the chosen tau, its product count and SpAMM time, the measured
error (the engine's exact product minus the SpAMM product, Frobenius; with symm_square the norm of sym(triu(.)); so at fp32
it includes the leaf GEMMs' rounding) and bound / error; and the tau a host search over hbsm_spamm_errors picks for the same
eps (a geometric grid of 128 taus, then 16 taus inside the bracket), its product count and SpAMM time.  Times are CUDA events
on the engine stream around calls that end in a host synchronisation: best and median of --reps after one warm-up call.
Writes one JSON object per line to --out (default profiles/r06_spamm_error_control.jsonl)."""
import argparse
import json
import os
import subprocess
import sys
import time

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
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    r = fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return r, e0.elapsed_time(e1)


def repeated(fn, stream, reps):
    """warm-up call, then reps timed calls: (last result, best ms, median ms)"""
    fn()
    ts = []
    r = None
    for _ in range(reps):
        r, t = timed(fn, stream)
        ts.append(t)
    return r, min(ts), float(np.median(ts))


def spamm_product(M, sym, tau, stream):
    P = H(M.dtype)
    if sym:
        (nm, _), ms = timed(lambda: H.symm_square_spamm(M, P, tau), stream)
    else:
        (nm, _), ms = timed(lambda: H.spamm(M, False, M, False, P, tau, True), stream)
    return P, nm, ms


def error_norm(Pex, P, sym, n):
    """||Pex - P||_F, or ||sym(triu(Pex - P))||_F = sqrt(2 ||D||_F^2 - ||diag D||^2) with symm_square (both upper)"""
    D = H(P.dtype)
    N = H(P.dtype)
    N.rescale(P, -1.0)
    H.add(Pex, N, D)
    f2 = float(D.get_frob_squared())
    if sym:
        idx = np.arange(n, dtype=np.int32)
        d = D.get_values(idx, idx).astype(np.float64)
        f2 = 2.0 * f2 - float(d @ d)
    return float(np.sqrt(max(f2, 0.0)))


def old_search(X, scale, epss):
    """per eps, the largest tau whose hbsm_spamm_errors estimate is <= eps, and that estimate: a geometric grid of 128 taus,
    then 16 taus inside each eps's bracket (all eps in one call)"""
    grid = np.geomspace(1e-18, 1.0, 128) * np.sqrt(scale)
    err = H.get_spamm_errors(X, False, X, False, grid).astype(np.float64)
    br = []
    for eps in epss:
        ok = np.flatnonzero(err <= eps)
        k = ok[-1] if len(ok) else -1
        br.append((grid[k] if k >= 0 else 0.0, err[k] if k >= 0 else 0.0, grid[k + 1] if k + 1 < len(grid) else None))
    fine = [np.linspace(lo, hi, 18)[1:-1] if hi is not None else np.zeros(16) for lo, _, hi in br]
    e2 = H.get_spamm_errors(X, False, X, False, np.concatenate(fine)).astype(np.float64).reshape(len(epss), 16)
    out = []
    for eps, (lo, elo, hi), f, e in zip(epss, br, fine, e2):
        k = np.flatnonzero(e <= eps) if hi is not None else []
        out.append((float(f[k[-1]]), float(e[k[-1]])) if len(k) else (float(lo), float(elo)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--b", type=int, default=64)
    ap.add_argument("--lam", type=float, default=0.01)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--rels", default="1e-4,1e-6,1e-8,1e-10")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_spamm_error_control.jsonl"))
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

    emit({"context": device_context(), "n": a.n, "b": a.b, "lambda": a.lam, "reps": a.reps,
          "eps": "rel * ||A||_F^2 (general), rel * ||sym(U)||_F^2 (symm_square)"})
    n, b = a.n, a.b
    W = G.decay_width(a.lam)
    rels = [float(x) for x in a.rels.split(",")]
    for dtype in (np.float64, np.float32):
        A = H(dtype, b)
        A.generate_decay(n, a.lam, W, 1)
        A.update_internal_info()
        S = H(dtype, b)
        S.generate_decay(n, a.lam, W, 2, symmetric=True)
        S.update_internal_info()
        U = H(dtype, b)
        S.get_upper_triangle(U)
        U.update_internal_info()
        for sym, M, X in ((False, A, A), (True, U, S)):   # X: the operand of the old estimator (sym: the full matrix)
            scale = float(X.get_frob_squared())
            Pex = H(dtype)
            if sym:
                _, ex_ms = timed(lambda: H.symm_square(M, Pex), stream)
            else:
                _, ex_ms = timed(lambda: H.multiply(M, False, M, False, Pex), stream)
            taus16 = list(np.geomspace(1e-14, 1e-2, 16) * np.sqrt(scale))
            (bnd16, ns16), bt_best, bt_med = repeated(lambda: H.spamm_error_bounds(M, 0, M, 0, taus16, symm_square=sym), stream, a.reps)
            t0 = time.perf_counter()
            old16 = H.get_spamm_errors(X, False, X, False, taus16).astype(np.float64)
            old16_ms = 1e3 * (time.perf_counter() - t0)
            epss = [r * scale for r in rels]
            t0 = time.perf_counter()
            old = old_search(X, scale, epss) if old16_ms < 60e3 else [(None, None)] * len(epss)
            old_search_ms = 1e3 * (time.perf_counter() - t0)
            emit({"dtype": np.dtype(dtype).name, "product": "symm_square(U)" if sym else "A*A", "frob_sq": scale,
                  "exact_product_ms": ex_ms,
                  "bounds16_ms_best": bt_best, "bounds16_ms_median": bt_med, "taus16": taus16, "bounds16": list(bnd16),
                  "n_skipped16": [int(x) for x in ns16], "spamm_errors16_ms": old16_ms,
                  "spamm_errors16": list(old16), "old_search_ms_all_eps": old_search_ms,
                  "old_estimator_operand": "S (full symmetric), general product" if sym else "A"})
            for rel, eps, (otau, oest) in zip(rels, epss, old):
                info, tf_best, tf_med = repeated(lambda: H.spamm_tau_for_error(M, 0, M, 0, eps, symm_square=sym), stream, a.reps)
                P, nm, sp_ms = spamm_product(M, sym, info["tau"], stream)
                _, nm2, sp_ms2 = spamm_product(M, sym, info["tau"], stream)
                err = error_norm(Pex, P, sym, n)
                del P
                onm = o_ms = o_ms2 = oerr = None
                if otau is not None:   # (the host estimator's search is skipped when one call takes over a minute)
                    Po, onm, o_ms = spamm_product(M, sym, otau, stream)
                    _, _, o_ms2 = spamm_product(M, sym, otau, stream)
                    oerr = error_norm(Pex, Po, sym, n)
                    del Po
                emit({"dtype": np.dtype(dtype).name, "product": "symm_square(U)" if sym else "A*A", "rel": rel, "eps": eps,
                      "tau_for_error_ms_best": tf_best, "tau_for_error_ms_median": tf_med, **info,
                      "products": nm, "spamm_ms": [sp_ms, sp_ms2], "measured_error": err,
                      "bound_over_error": (info["bound"] / err) if err > 0 else None,
                      "old_tau": otau, "old_products": onm, "old_spamm_ms": [o_ms, o_ms2] if o_ms is not None else None, "old_measured_error": oerr,
                      "old_estimate_at_old_tau": oest})
            del Pex
        del A, S, U
    out.close()


if __name__ == "__main__":
    main()
