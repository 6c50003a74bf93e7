#!/usr/bin/env python
"""bench.py -- the hot path on the configuration BASELINE.json's metric is quoted on:
fp64 SpAMM C = A*B (tau = 1e-6) of two N = 65536 exponential-decay matrices, leaf 64 (SURVEY 8d cfg-2 law,
lambda = 0.01), at 1/2/4/8 B200 (strong scaling: C sharded by block rows, B halo exchanged over NCCL).

One JSON line on stdout (rank 0).  `value` = leaf-GEMM FP64 TFLOP/s over the WHOLE multiply (2 b^3 P / time per
multiply, task-list build included, inputs resident in HBM); `ms_per_step` = time per multiply; `e2e` = the same
through the C ABI with HOST buffers (pinned H2D of A and B tiles, norm refresh, SpAMM, D2H of all C tiles).
`--impl reference` times the unmodified reference (oracle/_ref, OpenMP on the host cores) on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
from hierarchical_block_sparse_lib_b200 import _capi  # noqa: E402

# bounded samples of the workload for the host-side legs: leading principal block of the same matrices, same law.
# cpu_baseline (inside the native arm's run): 8192; reference arm (its own run, a minute of host time): 16384 = the size of
# BASELINE.json configs[1].  HBSM_CPU_SAMPLE_N=65536 runs the FULL problem (one step: profiles/r02_reference_full_size.json).
CPU_SAMPLE_N = int(os.environ.get("HBSM_CPU_SAMPLE_N", "8192"))
REF_ARM_SAMPLE_N = int(os.environ.get("HBSM_CPU_SAMPLE_N", "16384"))
PROFILES = os.path.join(ROOT, "profiles")


def _first_json(*names):
    for nm in names:
        try:
            return json.loads(open(os.path.join(PROFILES, nm)).read().strip().splitlines()[0]), nm
        except Exception:
            continue
    return None, None


def fp64_peak():
    """FP64 DMMA peak: MEASURED_PEAKS.json has no FP64 entry, so the denominator is this repo's own probe
    (tools/peak_fp64.cu, run on this pool's B200s); 148 SM x 128 flop/clk x 1.965 GHz = 37.2 is the same number."""
    d, nm = _first_json("r02_peak_fp64.json", "r01_peak_fp64.json")
    if d is not None:
        return float(d["dmma884_sustained_tflops"]), "measured: tools/peak_fp64.cu (mma.sync DMMA, sustained 2 s) on this pool's B200, profiles/%s; MEASURED_PEAKS.json has no FP64 entry" % nm
    return 37.2, "FALLBACK (no probe file): 148 SM x 128 FP64 flop/clk x 1.965 GHz"


def tf32_peak():
    """TF32 tcgen05 peak (tools/peak_tf32.cu, M=128 N=256, sustained).  The fp32 leaf GEMM issues three TF32 MMAs per
    fp32 product (hi*hi + hi*lo + lo*hi), so its fp32 result rate is bounded by a third of this."""
    d, nm = _first_json("r02_peak_tf32.json")
    if d is not None:
        return float(d["tf32_m128n256_sustained_tflops"]), "measured: tools/peak_tf32.cu (tcgen05.mma kind::tf32 M=128 N=256, sustained) on this pool's B200, profiles/%s" % nm
    return 1125.0, "FALLBACK (no probe file): nominal dense TF32 = bf16/2"


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (driver-written copy bandwidth)"
    except Exception:
        return 6650.0, "FALLBACK: B200_PROFILING.md copy bandwidth (of fallback)"


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (nvidia-smi, every 50 ms)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------
# workloads: the headline (BASELINE.json `metric`) and BASELINE.json configs[0..4] (--config 1..5)
# ---------------------------------------------------------------------------------------------------
def config_cases(cfg, n=None, b=None, lam=None):
    """List of cases of a configuration; the FIRST is the primary one (`value`, `ms_per_step`, `roofline` are quoted on it)."""
    if cfg == "headline":
        return [dict(name="spamm NN", op="spamm", gen="decay", n=n or 65536, b=b or 64, lam=lam or 0.01, tau=1e-6, dtype="f64", tA=0, tB=0)]
    if cfg == "1":
        return [dict(name="multiply NN random 30%", op="multiply", gen="random", fill=0.3, n=n or 1024, b=b or 32, tau=0.0, dtype="f64", tA=0, tB=0)]
    if cfg == "2":
        return [dict(name="spamm NN lambda=%g" % l, op="spamm", gen="decay", n=n or 16384, b=b or 64, lam=l, tau=1e-6, dtype="f64", tA=0, tB=0)
                for l in ((lam,) if lam else (0.01, 0.05))]
    if cfg == "3":
        cs = [dict(name="symm_square_spamm tau=%g" % t, op="symm_square_spamm", gen="decay", symmetric=True, n=n or 65536, b=b or 64,
                   lam=lam or 0.05, tau=t, dtype="f64", tA=0, tB=0) for t in (1e-6, 1e-4, 1e-8, 1e-10)]
        cs.append(dict(name="symm_square exact", op="symm_square", gen="decay", symmetric=True, n=n or 65536, b=b or 64, lam=lam or 0.05,
                       tau=0.0, dtype="f64", tA=0, tB=0))
        return cs
    if cfg == "4":
        return [dict(name="spamm NN", op="spamm", gen="decay", n=n or 262144, b=b or 128, lam=lam or 0.01, tau=1e-6, dtype="f64", tA=0, tB=0)]
    if cfg == "5":
        cs = []
        for bb in ((b,) if b else (64, 32, 128, 256)):
            cs.append(dict(name="spamm A^T*B leaf %d" % bb, op="spamm", gen="decay", n=n or 65536, b=bb, lam=lam or 0.02, tau=1e-6, dtype="f32", tA=1, tB=0))
            cs.append(dict(name="spamm A*B^T leaf %d" % bb, op="spamm", gen="decay", n=n or 65536, b=bb, lam=lam or 0.02, tau=1e-6, dtype="f32", tA=0, tB=1))
            cs.append(dict(name="add leaf %d" % bb, op="add", gen="decay", n=n or 65536, b=bb, lam=lam or 0.02, tau=0.0, dtype="f32", tA=0, tB=0))
        return cs
    raise SystemExit("unknown --config %r" % cfg)


def case_config(c, n_gpus, cfg):
    law = ("exponential-decay a_ij=(0.5+0.5u)exp(-%g|i-j|) truncated at 1e-12%s" % (c["lam"], ", symmetric" if c.get("symmetric") else "")
           if c["gen"] == "decay" else "random block-sparse, %g block fill, entries uniform [-1,1)" % c["fill"])
    what = {"spamm": "SpAMM C=op(A)*op(B)", "multiply": "exact multiply C=A*B", "symm_square_spamm": "SpAMM-pruned symmetric square C=triu(A*A)",
            "symm_square": "exact symmetric square C=triu(A*A)", "add": "add C=A+B"}[c["op"]]
    which = "BASELINE.json metric workload (configs[1] law at the metric's N=65536)" if cfg == "headline" else "BASELINE.json configs[%d]" % (int(cfg) - 1)
    out = {"workload": "%s %s, %s, N=%d, leaf %d%s (%s)" % ({"f64": "fp64", "f32": "fp32"}[c["dtype"]], what, law, c["n"], c["b"],
                                                           ", tau=%g" % c["tau"] if "spamm" in c["op"] else "", which),
           "n": c["n"], "leaf": c["b"], "tau": c["tau"], "tA": c["tA"], "tB": c["tB"],
           "sharding": "single GPU" if n_gpus == 1 else "C and A by block rows over %d ranks, op(B) halo tiles exchanged over NCCL" % n_gpus,
           "l2": "operands and result exceed the 126 MB L2 many times over (no flush needed)" if c["n"] >= 16384 else
                 "small case: operands fit L2 (launch-latency bound; reported for completeness, not a bandwidth claim)"}
    if c["gen"] == "decay":
        out["lambda"] = c["lam"]
    return out


def np_dtype(c):
    return np.float64 if c["dtype"] == "f64" else np.float32


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the UNMODIFIED reference (oracle/_ref) on the host cores
# ---------------------------------------------------------------------------------------------------
def run_reference_cpu(c, steps, warmup, n_sample=None):
    """The reference's own OpenMP implementation (oracle/_ref = unmodified header compiled in place; the pinned plain-C port
    if that build did not travel) on the host cores, on the leading n_sample x n_sample block of the case's matrices (same law,
    same seeds).  Returns (tflops, ms, info)."""
    cores = host_threads()
    if "HBSM_REF_THREADS" in os.environ:
        os.environ["OMP_NUM_THREADS"] = os.environ["HBSM_REF_THREADS"]
    elif "TORCHELASTIC_RUN_ID" in os.environ or "OMP_NUM_THREADS" not in os.environ:
        # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is ONE process that gets all host threads
        os.environ["OMP_NUM_THREADS"] = str(cores)
    cores = int(os.environ["OMP_NUM_THREADS"])      # what the run really uses (reported as cpu_baseline.cores)
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    from oracle import pyoracle as po
    from hierarchical_block_sparse_lib_b200 import generators as G
    n_sample = min(n_sample or CPU_SAMPLE_N, c["n"])
    dt = np_dtype(c)
    kind = "reference" if os.path.exists(po.REF_SO) else "port"
    cls = po.RefMatrix if kind == "reference" else po.OrcMatrix
    t_asm = time.perf_counter()
    mats = []
    for seed in (1, 2):
        if c["gen"] == "decay":
            W = G.decay_width(c["lam"], 1e-12)
            r, cc, v = G.decay_coo(n_sample, c["lam"], min(W, n_sample - 1), 3 if c.get("symmetric") else seed, bool(c.get("symmetric")), dt)
        else:
            r, cc, v = G.random_block_sparse_coo(n_sample, c["b"], c["fill"], seed, dt)
        mats.append(po.from_coo(cls, c["b"], n_sample, n_sample, r, cc, v, dt))   # norms refreshed (updated=true)
        del r, cc, v
        if c.get("symmetric"):
            break
    if c.get("symmetric"):
        mats = [cls.upper(mats[0])] if c["op"] == "symm_square" else [mats[0], mats[0]]
        for m in mats:
            m.update()
    t_asm = time.perf_counter() - t_asm
    times, nm = [], 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        if c["op"] == "add":
            Cm = cls.add(mats[0], mats[1]); nm = Cm.n_blocks()
        elif c["op"] == "symm_square":
            Cm = cls.symm_square(mats[0]); nm = Cm.n_mults()
        else:   # spamm / multiply; the reference has no pruned symm_square: its spamm() on the full symmetric matrix stands in
            Cm, nm, nb, _ = cls.product(mats[0], c["tA"], mats[1], c["tB"], spamm="spamm" in c["op"], tau=c["tau"])
        dtm = time.perf_counter() - t0
        del Cm
        if i >= warmup:
            times.append(dtm)
    ms = 1e3 * float(np.mean(times))
    g = -(-n_sample // c["b"])
    if c["op"] == "add":
        rate = 3.0 * nm * c["b"] ** 2 * np.dtype(dt).itemsize / (ms * 1e-3) / 1e9
    else:
        rate = 2.0 * c["b"] ** 3 * nm / (ms * 1e-3) / 1e12
    blas = po.RefMatrix.blas_kind() if kind == "reference" else "builtin loops"
    info = {"kind": kind, "cores": cores if kind == "reference" else 1, "n_sample": n_sample,
            "sample": "%s of the same matrices (%s, b=%d): %d leaf %s per call, whole %s() call (bucket reserve + symbolic + numeric; "
                      "(N/b+1)^3 = %d hash buckets, H:3968-3970), OpenMP over hash buckets, BLAS=%s; assembly (not timed) %.1f s"
                      % ("the FULL %dx%d problem" % (n_sample, n_sample) if n_sample == c["n"] else "leading %dx%d block" % (n_sample, n_sample),
                         c["name"], c["b"], nm, "blocks" if c["op"] == "add" else "products", c["op"], (g + 1) ** 3,
                         os.path.basename(blas), t_asm),
            "ms_per_call": ms, "products": nm}
    return rate, ms, info


def metric_of(c):
    if c["op"] == "add":
        return "add_%s_GBps" % c["dtype"], "GB/s"
    return ("%s_fp%s_leaf_tflops" % ("spamm" if "spamm" in c["op"] else "multiply", c["dtype"][1:])), "TFLOP/s"


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = config_cases(args.config, args.n, args.leaf, args.lam)[0]
    rate, ms, info = run_reference_cpu(c, args.steps, args.warmup, REF_ARM_SAMPLE_N)
    metric, unit = metric_of(c)
    cfg = case_config(c, args.gpus, args.config)
    # the arm runs a bounded SAMPLE of the workload: say so where the driver compares configs (n = what was really run)
    cfg["sharding"] = "host cores only (no GPU)"
    if info["n_sample"] != c["n"]:
        cfg["n"] = info["n_sample"]; cfg["sample_of"] = c["n"]
        cfg["workload"] += " -- reference arm timed on the leading %dx%d block (rates are compared, not times)" % (info["n_sample"], info["n_sample"])
    line = {"metric": metric, "value": rate, "unit": unit, "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": c["dtype"], "data": "synthetic",
            "config": cfg, "products_per_multiply": info["products"],
            "cpu_baseline": {"value": rate, "unit": unit, "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]},
            "e2e": {"value": rate, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# native arm, one GPU
# ---------------------------------------------------------------------------------------------------
def build_operands(H, G, c, lo=0, hi=-1):
    """Engine operands of a case with refreshed norms (device generator for the decay law; COO assembly for cfg 1)."""
    dt = np_dtype(c)
    if c["gen"] == "decay":
        W = G.decay_width(c["lam"], 1e-12)
        if c.get("symmetric"):
            F = H(dt, c["b"]); F.generate_decay(c["n"], c["lam"], W, 3, True, lo, hi); F.update_internal_info()
            return [F]
        out = []
        for seed in (1, 2):
            M = H(dt, c["b"]); M.generate_decay(c["n"], c["lam"], W, seed, False, lo, hi); M.update_internal_info()
            out.append(M)
        return out
    out = []
    for seed in (1, 2):
        r, cc, v = G.random_block_sparse_coo(c["n"], c["b"], c["fill"], seed, dt)
        M = H(dt, c["b"]); M.resize(c["n"], c["n"]); M.assign_from_vectors(r, cc, v); M.update_internal_info()
        out.append(M)
    return out


def make_step(H, c, ops):
    dt = np_dtype(c)
    if c["op"] == "spamm":
        def step():
            Cm = H(dt); nm, nr = H.spamm(ops[0], c["tA"], ops[1], c["tB"], Cm, c["tau"], True); return Cm, nm, nr
    elif c["op"] == "multiply":
        def step():
            Cm = H(dt); nm, nr = H.multiply(ops[0], c["tA"], ops[1], c["tB"], Cm); return Cm, nm, nr
    elif c["op"] == "symm_square_spamm":
        U = H(dt); ops[0].get_upper_triangle(U); U.update_internal_info(); ops.append(U)
        def step():
            Cm = H(dt); nm, nr = H.symm_square_spamm(U, Cm, c["tau"]); return Cm, nm, nr
    elif c["op"] == "symm_square":
        U = H(dt); ops[0].get_upper_triangle(U); U.update_internal_info(); ops.append(U)
        def step():
            Cm = H(dt); H.symm_square(U, Cm); return Cm, Cm.get_n_block_multiplications(), Cm.get_n_blocks()
    else:
        def step():
            Cm = H(dt); H.add(ops[0], ops[1], Cm); return Cm, 0, Cm.get_n_blocks()
    return step


def time_case(hb, H, torch, stream, c, ops, steps, warmup, keep_last=False):
    """W untimed + K timed calls of the case's operation, CUDA events on the engine's stream; results dropped at once,
    except the last step's (Cm, n_mults, n_blocks) when keep_last is set.  Returns (timings, last step's result or None)."""
    step = make_step(H, c, ops)
    for _ in range(warmup):
        r = step(); del r
    torch.cuda.synchronize()
    l0 = hb.kernel_launch_count()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    gemm_ms, task_ms = [], []
    last = None
    ev0.record(stream)
    for i in range(steps):
        Cm, nm, nr = step()
        st = hb.stage_times()
        gemm_ms.append(st["gemm_ms"]); task_ms.append(st["tasklist_ms"])
        if keep_last and i == steps - 1:
            last = (Cm, nm, nr)
        del Cm
    ev1.record(stream)
    torch.cuda.synchronize()
    launches = hb.kernel_launch_count() - l0
    ms = ev0.elapsed_time(ev1) / steps
    esz = 8 if c["dtype"] == "f64" else 4
    res = {"case": c["name"], "n": c["n"], "leaf": c["b"], "dtype": c["dtype"], "ms_per_call": ms, "gpu_launches": int(launches)}
    if c["op"] == "add":
        byts = 3.0 * nr * c["b"] ** 2 * esz
        peak, src = hbm_peak()
        res.update(c_tiles=int(nr), value=byts / (ms * 1e-3) / 1e9, unit="GB/s",
                   roofline={"bound": "hbm", "kernel": "k_add_tiles (+ key merge)", "achieved": byts / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": byts / (ms * 1e-3) / 1e9 / peak, "peak_source": src, "traffic": None,
                             "algorithmic": "read A tile + read B tile + write C tile = 3*b^2*%d B per C tile x %d tiles (union structure)" % (esz, nr)})
        return res, last
    flops = 2.0 * c["b"] ** 3 * nm
    g_ms = float(np.mean(gemm_ms))
    if c["dtype"] == "f64":
        peak, src = fp64_peak(); kname = "k_gemm_f64_tma<%d> (FP64 DMMA mma.sync leaf GEMM, TMA-staged)" % c["b"]
    else:
        p3, src = tf32_peak(); peak = p3 / 3.0
        src = "one third of the TF32 tensor peak (3 TF32 MMAs per fp32 product: hi*hi + hi*lo + lo*hi); " + src
        kname = "k_gemm_f32 leaf %d (tcgen05.mma kind::tf32 x3 split, TMEM accumulators, TMA-staged)" % c["b"]
    achieved = flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    res.update(products=int(nm), c_tiles=int(nr), candidates=int(st["n_candidates"]), value=flops / (ms * 1e-3) / 1e12, unit="TFLOP/s",
               stage_ms={"tasklist": float(np.mean(task_ms)), "gemm": g_ms}, gemm_kernel=int(st["gemm_kernel"]),
               roofline={"bound": "tensor", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "peak_source": src,
                         "algorithmic": "2*b^3 flops per leaf product x %d products per launch" % nm,
                         "kernel_ms": g_ms, "share_of_step": g_ms / ms if ms > 0 else None,
                         "traffic": traffic_from_profile(c)})
    return res, last


DUMP_TABLE_MAX = 1 << 19              # C tiles listed in the per-tile tables (3 float64 tables: 12 MiB at most)
DUMP_TILE_BYTES = 24 << 20            # whole C tiles kept in the sample


def _seeded_pick(n, k):
    """Sorted positions of a fixed, seeded sample of min(n, k) out of n (all of them when k >= n)."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def dump_outputs(out_dir, Cm, nm, nr):
    """Writes what a caller of the timed call receives -- the result matrix C and the two counts -- as .npy files:
      counts          [block multiplications, C tiles]  (float64)
      c_tiles_*       row, column and squared Frobenius norm (float64) of every C tile, in (row, col) order
                      (a fixed, seeded sample of DUMP_TABLE_MAX tiles when C has more)
      c_sample_*      a fixed, seeded sample of whole C tiles: coordinates and the b x b tiles (row-major, C's dtype)
    so that two builds can be compared output for output on the same seeded inputs."""
    os.makedirs(out_dir, exist_ok=True)
    bi, bj, _, t = Cm.export_leaves(norms=False)
    b = Cm.get_params().blocksize
    order = np.lexsort((bj, bi))
    rows = order[_seeded_pick(len(order), DUMP_TABLE_MAX)]
    tiles = order[_seeded_pick(len(order), DUMP_TILE_BYTES // (b * b * t.itemsize))]
    arrays = {"counts": np.array([nm, nr], np.float64),
              "c_tiles_row": bi[rows].astype(np.float64), "c_tiles_col": bj[rows].astype(np.float64),
              "c_tiles_frob_sq": np.einsum("ij,ij->i", t, t, dtype=np.float64)[rows],
              "c_sample_row": bi[tiles].astype(np.float64), "c_sample_col": bj[tiles].astype(np.float64),
              "c_sample_tiles": t[tiles].reshape(-1, b, b).transpose(0, 2, 1)}     # exported tiles are column-major
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def traffic_from_profile(c):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE leaf-GEMM launch of this workload from an `ncu --set full` capture
    (a static record: ncu cannot run inside the timed bench); null for workloads without a capture."""
    if not (c["dtype"] == "f64" and c["b"] == 64 and c["n"] == 65536 and c["op"] == "spamm" and c.get("lam") == 0.01):
        return None
    for nm in ("r02_gemm_f64_b64_traffic.json", "r01_gemm_f64_b64_traffic.json"):
        try:
            return json.load(open(os.path.join(PROFILES, nm)))["dram_bytes_per_launch"]
        except Exception:
            continue
    return None


def expected_results():
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "bench_expected.json")))
    except Exception:
        return {}


def expected_key(c):
    return "%s|%s|n=%d|b=%d|lam=%g|tau=%g|t=%d%d" % (c["op"], c["dtype"], c["n"], c["b"], c.get("lam", 0.0), c["tau"], c["tA"], c["tB"])


def run_check(c, ops, Cm, nm, n_samples, dist=None, torch=None):
    """Parity of the benchmarked product itself (outside the timed region; oracle/ is the checker only):
      * n_samples C tiles + 2 absent coordinates recomputed by the unmodified reference on the tile's own sub-problem
        (oracle/sampled_check.py): k-lists and leaf norms bit-exact, values within the stated tolerance;
      * the engine's executed-product checksum against the flat leaf-pair rule evaluated in numpy on the exported leaf norms;
      * ||C||_F^2 (and the checksum, summed over ranks) against the committed single-GPU values, so every world size is
        checked against the same answer."""
    from oracle import sampled_check as sc
    from hierarchical_block_sparse_lib_b200 import generators as G
    dt = np_dtype(c)
    tol = 1e-12 if c["dtype"] == "f64" else 1e-5
    W = G.decay_width(c["lam"], 1e-12)
    t0 = time.perf_counter()
    res = sc.sampled_check(Cm, ops[0], ops[1], c["n"], c["b"], c["lam"], W, (1, 2), True, c["tau"], dt, n_samples=n_samples)
    cs = Cm.task_checksum()
    fro = float(Cm.get_frob_squared())
    abi, abj, an, _ = ops[0].export_leaves(tiles=False)
    bbi, bbj, bn, _ = ops[1].export_leaves(tiles=False)
    world = dist.get_world_size() if dist is not None else 1
    if world > 1:      # gather the (small) norm tables: every rank evaluates the flat rule for ITS block rows against all of B
        parts = [None] * world
        dist.all_gather_object(parts, (bbi, bbj, bn))
        bbi = np.concatenate([p[0] for p in parts]); bbj = np.concatenate([p[1] for p in parts]); bn = np.concatenate([p[2] for p in parts])
    want_cs, want_cnt = sc.flat_rule_checksum(abi, abj, an, bbi, bbj, bn, True, c["tau"], dt)
    ok_flat = (want_cs == cs) and (want_cnt == nm)
    out = {"checker": res["checker"], "sampled_c_tiles": res["sampled_c_tiles"], "absent_tiles_confirmed": res["absent_tiles_confirmed"],
           "task_set_equal": bool(res["task_set_equal"] and ok_flat), "sampled_k_lists_equal": bool(res["task_set_equal"]),
           "flat_rule_checksum_equal": bool(ok_flat), "leaf_norms_bit_equal": bool(res["leaf_norms_bit_equal"]),
           "leaf_norms_compared": res["leaf_norms_compared"], "rel_err": res["rel_err_max"], "tolerance": tol,
           "task_checksum": cs, "c_frob_sq": fro}
    if world > 1:
        objs = [None] * world
        dist.all_gather_object(objs, out)
        out = dict(objs[0])
        for k in ("sampled_c_tiles", "absent_tiles_confirmed", "leaf_norms_compared"):
            out[k] = int(sum(o[k] for o in objs))
        for k in ("task_set_equal", "sampled_k_lists_equal", "flat_rule_checksum_equal", "leaf_norms_bit_equal"):
            out[k] = bool(all(o[k] for o in objs))
        out["rel_err"] = float(max(o["rel_err"] for o in objs))
        out["task_checksum"] = int(sum(o["task_checksum"] for o in objs) % (1 << 64))
        out["c_frob_sq"] = float(sum(o["c_frob_sq"] for o in objs))
    exp = expected_results().get(expected_key(c))
    if exp:
        out["task_checksum_equals_1gpu"] = bool(int(exp["task_checksum"]) == out["task_checksum"])
        out["c_frob_sq_rel_diff_vs_1gpu"] = abs(out["c_frob_sq"] - exp["c_frob_sq"]) / exp["c_frob_sq"]
    out["task_checksum"] = "0x%016x" % out["task_checksum"]
    out["pass"] = bool(out["task_set_equal"] and out["leaf_norms_bit_equal"] and out["rel_err"] <= tol
                       and out.get("task_checksum_equals_1gpu", True) and out.get("c_frob_sq_rel_diff_vs_1gpu", 0.0) <= 1e-12)
    out["seconds"] = time.perf_counter() - t0
    return out


def native_arm(args):
    import torch
    import hierarchical_block_sparse_lib_b200 as hb
    from hierarchical_block_sparse_lib_b200 import generators as G
    H = hb.HierarchicalBlockSparseMatrix

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cases = config_cases(args.config, args.n, args.leaf, args.lam)
    if world > 1:
        from hierarchical_block_sparse_lib_b200 import sharded
        return sharded.bench_main(args, cases[0], sys.modules[__name__])

    torch.cuda.set_device(local_rank)
    hb.init(local_rank)
    stream = torch.cuda.ExternalStream(_capi.lib().hbsm_stream())
    sampler = ClockSampler(local_rank); sampler.start()
    results = []
    primary_ops = None
    last_key = None
    ops = None
    for i, c in enumerate(cases):
        key = (c["gen"], c["n"], c["b"], c.get("lam"), c.get("fill"), c["dtype"], bool(c.get("symmetric")))
        if key != last_key:      # cases of one configuration that share operands reuse them
            ops = None
            ops = build_operands(H, G, c)
            last_key = key
        res, last = time_case(hb, H, torch, stream, c, ops, args.steps, args.warmup, keep_last=i == 0 and bool(args.dump_outputs))
        results.append(res)
        if i == 0:
            primary_ops = ops
        if last is not None:       # the primary case's last timed step, written before its C is dropped
            dump_outputs(args.dump_outputs, *last)
            del last
    clocks = sampler.stop()
    c = cases[0]; r = results[0]
    ops = primary_ops if len(cases) == 1 or last_key == (c["gen"], c["n"], c["b"], c.get("lam"), c.get("fill"), c["dtype"], bool(c.get("symmetric"))) \
        else build_operands(H, G, c)

    check = None
    if not args.no_check and c["op"] == "spamm" and c["gen"] == "decay" and c["tA"] == 0 and c["tB"] == 0:
        try:
            Cm, nm, nr = make_step(H, c, ops)()
            check = run_check(c, ops, Cm, nm, args.check_samples)
            del Cm
        except Exception as ex:  # noqa: BLE001 -- the checker is optional equipment; say why it did not run
            check = {"pass": None, "error": repr(ex)}

    # ---- e2e: host buffers through the C ABI (headline-shaped cases: spamm NN fp64) ----
    e2e = None
    if not args.no_e2e and c["op"] == "spamm" and c["dtype"] == "f64" and c["tA"] == 0 and c["tB"] == 0:
        e2e = measure_e2e(hb, H, ops[0], ops[1], c, args.steps, torch)

    # ---- CPU baseline beside it (bounded sample) ----
    cpu = None
    if not args.no_cpu_baseline:
        try:
            rate, cms, info = run_reference_cpu(c, 1, 1)
            cpu = {"value": rate, "unit": r["unit"], "cores": info["cores"], "kind": info["kind"], "sample": info["sample"],
                   "ms_per_call_on_sample": cms}
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": r["unit"], "cores": host_threads(), "kind": "unavailable", "sample": repr(ex)}

    metric, unit = metric_of(c)
    line = {"metric": metric, "value": r["value"], "unit": unit, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_call"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": c["dtype"], "data": "synthetic", "config": case_config(c, 1, args.config),
            "products_per_multiply": r.get("products"), "c_tiles": r.get("c_tiles"), "candidates": r.get("candidates"),
            "stage_ms": r.get("stage_ms"), "roofline": r["roofline"], "check": check, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": r["gpu_launches"], "clocks": clocks}
    if len(results) > 1:
        line["cases"] = results
    print(json.dumps(line), flush=True)


def measure_e2e(hb, H, A, B, w, steps, torch):
    """Same multiply through the C ABI with HOST buffers: pinned H2D of the A and B tiles, norm refresh, SpAMM, D2H
    of every C tile."""
    b, n, tau = w["b"], w["n"], w["tau"]

    def pinned_leaves(Mx):
        bi, bj, _, t = Mx.export_leaves(norms=False)
        pt = torch.empty(t.shape, dtype=torch.float64, pin_memory=True)
        pt.numpy()[...] = t
        return bi.astype(np.int32), bj.astype(np.int32), pt

    abi, abj, at = pinned_leaves(A)
    bbi, bbj, bt = pinned_leaves(B)
    h2d = at.numel() * 8 + bt.numel() * 8 + 4 * (len(abi) + len(abj) + len(bbi) + len(bbj))
    out = None
    times = []
    times_pipe = []
    d2h = 0
    nm = 0
    n_slabs = int(os.environ.get("HBSM_E2E_SLABS", "0"))
    import ctypes as Ct
    # schedule: two-call warm-up (learns the size of C), `steps` two-call passes, two pipelined warm-ups, `steps` pipelined
    # passes -- not interleaved, so that the stream-ordered memory pool is in steady state for both
    schedule = [False] * (steps + 1) + [True] * (steps + 2)
    untimed = {0, steps + 1, steps + 2}
    for i, pipelined in enumerate(schedule):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        A2 = H(np.float64, b); A2.resize(n, n)
        B2 = H(np.float64, b); B2.resize(n, n)
        C = H(np.float64)
        m = Ct.c_size_t(0)
        if pipelined:
            # ONE call: uploads, norm refresh, task lists, leaf GEMMs and downloads overlapped slab by slab
            nm, nr, cbi, cbj = H.product_from_host(A2, abi, abj, at.numpy(), False, B2, bbi, bbj, bt.numpy(), False, C, True, tau,
                                                   out.numpy(), n_slabs)
        else:
            A2.assign_tiles(abi, abj, at.numpy()); A2.update_internal_info()
            B2.assign_tiles(bbi, bbj, bt.numpy()); B2.update_internal_info()
            if out is None:      # warm-up pass: learn the size of C, allocate the pinned result buffer once
                nm, nr = H.spamm(A2, False, B2, False, C, tau, True)
                out = torch.empty((nr + nr // 8, b * b), dtype=torch.float64, pin_memory=True)
                _capi.check(_capi.lib().hbsm_export_leaves(C._h, nr, None, None, None, Ct.c_void_p(out.data_ptr()), Ct.byref(m)))
            else:                # SpAMM with the C tiles streaming to pinned host memory while the remaining leaf GEMMs run
                cnm = Ct.c_size_t(0); cnr = Ct.c_size_t(0)
                _capi.check(_capi.lib().hbsm_product_to_host(A2._h, 0, B2._h, 0, C._h, 1, float(tau), 1, Ct.c_void_p(out.data_ptr()),
                                                              out.shape[0], Ct.byref(cnm), Ct.byref(cnr)))
                nm, nr = cnm.value, cnr.value
            cbi = np.zeros(nr, np.int64); cbj = np.zeros(nr, np.int64)
            _capi.check(_capi.lib().hbsm_export_leaves(C._h, nr, cbi.ctypes.data_as(Ct.c_void_p), cbj.ctypes.data_as(Ct.c_void_p),
                                                        None, None, Ct.byref(m)))
        dt = time.perf_counter() - t0
        d2h = nr * b * b * 8 + 16 * nr
        del A2, B2, C
        if i not in untimed:
            (times_pipe if pipelined else times).append(dt)
    ms_two = 1e3 * float(np.mean(times))
    ms = 1e3 * float(np.mean(times_pipe))
    return {"value": 2.0 * b ** 3 * nm / (ms * 1e-3) / 1e12, "unit": "TFLOP/s", "ms_per_step": ms,
            "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "path": "hbsm_product_from_host: A, B tiles from pinned host memory, norm refresh, SpAMM task lists, leaf GEMMs and "
                    "the D2H of every C tile (+ coordinates) pipelined over block-row slabs of C on three streams",
            "ms_per_step_unpipelined": ms_two,
            "unpipelined_path": "hbsm_assign_tiles(A,B) + hbsm_update_norms + hbsm_product_to_host + hbsm_export_leaves(C keys)"}


def main():
    # stdout carries exactly ONE line (the JSON): everything else that writes to fd 1 (e.g. NCCL's version banner) is sent
    # to stderr; print() below writes through the saved descriptor
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="headline", choices=["headline", "1", "2", "3", "4", "5"],
                    help="headline = the BASELINE.json metric's workload (default); 1..5 = BASELINE.json configs[0..4]")
    ap.add_argument("--no-check", action="store_true", help="skip the parity check of the benchmarked product (runs outside the timed region)")
    ap.add_argument("--check-samples", type=int, default=16, help="C tiles recomputed by the reference in the check")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-to-host measurement (used for the ncu launch list of the timed region)")
    ap.add_argument("--n", "--size", dest="n", type=int, default=None, help="override N (the judged run uses the default); use --size under torchrun")
    ap.add_argument("--lam", type=float, default=None)
    ap.add_argument("--leaf", type=int, default=None, help="override the leaf size")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step (first case of the config) to DIR/<name>.npy (one GPU only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the native product of a single-GPU run")
    if args.impl == "reference":
        reference_arm(args)
    else:
        native_arm(args)


if __name__ == "__main__":
    main()
