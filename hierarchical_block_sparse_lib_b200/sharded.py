"""Multi-GPU multiply / SpAMM: one process per GPU, C sharded by block rows (SURVEY 8e).

The product path lives in the library: csrc/sharded.cu behind the C ABI (hbsm_comm_init / hbsm_publish /
hbsm_sharded_product / hbsm_sharded_row_weights / hbsm_shard_rows_balanced; NCCL is loaded by libhbsm_b200.so itself).
This module is
  * the thin ctypes caller of those entry points (comm_init, publish, sharded_product, row_weights, ...), which only uses
    torch.distributed to hand the 128-byte NCCL id to the peers;
  * the protocol MODEL as device-agnostic torch ops (request_thresholds, publish_table, exchange_b_allgather, and the
    self-contained three-round exchange_b), which tests/test_sharded_cpu.py runs over `gloo` at world 2 and 4 against the
    oracle's single-process executed-product set;
  * bench.py's N > 1 arm (bench_main).

Rank r owns a contiguous slab of block rows (equal slabs = the top-level quadtree block rows for world in {2,4,8}, or
boundaries balanced on the per-row product counts).  It holds the tiles of op(A) whose C-row index ci lies in its slab and the
tiles of op(B) whose contraction index k lies in its slab.  One product is

  1. request   every rank computes, per k, the largest leaf norm^2 among its op(A) tiles (ci,k); the thresholds are all-gathered
  2. select    requester and owner evaluate the same predicate on the published (key, norm^2) table of op(B):
               fl(max_na * nb) > fl(tau*tau) (monotone rounding => exactly the tiles that at least one executed product of the
               requester touches; exact multiply: every tile of a requested row) -- no masks, no counts travel
  3. exchange  the selected op(B) tiles, straight into the halo tail behind the requester's own tiles
  4. multiply  task list + leaf GEMMs on (A_r, own + halo B tiles) -> C_r; the GEMMs that need no halo tile overlap step 3

There is NO reduction: each rank owns whole block rows of C.  The executed-product set is the disjoint union of
the per-rank sets and is bit-identical to the single-GPU one because the predicate is per leaf pair.
"""
import ctypes as C
import os
import time

import numpy as np
import torch
import torch.distributed as dist

TRACE = int(os.environ.get("HBSM_SHARD_TRACE", "0"))    # 1 = synchronising phase timer, 2 = host timestamps only (no syncs)


class _Trace:
    """Synchronising phase timer, only active with HBSM_SHARD_TRACE=1 (diagnosis; perturbs the timings it reports)."""

    def __init__(self, sink):
        self.sink = sink if TRACE else None
        self.t = time.perf_counter()

    def mark(self, name):
        if self.sink is None:
            return
        if TRACE == 1 and torch.cuda.is_available():
            torch.cuda.synchronize()
        now = time.perf_counter()
        self.sink[name] = self.sink.get(name, 0.0) + (now - self.t)
        self.t = now

# ---------------------------------------------------------------------------------------------------
# Morton helpers on int64 tensors (digit = 2*colbit + rowbit, H:52-56; same bit tricks as csrc/common.cuh)
# ---------------------------------------------------------------------------------------------------
_M = [0x5555555555555555, 0x3333333333333333, 0x0F0F0F0F0F0F0F0F, 0x00FF00FF00FF00FF, 0x0000FFFF0000FFFF,
      0x00000000FFFFFFFF]


def _compact(v):
    v = v & _M[0]
    for s, m in zip((1, 2, 4, 8, 16), _M[1:]):
        v = (v | (v >> s)) & m
    return v


def _spread(v):
    v = v & _M[5]
    for s, m in zip((16, 8, 4, 2, 1), reversed(_M[:5])):
        v = (v | (v << s)) & m
    return v


def morton_decode(keys):
    """int64 keys -> (block row, block col)."""
    return _compact(keys), _compact(keys >> 1)


def morton_encode(bi, bj):
    return _spread(bi) | (_spread(bj) << 1)


def slab_bounds(grid_side, world, rank):
    """Block rows [lo, hi) owned by `rank`: top-level quadtree block rows for world in {2,4,8}."""
    if grid_side % world != 0:
        raise ValueError("block grid side %d is not divisible by the world size %d" % (grid_side, world))
    rows = grid_side // world
    return rank * rows, (rank + 1) * rows


def owner_of(line, grid_side, world):
    return line // (grid_side // world)


# ---------------------------------------------------------------------------------------------------
# steps 1-3: plan + exchange (device-agnostic)
# ---------------------------------------------------------------------------------------------------
def request_thresholds(a_keys, a_norms, tA, grid_side):
    """Per contraction index k: max leaf norm^2 over this rank's op(A) tiles (., k); -1 where no tile has that k."""
    ar, ac = morton_decode(a_keys)
    k = ar if tA else ac
    thr = torch.full((grid_side,), -1.0, dtype=a_norms.dtype, device=a_norms.device)
    if k.numel():
        thr.scatter_reduce_(0, k, a_norms, reduce="amax", include_self=True)
    return thr


def select_for_peers(b_keys, b_norms, tB, thr_from_peers, lo, spamm, tau):
    """thr_from_peers[q, k - lo] = request of rank q for my row k (-1 = none).  Returns (send_index, counts[q]):
    indices into my op(B) tile list, grouped by destination rank, ascending Morton key inside a group."""
    br, bc = morton_decode(b_keys)
    k = (bc if tB else br) - lo
    world = thr_from_peers.shape[0]
    if k.numel() == 0:
        return torch.zeros(0, dtype=torch.int64, device=b_keys.device), [0] * world
    t = thr_from_peers[:, k]                          # [world, L_b]
    keep = t >= 0
    if spamm:
        tau2 = torch.tensor(tau, dtype=b_norms.dtype, device=b_norms.device)
        tau2 = tau2 * tau2                            # fl(tau*tau) in Treal, H:2008
        keep &= (t * b_norms.unsqueeze(0)) > tau2     # fl(max_na * nb) > fl(tau^2): same rounding as the leaf-pair test
    nz = torch.nonzero(keep, as_tuple=False)          # row-major: grouped by peer, ascending tile index inside
    counts = torch.bincount(nz[:, 0], minlength=world).tolist()
    return nz[:, 1].contiguous(), [int(c) for c in counts]


def exchange_b(a_keys, a_norms, tA, b_keys, b_norms, b_tiles, tB, grid_side, spamm, tau, group=None, timers=None,
               recv_alloc=None):
    """Runs steps 1-3.  Returns (keys, norms, tiles) of the REMOTE op(B) tiles this rank's products can touch (the
    rank's own tiles never move).  `recv_alloc(n)` may supply the three receive buffers (the engine's halo tail, so
    NCCL writes in place); by default they are fresh tensors."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    lo, hi = slab_bounds(grid_side, world, rank)
    rows = hi - lo
    t0 = time.perf_counter()
    tr = _Trace(timers.setdefault("trace", {}) if timers is not None else None)
    thr = request_thresholds(a_keys, a_norms, tA, grid_side)              # [g] -> slice p goes to rank p
    tr.mark("request")
    thr_in = torch.empty_like(thr)
    dist.all_to_all_single(thr_in, thr, group=group)                      # equal splits of `rows`
    tr.mark("a2a_thr")
    thr_in = thr_in.view(world, rows).clone()
    thr_in[rank] = -1.0                                                   # own tiles are already here
    send_idx, counts = select_for_peers(b_keys, b_norms, tB, thr_in, lo, spamm, tau)
    tr.mark("select")
    cnt_out = torch.tensor(counts, dtype=torch.int64, device=b_keys.device)
    cnt_in = torch.empty_like(cnt_out)
    dist.all_to_all_single(cnt_in, cnt_out, group=group)
    recv_counts = [int(x) for x in cnt_in.tolist()]                       # the one host sync of the plan
    n_in = sum(recv_counts)
    tr.mark("a2a_counts")
    t1 = time.perf_counter()
    keys_out = b_keys.index_select(0, send_idx)
    norms_out = b_norms.index_select(0, send_idx)
    tiles_out = b_tiles.index_select(0, send_idx)
    tr.mark("pack")
    if recv_alloc is not None:
        keys_in, norms_in, tiles_in = recv_alloc(n_in)
    else:
        keys_in = torch.empty((n_in,), dtype=b_keys.dtype, device=b_keys.device)
        norms_in = torch.empty((n_in,), dtype=b_norms.dtype, device=b_keys.device)
        tiles_in = torch.empty((n_in, b_tiles.shape[1]), dtype=b_tiles.dtype, device=b_keys.device)
    dist.all_to_all_single(keys_in, keys_out, recv_counts, counts, group=group)
    dist.all_to_all_single(norms_in, norms_out, recv_counts, counts, group=group)
    dist.all_to_all_single(tiles_in, tiles_out, recv_counts, counts, group=group)
    tr.mark("a2a_tiles")
    if timers is not None:
        timers["plan_s"] = t1 - t0
        timers["sent_tiles"] = sum(counts)
        timers["recv_tiles"] = n_in
    return keys_in, norms_in, tiles_in


# ---------------------------------------------------------------------------------------------------
# published block tables + the all-gather protocol (what csrc/sharded.cu runs), as device-agnostic torch ops
# ---------------------------------------------------------------------------------------------------
class PublishedTable:
    """The (Morton key, leaf norm^2) table of a row-sharded matrix, gathered once on every rank -- the distributed part
    of update_internal_info() (H:3905): like the cached norms it is valid until the matrix changes (csrc/sharded.cu
    publish())."""

    def __init__(self, keys_all, norms_all, counts):
        self.keys_all = keys_all                # [sum L_q] int64, rank-major, each rank's part in its local tile order
        self.norms_all = norms_all              # [sum L_q]
        self.counts = [int(c) for c in counts]  # L_q
        self.offsets = [0]
        for c in self.counts:
            self.offsets.append(self.offsets[-1] + c)

    def k_of(self, tB):
        """Contraction index k of every published tile of op(B)."""
        br, bc = morton_decode(self.keys_all)
        return (bc if tB else br).contiguous()


def publish_table(b_keys, b_norms, group=None):
    """all_gather of this rank's (keys, norms) -- variable lengths, padded to the longest."""
    world = dist.get_world_size(group)
    n = torch.tensor([b_keys.numel()], dtype=torch.int64, device=b_keys.device)
    ns = [torch.empty_like(n) for _ in range(world)]
    dist.all_gather(ns, n, group=group)
    counts = [int(x.item()) for x in ns]
    m = max(max(counts), 1)
    kp = torch.zeros((m,), dtype=b_keys.dtype, device=b_keys.device); kp[:b_keys.numel()] = b_keys
    np_ = torch.zeros((m,), dtype=b_norms.dtype, device=b_norms.device); np_[:b_norms.numel()] = b_norms
    kall = [torch.empty_like(kp) for _ in range(world)]; nall = [torch.empty_like(np_) for _ in range(world)]
    dist.all_gather(kall, kp, group=group)
    dist.all_gather(nall, np_, group=group)
    keys_all = torch.cat([kall[q][:counts[q]] for q in range(world)])
    norms_all = torch.cat([nall[q][:counts[q]] for q in range(world)])
    return PublishedTable(keys_all, norms_all, counts)


def exchange_b_allgather(thr, table, b_tiles, tB, spamm, tau, group=None, timers=None):
    """The protocol of csrc/sharded.cu sharded_product(): all-gather the request thresholds; requester AND owner then
    evaluate the same predicate  thr_q[k] >= 0 and (not spamm or fl(thr_q[k] * nsq) > fl(tau*tau))  on the same published
    numbers, so both know the transfer lists without another message; one all-to-all moves the tiles.
    Returns (keys, norms, tiles) of the remote tiles this rank's products touch (peer-major, owner's tile order)."""
    world = dist.get_world_size(group); rank = dist.get_rank(group)
    thr_all = [torch.empty_like(thr) for _ in range(world)]
    dist.all_gather(thr_all, thr, group=group)
    thr_all = torch.stack(thr_all)                                   # [world, g]
    k_all = table.k_of(bool(tB))
    lo_r, hi_r = table.offsets[rank], table.offsets[rank + 1]
    tau2 = torch.tensor(tau, dtype=table.norms_all.dtype)
    tau2 = tau2 * tau2

    def wanted_by(q, sl):
        t = thr_all[q][k_all[sl]]
        keep = t >= 0
        if spamm:
            keep &= (t * table.norms_all[sl]) > tau2
        return keep

    need = wanted_by(rank, slice(0, table.offsets[-1])).clone()
    need[lo_r:hi_r] = False                                           # own tiles are already here
    recv_idx = torch.nonzero(need).flatten()
    recv_counts = [int(need[table.offsets[q]:table.offsets[q + 1]].sum()) for q in range(world)]
    send_lists = [torch.nonzero(wanted_by(q, slice(lo_r, hi_r))).flatten() if q != rank else torch.zeros(0, dtype=torch.int64)
                  for q in range(world)]
    send_counts = [int(x.numel()) for x in send_lists]
    tiles_out = b_tiles.index_select(0, torch.cat(send_lists))
    tiles_in = torch.empty((sum(recv_counts), b_tiles.shape[1]), dtype=b_tiles.dtype)
    dist.all_to_all_single(tiles_in, tiles_out, recv_counts, send_counts, group=group)
    if timers is not None:
        timers["sent_tiles"] = sum(send_counts)
        timers["recv_tiles"] = sum(recv_counts)
    return table.keys_all[recv_idx], table.norms_all[recv_idx], tiles_in


def balanced_bounds(row_weights, world):
    """Slab boundaries on the prefix sums of per-block-row weights (same rule as hbsm_shard_rows_balanced): boundary r is
    the row at which the running weight is nearest to r/world of the total."""
    w = np.asarray(row_weights, np.float64)
    g = len(w)
    total = float(w.sum())
    bounds = [0]
    acc = 0.0
    row = 0
    for r in range(1, world):
        want = total * r / world
        while row < g and acc + w[row] <= want:
            acc += w[row]; row += 1
        if row < g and want - acc > acc + w[row] - want:
            acc += w[row]; row += 1
        bounds.append(max(row, bounds[-1]))
    bounds.append(g)
    return bounds


# ---------------------------------------------------------------------------------------------------
# engine glue (GPU only): thin callers of the C ABI (include/hbsm_b200.h "multi-GPU"); NCCL lives inside the library
# ---------------------------------------------------------------------------------------------------
class ShardStats(C.Structure):
    _fields_ = [("plan_ms", C.c_double), ("exchange_ms", C.c_double), ("publish_ms", C.c_double),
                ("sent_tiles", C.c_uint64), ("recv_tiles", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def comm_init(group=None):
    """Creates the library's own NCCL communicator over the ranks of `group` (default: the world): rank 0 makes the
    unique id, torch.distributed only carries its 128 bytes to the peers (any transport would do)."""
    from . import _capi
    L = _capi.lib()
    rank = dist.get_rank(group); world = dist.get_world_size(group)
    buf = (C.c_ubyte * 128)()
    if rank == 0:
        _capi.check(L.hbsm_comm_unique_id(buf))
    box = [bytes(buf)]
    dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    ident = (C.c_ubyte * 128).from_buffer_copy(box[0])
    _capi.check(L.hbsm_comm_init(ident, rank, world))


def comm_finalize():
    from . import _capi
    _capi.check(_capi.lib().hbsm_comm_finalize())


def comm_info():
    from . import _capi
    r = C.c_int(0); w = C.c_int(1); v = C.c_int(0)
    _capi.check(_capi.lib().hbsm_comm_info(C.byref(r), C.byref(w), C.byref(v)))
    return r.value, w.value, v.value


def allreduce(vals, take_max=False):
    """Sum (or max) of a few host scalars over the ranks through the library's communicator."""
    from . import _capi
    a = (C.c_double * len(vals))(*[float(v) for v in vals])
    _capi.check(_capi.lib().hbsm_comm_allreduce_f64(a, len(vals), int(bool(take_max))))
    return [float(x) for x in a]


def shard_stats():
    from . import _capi
    st = ShardStats()
    _capi.check(_capi.lib().hbsm_shard_stats_last(C.byref(st)))
    return st.as_dict()


def publish(B_loc):
    """Distributed half of update_internal_info() for a matrix that will be the right operand of sharded products
    (hbsm_publish): call after the norms are refreshed; valid until B_loc changes.  Collective."""
    from . import _capi
    _capi.check(_capi.lib().hbsm_publish(B_loc._h))


def row_weights(A_loc, tA, B_loc, tB, spamm=False, tau=0.0, upper_only=False):
    """Leaf products per C block row of op(A)*op(B) over ALL ranks (count-only join of each rank's rows against the
    published table of op(B), summed over the ranks): the weights hbsm_shard_rows_balanced wants.  Collective."""
    from . import _capi
    g = 1 << max(A_loc.expected_depth(), B_loc.expected_depth())
    w = np.zeros(g, np.uint64)
    _capi.check(_capi.lib().hbsm_sharded_row_weights(A_loc._h, int(bool(tA)), B_loc._h, int(bool(tB)), int(bool(spamm)), float(tau),
                                                      int(bool(upper_only)), g, w.ctypes.data_as(C.c_void_p)))
    return w


def sharded_product(A_loc, tA, B_loc, tB, spamm=False, tau=0.0, upper_only=False):
    """C_r = op(A)_r * op(B): A_loc / B_loc are this rank's engine matrices (full logical dims, only the slab's tiles; norms
    refreshed, publish(B_loc) called).  Returns (C_loc, n_mults_local, n_blocks_local).  Collective (hbsm_sharded_product)."""
    from . import _capi
    from .matrix import HierarchicalBlockSparseMatrix as H
    Cm = H(A_loc.dtype)
    nm = C.c_size_t(0); nb = C.c_size_t(0)
    _capi.check(_capi.lib().hbsm_sharded_product(A_loc._h, int(bool(tA)), B_loc._h, int(bool(tB)), Cm._h, int(bool(spamm)), float(tau),
                                                  int(bool(upper_only)), C.byref(nm), C.byref(nb)))
    return Cm, nm.value, nb.value


def sharded_symm_square_spamm(F_loc, tau):
    """BASELINE config 3 across GPUs: this rank's block rows of triu(spamm(F, F, tau)) for a symmetric F held in FULL storage
    and sharded by block rows like any other operand (norms refreshed, publish(F_loc) called).  tau = None: exact symmetric
    square.  Only C tiles with ci <= cj are planned, the diagonal tiles are masked: on one GPU this is symm_square_spamm of
    F's upper triangle (H:3563 with the prune of H:3931).  The triangular load is balanced by the slab boundaries
    (row_weights(..., upper_only=True) + balanced_bounds), not by pairing slabs."""
    return sharded_product(F_loc, False, F_loc, False, tau is not None, 0.0 if tau is None else tau, upper_only=True)


def bind_near_gpu(local_rank, local_world=1):
    """Pin this rank's host threads to its own share of the CPUs next to its GPU (sysfs local_cpulist of the GPU's PCI
    function, split evenly among the ranks of the box) BEFORE pinned host buffers, NCCL's proxy threads and the engine's
    streams exist: first touch then places pinned memory on the GPU's NUMA node, and the ranks' launch threads stop
    migrating over each other's cores (the step of a sharded product is ~50 short launches and four host reads: host jitter
    on ONE rank delays every rank at the next all-gather).  Returns the cpu list used or None."""
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-"); cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        use = sorted(cpus & os.sched_getaffinity(0))
        if local_world > 1 and len(use) >= 2 * local_world:
            per = len(use) // local_world
            use = use[local_rank * per:(local_rank + 1) * per]
        if use:
            os.sched_setaffinity(0, set(use))
            return "%d-%d" % (use[0], use[-1]) if use == list(range(use[0], use[-1] + 1)) else ",".join(map(str, use))
    except Exception:
        pass
    return None


# ---------------------------------------------------------------------------------------------------
# bench.py --gpus N (N > 1): strong scaling of the BASELINE workload, one rank per GPU under torchrun
# ---------------------------------------------------------------------------------------------------
def bench_main(args, w, bm):
    """bm = the bench.py module (config text, peaks, clock sampler, parity check)."""
    import json
    import hierarchical_block_sparse_lib_b200 as hb
    from . import _capi
    from . import generators as G
    H = hb.HierarchicalBlockSparseMatrix
    if w["op"] != "spamm" or w["dtype"] != "f64" or w["tA"] or w["tB"]:
        raise SystemExit("bench.py --gpus N>1 runs the fp64 SpAMM NN cases (headline, --config 2, --config 4)")
    world = int(os.environ["WORLD_SIZE"]); rank = int(os.environ["RANK"]); local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    # CPUs next to the GPU; HBSM_BIND_CORES=split additionally gives every rank its own share of them (untested at scale:
    # at 2 GPUs it changed nothing, 17.73 vs 17.70 ms)
    cpulist = bind_near_gpu(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)) if os.environ.get("HBSM_BIND_CORES") == "split" else 1)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    hb.init(local_rank)
    comm_init()
    n, b, lam, tau = w["n"], w["b"], w["lam"], w["tau"]
    W = G.decay_width(lam, 1e-12)
    g = n // b
    ext = torch.cuda.ExternalStream(int(_capi.lib().hbsm_stream()))

    def build(lo, hi):
        A = H(np.float64, b); A.generate_decay(n, lam, W, 1, False, lo, hi); A.update_internal_info()
        B = H(np.float64, b); B.generate_decay(n, lam, W, 2, False, lo, hi); B.update_internal_info()
        publish(B)     # the distributed half of update_internal_info(): outside the timed region like the norm refresh itself
        return A, B

    # slabs: equal block rows first; then boundaries on the prefix sums of the per-row product counts (the band is clipped at
    # the matrix edges, so equal slabs leave the edge ranks lighter), and the operands are re-made on the balanced slabs
    lo, hi = slab_bounds(g, world, rank)
    A, B = build(lo, hi)
    bounds = [int(g * r // world) for r in range(world + 1)]
    if os.environ.get("HBSM_SHARD_BALANCE", "1") == "1":
        wts = row_weights(A, False, B, False, True, tau)
        bounds = balanced_bounds(wts, world)
        if (bounds[rank], bounds[rank + 1]) != (lo, hi):
            del A, B
            lo, hi = bounds[rank], bounds[rank + 1]
            A, B = build(lo, hi)
    publish_ms = shard_stats()["publish_ms"]

    def step():
        Cm, nm, nb = sharded_product(A, False, B, False, True, tau)
        return Cm, nm, nb, hb.stage_times(), shard_stats()

    for _ in range(args.warmup):
        Cm, nm, nb, st, ss = step()
        del Cm
    sampler = bm.ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    l0 = hb.kernel_launch_count()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    gemm_ms, task_ms, plan_ms, xchg_ms, host_ms = [], [], [], [], []
    ev0.record(ext)
    for _ in range(args.steps):
        t0 = time.perf_counter()
        Cm, nm, nb, st, ss = step()
        host_ms.append(1e3 * (time.perf_counter() - t0))
        gemm_ms.append(st["gemm_ms"]); task_ms.append(st["tasklist_ms"]); plan_ms.append(ss["plan_ms"]); xchg_ms.append(ss["exchange_ms"])
        del Cm
    ev1.record(ext)
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    launches = hb.kernel_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    ms_local = ev0.elapsed_time(ev1) / args.steps
    mine = {"rank": rank, "rows": [lo, hi], "step_ms": ms_local, "host_ms": float(np.mean(host_ms)), "plan_ms": float(np.mean(plan_ms)),
            "exchange_ms": float(np.mean(xchg_ms)), "tasklist_ms": float(np.mean(task_ms)), "gemm_ms": float(np.mean(gemm_ms)),
            "index_ms": float(st["index_ms"]), "products": int(nm), "c_tiles": int(nb), "recv_tiles": int(ss["recv_tiles"]),
            "sent_tiles": int(ss["sent_tiles"]), "launches_per_step": launches / args.steps}
    per_rank = [None] * world
    dist.all_gather_object(per_rank, mine)
    ms = max(r["step_ms"] for r in per_rank)
    P = sum(r["products"] for r in per_rank)
    flops = 2.0 * b ** 3 * P

    check = None
    if not args.no_check:
        try:
            Cm, nm_c, nb_c = sharded_product(A, False, B, False, True, tau)
            check = bm.run_check(w, [A, B], Cm, nm_c, max(2, -(-args.check_samples // world)), dist, torch)
            del Cm
        except Exception as ex:  # noqa: BLE001
            check = {"pass": None, "error": repr(ex)}
            objs = [None] * world
            dist.all_gather_object(objs, check)

    e2e = None if args.no_e2e else _e2e_sharded(hb, H, A, B, w, args.steps, local_rank)

    if rank == 0:
        peak, peak_src = bm.fp64_peak()
        g_ms = float(np.mean(gemm_ms))
        g_max = max(r["gemm_ms"] for r in per_rank); g_mean = float(np.mean([r["gemm_ms"] for r in per_rank]))
        achieved = 2.0 * b ** 3 * nm / (g_ms * 1e-3) / 1e12
        slow = max(per_rank, key=lambda r: r["step_ms"])
        resid = {"imbalance_ms": g_max - g_mean, "plan_ms": slow["plan_ms"], "tasklist_ms": slow["tasklist_ms"],
                 "other_ms": ms - slow["gemm_ms"] - slow["plan_ms"] - slow["tasklist_ms"]}
        cfg = bm.case_config(w, world, args.config)
        cfg["slabs"] = {"bounds": bounds, "rule": "prefix sums of per-block-row leaf-product counts (hbsm_sharded_row_weights + "
                                                  "hbsm_shard_rows_balanced)" if os.environ.get("HBSM_SHARD_BALANCE", "1") == "1" else "equal block rows"}
        line = {"metric": "spamm_fp64_leaf_tflops", "value": flops / (ms * 1e-3) / 1e12, "unit": "TFLOP/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
                "products_per_multiply": P, "c_tiles": sum(r["c_tiles"] for r in per_rank),
                "stage_ms": {"plan_slowest_rank": slow["plan_ms"], "tasklist_slowest_rank": slow["tasklist_ms"], "gemm_slowest_rank": slow["gemm_ms"],
                             "gemm_max_over_ranks": g_max, "gemm_mean_over_ranks": g_mean, "exchange_max_over_ranks": max(r["exchange_ms"] for r in per_rank),
                             "publish_ms_outside_timed_region": publish_ms},
                "residual_over_mean_gemm": dict(resid, largest=max(resid, key=resid.get)),
                "halo_tiles_received_total": sum(r["recv_tiles"] for r in per_rank), "per_rank": per_rank,
                "roofline": {"bound": "tensor", "kernel": "k_gemm_f64_tma<%d> (FP64 DMMA leaf GEMM), rank 0's launches" % b,
                             "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "peak_source": peak_src,
                             "algorithmic": "2*b^3 flops per leaf product x %d products in rank 0's launches" % nm,
                             "kernel_ms": g_ms, "share_of_step": g_ms / ms, "traffic": None},
                "check": check, "cpu_baseline": None, "e2e": e2e, "gpu_launches": int(sum(r["launches_per_step"] for r in per_rank) * args.steps),
                "host_cpulist_rank0": cpulist, "clocks": clocks}
        print(json.dumps(line), flush=True)
    comm_finalize()
    dist.destroy_process_group()


def _e2e_sharded(hb, H, A, B, w, steps, local_rank):
    """Per rank: pinned host tiles of its slabs -> device, norm refresh, publish, halo exchange, SpAMM, all local C tiles back
    to pinned host memory.  Max over ranks of the wall time between two barriers."""
    from . import _capi
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
    nm_tot = 0
    d2h = 0
    phases = None
    phases_all = []
    WARM = 4                        # untimed passes: the stream-ordered pool, the halo tail and NCCL's buffers reach their steady state
    for i in range(steps + WARM):   # (measured at 4 GPUs: 186, 102, 73 ms for passes 3-5 with only two warm-ups)
        # (barrier() only ENQUEUES its NCCL kernel: without the second synchronize the clock starts while that kernel still waits
        # for the slowest rank, and the first call that happens to wait for the device is billed the skew -- 60-340 ms at 2 GPUs)
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        marks = []

        def mark(name):
            marks.append((name, time.perf_counter()))

        if os.environ.get("HBSM_E2E_ORDER", "BA") == "AB":
            A2 = H(np.float64, b); A2.resize(n, n); A2.assign_tiles(abi, abj, at.numpy()); mark("upload_A")
            A2.update_internal_info(); mark("norms_A")
            B2 = H(np.float64, b); B2.resize(n, n); B2.assign_tiles(bbi, bbj, bt.numpy()); mark("upload_B")
            B2.update_internal_info(); mark("norms_B")
            publish(B2); mark("publish_B")
        else:
            # B first: its norms and published table are what the peers wait for
            B2 = H(np.float64, b); B2.resize(n, n); B2.assign_tiles(bbi, bbj, bt.numpy()); mark("upload_B")
            B2.update_internal_info(); mark("norms_B")
            publish(B2); mark("publish_B")                      # inside the e2e region: B2 is a new matrix every step
            A2 = H(np.float64, b); A2.resize(n, n); A2.assign_tiles(abi, abj, at.numpy()); mark("upload_A")
            A2.update_internal_info(); mark("norms_A")
        t_up = time.perf_counter() - t0
        Cm, nm, nr = sharded_product(A2, False, B2, False, True, tau); mark("sharded_product")
        t_prod = time.perf_counter() - t0 - t_up
        if out is None or out.shape[0] < nr:
            out = torch.empty((nr, b * b), dtype=torch.float64, pin_memory=True)
        cbi = np.zeros(nr, np.int64); cbj = np.zeros(nr, np.int64)
        m = C.c_size_t(0)
        _capi.check(_capi.lib().hbsm_export_leaves(Cm._h, nr, cbi.ctypes.data_as(C.c_void_p), cbj.ctypes.data_as(C.c_void_p),
                                                    None, C.c_void_p(out.data_ptr()), C.byref(m)))
        torch.cuda.synchronize()
        t_local = time.perf_counter() - t0          # this rank's own work (uploads wait for nobody; the product waits for the peers' thresholds / tiles)
        dist.barrier(); torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        del A2, B2, Cm
        v = torch.tensor([dt, float(nm), float(h2d), float(nr * b * b * 8 + 16 * nr)], dtype=torch.float64, device="cuda")
        mx = v.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = v.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        if i >= WARM:
            times.append(float(mx[0]))
            per_rank_ms = [None] * dist.get_world_size()
            dist.all_gather_object(per_rank_ms, round(1e3 * t_local, 2))
            phases = {}
            prev = t0
            for name, t in marks:
                phases[name + "_ms"] = round(1e3 * (t - prev), 3); prev = t
            phases["download_C_ms"] = round(1e3 * (t0 + dt - prev), 3)
            phases["engine_stage_ms"] = {k: round(v, 3) for k, v in hb.stage_times().items() if k.endswith("_ms")}
            phases_all.append({k: v for k, v in phases.items() if k.endswith("_ms") and not isinstance(v, dict)})
            phases["shard_stats"] = shard_stats()
        nm_tot = int(sm[1]); h2d_tot = int(sm[2]); d2h = int(sm[3])
    ms = 1e3 * float(np.mean(times))
    return {"value": 2.0 * b ** 3 * nm_tot / (ms * 1e-3) / 1e12, "unit": "TFLOP/s", "ms_per_step": ms,
            "h2d_bytes_per_step": h2d_tot, "d2h_bytes_per_step": d2h, "ms_per_step_all": [round(1e3 * t, 2) for t in times],
            "last_step_ms_per_rank": per_rank_ms, "rank0_phases": phases, "rank0_phases_all": phases_all,
            "path": "per rank: hbsm_assign_tiles(A_r,B_r from pinned host) + hbsm_update_norms + hbsm_publish + hbsm_sharded_product "
                    "(NCCL halo exchange inside the library) + hbsm_export_leaves(C_r to pinned host); max over ranks"}
