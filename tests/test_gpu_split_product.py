"""Split products on one GPU.  B_full is cut into B's own tiles plus a committed halo (hbsm_halo_reserve / hbsm_halo_commit,
written in shuffled order), and op(A)*op(B) runs through hbsm_product_begin_ex (defer_halo_tiles 1 or 2) +
hbsm_product_finish: the C tiles that read only own tiles and the halo readers are two launches of the leaf kernel on
subsets of C's table, and the fp32 2x2 groups of the 32 / 64 leaves can be cut between the two.  Every result is checked
against the same call on the unsplit B_full, and against a float64 sum over each C tile's exported k-list.  Also: halo
tiles that land after begin (finish waits for the caller's event), the chunked leaf-GEMM launches of hbsm_product_to_host,
and the state of C after a rejected or aborted product."""
import ctypes as C

import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import _capi
from hierarchical_block_sparse_lib_b200 import generators as G
from helpers import bits, check_exact, commit_halo, grouped_bound, klist_sums, morton, tiles_rc

HM = hb.HierarchicalBlockSparseMatrix
gpu = pytest.mark.gpu
TRANS = [(0, 0), (0, 1), (1, 0), (1, 1)]
PATTERNS = ["odd", "kslab", "random", "all", "none"]
GRID = {32: 10, 48: 10, 64: 10, 128: 8, 256: 6}   # block grid side of the operands per leaf size
GROUPED = (32, 64)                                 # fp32 leaves whose kernels compute 2 x 2 groups of C tiles


@pytest.fixture(scope="module")
def engine():
    hb.init(0)


def L():
    return _capi.lib()


# ---------------------------------------------------------------------------------------------------
# operands
# ---------------------------------------------------------------------------------------------------
def integer_operand(dtype, b, n, seed, fill=0.45):
    """random block structure, integer values in [-4, 4] with exact zeros: every sum of products is an exact integer"""
    r, c, v = G.random_block_sparse_coo(n, b, fill, seed, np.float64)
    X = HM(dtype, b)
    X.resize(n, n)
    X.assign_from_vectors(r, c, np.round(4.0 * v).astype(dtype))
    X.update_internal_info()
    return X


def decay_operand(dtype, b, n, seed, W=None):
    W = W if W is not None else min(G.decay_width(8.0 / b), n - 1)
    X = HM(dtype, b)
    X.generate_decay(n, 8.0 / b, W, seed)
    X.update_internal_info()
    return X


def operands(dtype, b, kind):
    n = GRID[b] * b - 5
    make = integer_operand if kind == "int" else decay_operand
    return make(dtype, b, n, 11 + b), make(dtype, b, n, 12 + b)


def median_tau(A, B):
    na = A.export_leaves(tiles=False)[2].astype(np.float64)
    nb = B.export_leaves(tiles=False)[2].astype(np.float64)
    return float(np.sqrt(np.median(na) * np.median(nb)))


def halo_mask(pattern, k, j, g, rng):
    """which tiles of op(B), at op(B) coordinates (k, j), are halo tiles"""
    if pattern == "odd":
        return j % 2 == 1
    if pattern == "kslab":   # a rank owns the block rows of op(B) in [g/4, 3g/4)
        return (k < g // 4) | (k >= 3 * g // 4)
    if pattern == "random":
        return rng.random(len(k)) < 0.3
    if pattern == "all":
        return np.ones(len(k), bool)
    return np.zeros(len(k), bool)


def split_b(Bf, tB, pattern, seed, nan_tiles=False):
    """B_own (B_full without the halo set, norms refreshed) with the halo committed in shuffled order, their exact leaf
    norms taken from B_full.  Returns (B_own, halo set in op(B) coordinates, device address of the halo tiles, the halo
    tiles in the order written)."""
    b = Bf.get_params().blocksize
    n = Bf.get_n_rows()
    bi, bj, nrm, t = Bf.export_leaves()
    k, j = (bj, bi) if tB else (bi, bj)
    rng = np.random.default_rng(seed)
    halo = halo_mask(pattern, k, j, -(-n // b), rng)
    Bo = HM(Bf.dtype, b)
    Bo.resize(n, Bf.get_n_cols())
    own = ~halo
    if own.any():
        Bo.assign_tiles(bi[own], bj[own], t[own])
    Bo.update_internal_info()
    assert Bo.get_n_blocks() == own.sum()
    order = rng.permutation(np.flatnonzero(halo))
    ptr = commit_halo(Bo, bi[order], bj[order], tiles=t[order], norms=nrm[order], nan_tiles=nan_tiles, capacity=8)
    return Bo, set(zip(k[halo].tolist(), j[halo].tolist())), ptr, t[order]


# ---------------------------------------------------------------------------------------------------
# products
# ---------------------------------------------------------------------------------------------------
def product(A, tA, B, tB, spamm, tau, defer, upper=0, event=None):
    """hbsm_product_begin_ex + hbsm_product_finish into a new C; returns (C, n_mults, n_blocks, gemm kernel)"""
    Cm = HM(A.dtype)
    nm, nr = C.c_size_t(0), C.c_size_t(0)
    _capi.check(L().hbsm_product_begin_ex(A._h, tA, B._h, tB, Cm._h, int(spamm), float(tau), 1, defer, upper))
    _capi.check(L().hbsm_product_finish(Cm._h, event, C.byref(nm), C.byref(nr)))
    return Cm, nm.value, nr.value, hb.stage_times()["gemm_kernel"]


def promised_kernel(dtype, b):
    """the kernel launch_leaf_gemm's dispatch table names (last_gemm_kernel): 1 fp64 DMMA, 3 fp32 tcgen05, 0 generic"""
    if b not in (32, 64, 128, 256):
        return 0
    return 1 if dtype == np.float64 else 3


def split_groups(ci, cj, in_second):
    """per C tile: does its 2 x 2 group (Morton key >> 2) have members in both launches?"""
    grp = (ci >> 1) * (1 << 21) + (cj >> 1)
    both = {}
    for gk, f in zip(grp.tolist(), in_second.tolist()):
        both.setdefault(gk, set()).add(bool(f))
    return np.array([len(both[gk]) == 2 for gk in grp.tolist()], bool)


def reads_halo(Cref, halo):
    """per C tile of Cref: does one of its products read a halo tile of op(B)?  (exported k-lists and the halo key set)"""
    ci, cj, _ = tiles_rc(Cref)
    return np.array([any((int(k), int(j)) in halo for k in Cref.tile_tasks(i, j)) for i, j in zip(ci.tolist(), cj.tolist())], bool)


# ---------------------------------------------------------------------------------------------------
# split products against the unsplit call
# ---------------------------------------------------------------------------------------------------
LEAF_CASES = [(d, b, 0) for d in (np.float64, np.float32) for b in (32, 64, 128, 256, 48)] + \
             [(np.float32, 32, 3), (np.float32, 64, 3)]


@gpu
@pytest.mark.parametrize("kind", ["int", "decay"])
@pytest.mark.parametrize("dtype,b,variant", LEAF_CASES,
                         ids=["%s-b%d-v%d" % ("f64" if d == np.float64 else "f32", b, v) for d, b, v in LEAF_CASES])
def test_split_product_equals_the_unsplit_product(engine, dtype, b, variant, kind):
    A, Bf = operands(dtype, b, kind)
    tau = median_tau(A, Bf)
    grouped = dtype == np.float32 and b in GROUPED and variant == 0
    kernel = 3 if variant == 3 else promised_kernel(dtype, b)
    hb.set_gemm_variant(variant)
    try:
        for tA, tB in TRANS:
            refs = {}
            for spamm in (0, 1):
                for upper in ((0, 1) if (tA, tB) == (0, 0) else (0,)):
                    R, rnm, rnr, _ = product(A, tA, Bf, tB, spamm, tau, 0, upper)
                    r, s, K = klist_sums(A, tA, Bf, tB, R)
                    ci, cj, rt = tiles_rc(R)
                    if upper:   # finish zeroes the strict lower part of the diagonal tiles
                        low = np.tril(np.ones((b, b), bool), -1)
                        r[ci == cj] *= ~low
                        s[ci == cj] *= ~low
                    if kind == "int":
                        assert 16 * K.max() < 2 ** 24   # every partial sum is an integer below 2^24: exact in fp32 and TF32
                        check_exact(rt, r)
                    refs[spamm, upper] = (R, rnm, rnr, r, s, K)
                if spamm:
                    assert 0 < refs[1, 0][1] < refs[0, 0][1], "the prune must drop some but not all products"
            for pattern in PATTERNS:
                if pattern != "odd" and (tA, tB) not in ((0, 0), (1, 1)):
                    continue
                Bo, halo, _, _ = split_b(Bf, tB, pattern, 7 * b + 3 * tA + tB)
                if pattern == "all":
                    assert Bo.get_n_blocks() == 0
                for (spamm, upper), (R, rnm, rnr, r, s, K) in refs.items():
                    if upper and pattern != "odd":
                        continue
                    ci, cj, rt = tiles_rc(R)
                    second = reads_halo(R, halo) if pattern != "none" else np.zeros(len(ci), bool)
                    cut = split_groups(ci, cj, second)
                    if pattern == "odd" and not spamm:
                        assert cut.any(), "the odd-column halo must cut some 2 x 2 groups"
                    if pattern == "all":
                        assert second.all()
                    for defer in (1, 2):
                        what = "t%d%d %s spamm=%d upper=%d defer=%d" % (tA, tB, pattern, spamm, upper, defer)
                        X, nm, nr, kern = product(A, tA, Bo, tB, spamm, tau, defer, upper)
                        assert (nm, nr) == (rnm, rnr), what
                        assert np.array_equal(X.export_tasks(), R.export_tasks()), what
                        xi, xj, xt = tiles_rc(X)
                        assert np.array_equal(xi, ci) and np.array_equal(xj, cj), what
                        assert kern == kernel, what
                        if kind == "int":
                            check_exact(xt, r)
                        elif not grouped:   # the same kernel, the same k order per tile
                            assert np.array_equal(bits(xt), bits(rt)), what
                        else:
                            whole = ~cut   # a group inside one launch gets the reference's super-product list
                            assert np.array_equal(bits(xt[whole]), bits(rt[whole])), what
                            err = np.abs(xt[cut].astype(np.float64) - r[cut])
                            assert (err <= grouped_bound(s[cut], K[cut])).all(), what
    finally:
        hb.set_gemm_variant(0)


# ---------------------------------------------------------------------------------------------------
# halo tiles that land after begin
# ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32)])
def test_halo_readers_wait_for_the_event(engine, dtype, b):
    """keys and norms are valid at begin, the tiles are NaN until a copy queued on another stream behind ~100 ms of sleep
    lands; finish gets the event recorded after that copy.  A halo reader launched before the event, or put into the
    first list, writes NaN into C.  The reference is the same split product with the tiles in place (for the grouped
    fp32 kernels a cut 2 x 2 group is not bitwise the unsplit product's: test_split_product_equals_the_unsplit_product)."""
    import torch
    cu = C.CDLL("libcuda.so.1")
    A, Bf = operands(dtype, b, "decay")
    tau = median_tau(A, Bf)
    for spamm in (0, 1):
        R, rnm, rnr, _ = product(A, 0, Bf, 0, spamm, tau, 0)
        for defer in (1, 2):
            Bo, halo, ptr, ht = split_b(Bf, 0, "odd", 5)
            assert halo
            W, _, _, _ = product(A, 0, Bo, 0, spamm, tau, defer)   # warm-up and reference, the true tiles in place
            _, _, rt = tiles_rc(W)
            if dtype == np.float64:
                assert_same(W, R)
            Bo, _, ptr, ht = split_b(Bf, 0, "odd", 5, nan_tiles=True)
            src = torch.from_numpy(np.ascontiguousarray(ht)).cuda()
            torch.cuda.synchronize()
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                torch.cuda._sleep(200_000_000)   # ~100 ms at B200 clocks
                assert cu.cuMemcpyDtoDAsync_v2(C.c_uint64(ptr), C.c_uint64(src.data_ptr()), C.c_size_t(src.numel() * src.element_size()),
                                               C.c_void_p(side.cuda_stream)) == 0
                ev = torch.cuda.Event()
                ev.record(side)
            X, nm, nr, _ = product(A, 0, Bo, 0, spamm, tau, defer, event=C.c_void_p(ev.cuda_event))
            torch.cuda.synchronize()
            _, _, xt = tiles_rc(X)
            assert (nm, nr) == (rnm, rnr)
            assert np.array_equal(X.export_tasks(), R.export_tasks())
            assert not np.isnan(xt).any(), "a halo reader ran before the halo tiles arrived"
            assert np.array_equal(bits(xt), bits(rt))


# ---------------------------------------------------------------------------------------------------
# chunked hbsm_product_to_host
# ---------------------------------------------------------------------------------------------------
def to_host(A, tA, B, tB, tau, n_tiles):
    import torch
    b = A.get_params().blocksize
    tdt = torch.float64 if A.dtype == np.float64 else torch.float32
    host = torch.zeros((n_tiles, b * b), dtype=tdt, pin_memory=True)
    Cm = HM(A.dtype)
    nm, nr = C.c_size_t(0), C.c_size_t(0)
    _capi.check(L().hbsm_product_to_host(A._h, tA, B._h, tB, Cm._h, 1, float(tau), 1, C.c_void_p(host.data_ptr()), n_tiles,
                                          C.byref(nm), C.byref(nr)))
    return Cm, nm.value, nr.value, host.numpy()[:nr.value], hb.stage_times()["gemm_kernel"]


CHUNK_CASES = [(np.float32, 32, "int"), (np.float32, 32, "decay"), (np.float32, 64, "int"), (np.float32, 64, "decay"),
               (np.float32, 128, "decay"), (np.float64, 256, "decay")]


@gpu
@pytest.mark.parametrize("dtype,b,kind", CHUNK_CASES,
                         ids=["%s-b%d-%s" % ("f64" if d == np.float64 else "f32", b, k) for d, b, k in CHUNK_CASES])
def test_product_to_host_in_eight_chunks(engine, dtype, b, kind):
    """more than 8 * 1024 C tiles: the leaf GEMM runs in 8 ranges of C's table, and a range boundary can cut a 2 x 2 group"""
    if kind == "int":   # ~72 % of a 128 x 128 grid of C tiles
        A, B = (integer_operand(dtype, b, 128 * b - 7, s, fill=0.1) for s in (21, 22))
    else:               # a band of +-5 tiles: C has up to 21 tile diagonals of a 512 x 512 grid
        A, B = (decay_operand(dtype, b, 512 * b - 7, s, W=5 * b) for s in (23, 24))
    na = A.export_leaves(tiles=False)[2].astype(np.float64)
    nb = B.export_leaves(tiles=False)[2].astype(np.float64)
    tau = float(np.sqrt(np.quantile(na, 0.1) * np.quantile(nb, 0.1)))   # a light prune: C keeps more than 8192 tiles
    R = HM(dtype)
    rnm, rnr = HM.spamm(A, 0, B, 1, R, tau, True)
    assert rnr > 8 * 1024, "8 chunks need more than 8192 C tiles"
    nchunks = 8
    X, nm, nr, host, kern = to_host(A, 0, B, 1, tau, rnr + 3)
    assert (nm, nr) == (rnm, rnr) and kern == promised_kernel(dtype, b)
    assert np.array_equal(X.export_tasks(), R.export_tasks())
    xi, xj, _, xt_cm = X.export_leaves(norms=False)
    ri, rj, _, rt_cm = R.export_leaves(norms=False)
    assert np.array_equal(xi, ri) and np.array_equal(xj, rj)
    assert np.array_equal(bits(host), bits(xt_cm)), "the host buffer differs from C"
    if dtype == np.float64 or b not in GROUPED:
        assert np.array_equal(bits(xt_cm), bits(rt_cm))
        return
    keys = np.array([morton(i, j) for i, j in zip(xi.tolist(), xj.tolist())], np.uint64)
    assert (np.diff(keys.astype(np.int64)) > 0).all()   # C's table order
    pos = np.arange(rnr)
    chunk = np.searchsorted([rnr * c // nchunks for c in range(1, nchunks)], pos, side="right")
    grp = keys >> np.uint64(2)
    cut = np.zeros(rnr, bool)
    for gk in np.unique(grp):
        m = grp == gk
        cut[m] = len(np.unique(chunk[m])) > 1
    assert cut.any(), "a chunk boundary must cut a 2 x 2 group"
    r, s, K = klist_sums(A, 0, B, 1, R)
    _, _, xt = tiles_rc(X)
    _, _, rt = tiles_rc(R)
    if kind == "int":
        assert 16 * K.max() < 2 ** 24
        check_exact(xt, r)
    else:
        assert np.array_equal(bits(xt[~cut]), bits(rt[~cut]))
        assert (np.abs(xt.astype(np.float64) - r) <= grouped_bound(s, K)).all()


# ---------------------------------------------------------------------------------------------------
# failure paths: C as it was
# ---------------------------------------------------------------------------------------------------
def small_case(dtype=np.float64, b=32):
    A, Bf = operands(dtype, b, "decay")
    return A, Bf, median_tau(A, Bf)


def assert_same(X, Y):
    xi, xj, xt = tiles_rc(X)
    yi, yj, yt = tiles_rc(Y)
    assert np.array_equal(xi, yi) and np.array_equal(xj, yj) and np.array_equal(bits(xt), bits(yt))
    assert np.array_equal(X.export_tasks(), Y.export_tasks())


@gpu
def test_rejected_spamm_leaves_c_empty(engine):
    """spamm(updated=0) with a halo on B is refused; C stays unsized and takes the next product"""
    A, Bf, tau = small_case()
    Bo, _, _, _ = split_b(Bf, 0, "odd", 1)
    want = HM(np.float64)
    HM.spamm(A, 0, Bf, 0, want, tau, True)
    Cm = HM(np.float64)
    assert L().hbsm_spamm(A._h, 0, Bo._h, 0, Cm._h, tau, 0, None, None) == _capi.HBSM_E_ARG
    assert Cm.empty()
    HM.spamm(A, 0, Bo, 0, Cm, tau, True)
    assert_same(Cm, want)
    # the same through the accumulating call into an unsized C
    acc_want = HM(np.float64)
    HM.spamm_accumulate(A, 0, Bf, 0, acc_want, -0.5, 2.0, tau, True)
    Ca = HM(np.float64)
    assert L().hbsm_multiply_accumulate(A._h, 0, Bo._h, 0, Ca._h, -0.5, 2.0, 1, tau, 0, None, None) == _capi.HBSM_E_ARG
    assert Ca.empty()
    HM.spamm_accumulate(A, 0, Bo, 0, Ca, -0.5, 2.0, tau, True)
    assert_same(Ca, acc_want)


@gpu
def test_too_deep_a_grid_leaves_c_empty(engine):
    """a block grid deeper than 21 levels does not fit the 64-bit task keys: refused, C stays unsized"""
    n = 3 << 20   # leaf size 1: 2^22 block rows
    A = HM(np.float64, 1)
    A.resize(n, n)
    Cm = HM(np.float64)
    assert L().hbsm_multiply(A._h, 0, A._h, 0, Cm._h, None, None) == _capi.HBSM_E_ARG
    assert Cm.empty()


@gpu
@pytest.mark.parametrize("defer", [1, 2])
def test_aborted_product_leaves_c_empty(engine, defer):
    A, Bf, tau = small_case(np.float32, 32)
    Bo, _, _, _ = split_b(Bf, 0, "odd", 2)
    R, rnm, rnr, _ = product(A, 0, Bo, 0, 1, tau, defer)   # the same split product, into a C of its own
    Cm = HM(np.float32)
    _capi.check(L().hbsm_product_begin(A._h, 0, Bo._h, 0, Cm._h, 1, tau, 1, defer))
    _capi.check(L().hbsm_product_abort())
    assert Cm.empty()
    nm, nr = C.c_size_t(0), C.c_size_t(0)
    _capi.check(L().hbsm_product_begin(A._h, 0, Bo._h, 0, Cm._h, 1, tau, 1, defer))
    _capi.check(L().hbsm_product_finish(Cm._h, None, C.byref(nm), C.byref(nr)))
    assert (nm.value, nr.value) == (rnm, rnr)
    assert_same(Cm, R)


@gpu
def test_begin_and_finish_out_of_order(engine):
    A, Bf, tau = small_case()
    Bo, _, _, _ = split_b(Bf, 0, "odd", 3)
    R, _, _, _ = product(A, 0, Bf, 0, 0, 0.0, 0)
    C1, C2 = HM(np.float64), HM(np.float64)
    assert L().hbsm_product_finish(C1._h, None, None, None) == _capi.HBSM_E_ARG   # no product in flight
    _capi.check(L().hbsm_product_begin(A._h, 0, Bo._h, 0, C1._h, 0, 0.0, 1, 1))
    assert L().hbsm_product_begin(A._h, 0, Bo._h, 0, C2._h, 0, 0.0, 1, 1) == _capi.HBSM_E_ARG   # one at a time
    assert C2.empty()
    assert L().hbsm_product_finish(C2._h, None, None, None) != _capi.HBSM_OK   # another C: refused, the product dropped
    assert C1.empty() and C2.empty()
    assert L().hbsm_product_finish(C1._h, None, None, None) == _capi.HBSM_E_ARG
    assert C1.empty()
    _capi.check(L().hbsm_product_begin(A._h, 0, Bo._h, 0, C1._h, 0, 0.0, 1, 1))
    _capi.check(L().hbsm_product_finish(C1._h, None, None, None))
    assert_same(C1, R)


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32)])
def test_halo_stays_usable(engine, dtype, b):
    """after a split product: commit(0) gives the own-only product; the halo committed again, and after
    update_internal_info(B), the split product again"""
    A, Bf = operands(dtype, b, "decay")
    tau = median_tau(A, Bf)
    Bo, halo, _, _ = split_b(Bf, 0, "odd", 4)
    R, _, _, _ = product(A, 0, Bf, 0, 1, tau, 0)
    first, _, _, _ = product(A, 0, Bo, 0, 1, tau, 1)
    assert np.array_equal(first.export_tasks(), R.export_tasks())
    if dtype == np.float64:   # (fp32 32-leaves: a cut 2 x 2 group is only error-bounded against R)
        assert_same(first, R)
    # the own tiles alone, as a matrix of their own
    bi, bj, _, t = Bo.export_leaves()
    Own = HM(dtype, b)
    Own.resize(Bf.get_n_rows(), Bf.get_n_cols())
    Own.assign_tiles(bi, bj, t)
    Own.update_internal_info()
    want_own = HM(dtype)
    HM.spamm(A, 0, Own, 0, want_own, tau, True)
    _capi.check(L().hbsm_halo_commit(Bo._h, 0))
    got_own = HM(dtype)
    HM.spamm(A, 0, Bo, 0, got_own, tau, True)
    assert_same(got_own, want_own)
    assert len(got_own.export_tasks()) < len(R.export_tasks())
    _capi.check(L().hbsm_halo_commit(Bo._h, len(halo)))   # the tail still holds the tiles
    again, _, _, _ = product(A, 0, Bo, 0, 1, tau, 2)
    assert_same(again, first)
    Bo.update_internal_info()
    after, _, _, _ = product(A, 0, Bo, 0, 1, tau, 1)
    assert_same(after, first)
