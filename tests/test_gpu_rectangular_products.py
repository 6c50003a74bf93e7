"""Rectangular and depth-mismatched products at every leaf kernel, tile by tile against exact references.

op(A) = M x K and op(B) = K x N (the stored operand is K x M when tA is set, N x K when tB is set), at shapes where the
operands and C have different depths: long contractions, outer products, single-leaf C from deep operands, single-leaf
operands, a K that crosses into the next depth, single elements.  Every shape runs with all four (tA, tB).  For each
product: C's shape and depth, the executed set against the flat rule on the exported leaf norms (and against the CPU
port of the reference's recursive rule at b = 32 and 64), the counters, the kernel that ran, and every C tile against
a float64 sum over its k-list -- exact for integer operands; for real operands bitwise equal to the same call on square
embeddings of the operands (same tiles at the same coordinates in S x S matrices of equal depth), and for fp64 within
2 gamma_K |A||B| of the float64 sum.  Then the other entry points on the same shapes: the accumulating product,
hbsm_product_to_host, hbsm_product_from_host (slab and bulk paths), the symmetric family, the SpAMM error bounds,
worth_to_multiply / worth_to_spamm, and the size refusals.  A single-leaf C whose product executes nothing is still
delivered to the host as its zero leaf."""
import ctypes as C
import zlib

import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import _capi
from oracle import pyoracle as po
from helpers import bits, check_call, check_exact, composition, copy_of, assert_bitwise, flat_rule_tasks, sort_tasks, tiles_rc
from test_gpu_spamm_error_control import Ref, check_choice, taus_for

HM = hb.HierarchicalBlockSparseMatrix
gpu = pytest.mark.gpu
TRANS = [(0, 0), (0, 1), (1, 0), (1, 1)]
LONG = {32: 24, 48: 20, 64: 16, 128: 10, 256: 8}   # the long side in blocks per leaf size
GROUPED = (32, 64)                                  # fp32 leaves whose kernels compute 2 x 2 groups of C tiles


# ---------------------------------------------------------------------------------------------------
# shapes (M, K, N) of op(A) = M x K, op(B) = K x N
# ---------------------------------------------------------------------------------------------------
def depth_rule(m, n, b):
    """Matrix::depth_for: 0 for a single leaf, else the smallest P >= 1 with 2^P blocks covering max(m, n)"""
    if m <= b and n <= b:
        return 0
    covers = -(-max(m, n) // b)
    P, two = 1, 2
    while covers > two:
        two *= 2
        P += 1
    return P


def shape(name, b):
    x, s, o = LONG[b] * b - 5, 2 * b + 3, b - 7
    return {"long_contraction": (s, x, o),
            "outer_product": (x, o, x - b),
            "a_deep_b_shallow": (x, s, o),
            "a_shallow_b_deep": (o, s, x),
            "single_leaf_c": (o, x, b),
            "single_leaf_a": (o, b - 3, x),
            "single_leaf_b": (x, b - 3, o),
            "depth_boundary": (4 * b, 4 * b + 1, 8 * b),
            "one_element": (1, 1, 1),
            "one_element_long_k": (1, x, 1)}[name]


def blocks(n, b):
    return -(-n // b)


def depth_claims(name, M, K, N, b):
    """what each row of the shape table is for, as depth relations of op(A), op(B) and C"""
    dA, dB, dC = depth_rule(M, K, b), depth_rule(K, N, b), depth_rule(M, N, b)
    return {"long_contraction": dA > dC and dB > dC,
            "outer_product": blocks(K, b) == 1 and dC == max(dA, dB) > 0,
            "a_deep_b_shallow": dA > dB > 0 and blocks(N, b) == 1,
            "a_shallow_b_deep": dB > dA > 0 and blocks(M, b) == 1,
            "single_leaf_c": dC == 0 and min(dA, dB) > 0 and N == b,
            "single_leaf_a": dA == 0 < dB,
            "single_leaf_b": dB == 0 < dA,
            "depth_boundary": dA == depth_rule(M, K - 1, b) + 1 and blocks(M, b) == 4 and dC == dA,
            "one_element": M == K == N == 1 and dA == dB == dC == 0,
            "one_element_long_k": M == N == 1 and dC == 0 and dA == dB > 0}[name]


SHAPES = ["long_contraction", "outer_product", "a_deep_b_shallow", "a_shallow_b_deep", "single_leaf_c", "single_leaf_a",
          "single_leaf_b", "depth_boundary", "one_element", "one_element_long_k"]
DEEP_OPERANDS = [s for s in SHAPES if all(depth_rule(*d, 32) > 0 for d in (shape(s, 32)[:2], shape(s, 32)[1:]))]


def stored(M, K, N, tA, tB):
    """(rows, cols) of the stored A and B"""
    return (K, M) if tA else (M, K), (N, K) if tB else (K, N)


# ---------------------------------------------------------------------------------------------------
# kernels: (dtype, leaf size, hbsm_set_gemm_variant)
# ---------------------------------------------------------------------------------------------------
KERNELS = [(d, b, 0) for d in (np.float64, np.float32) for b in (32, 64, 128, 256, 48)] + \
          [(np.float32, 32, 3), (np.float32, 64, 3), (np.float64, 64, 1)]
KIDS = ["%s-b%d-v%d" % ("f64" if d == np.float64 else "f32", b, v) for d, b, v in KERNELS]


def promised_kernel(dtype, b, variant):
    """the kernel launch_leaf_gemm's dispatch table names: 1 fp64 DMMA, 3 fp32 tcgen05, 0 generic FMA"""
    if variant == 1 or b not in (32, 64, 128, 256):
        return 0
    return 1 if dtype == np.float64 else 3


# ---------------------------------------------------------------------------------------------------
# operands
# ---------------------------------------------------------------------------------------------------
class Operand:
    """a block-sparse rows x cols operand held in numpy: tiles t[n] indexed (row, col) at (bi[n], bj[n]), and the padded
    float64 dense matrix D of whole blocks (zero outside the tiles)"""

    def __init__(self, dtype, b, rows, cols, bi, bj, t):
        self.dtype, self.b, self.rows, self.cols = np.dtype(dtype), b, rows, cols
        self.bi, self.bj = np.asarray(bi, np.int64), np.asarray(bj, np.int64)
        t = np.array(t, np.float64).reshape(len(self.bi), b, b)
        r = np.arange(b)
        for p in range(len(self.bi)):   # padding rows and columns are zero, as assembly leaves them
            t[p][self.bi[p] * b + r >= rows, :] = 0.0
            t[p][:, self.bj[p] * b + r >= cols] = 0.0
        self.t = t.astype(dtype)
        self.D = np.zeros((blocks(rows, b) * b, blocks(cols, b) * b))
        for p in range(len(self.bi)):
            self.D[self.bi[p] * b:(self.bi[p] + 1) * b, self.bj[p] * b:(self.bj[p] + 1) * b] = self.t[p]

    def subset(self, keep):
        return Operand(self.dtype, self.b, self.rows, self.cols, self.bi[keep], self.bj[keep], self.t[keep])

    def colmajor(self):
        return np.ascontiguousarray(self.t.transpose(0, 2, 1).reshape(len(self.bi), -1))

    def gpu(self, rows=None, cols=None, update=True):
        """the engine's matrix (rows x cols: an embedding with the same tiles at the same coordinates)"""
        X = HM(self.dtype, self.b)
        X.resize(rows or self.rows, cols or self.cols)
        if len(self.bi):
            X.assign_tiles(self.bi, self.bj, self.colmajor())
        if update:
            X.update_internal_info()
        return X

    def oracle(self):
        """the CPU port's matrix: every element of every tile (zeros included) assigned"""
        b, rr, cc, vv = self.b, [], [], []
        for p in range(len(self.bi)):
            r, c = np.meshgrid(np.arange(self.bi[p] * b, min((self.bi[p] + 1) * b, self.rows)),
                               np.arange(self.bj[p] * b, min((self.bj[p] + 1) * b, self.cols)), indexing="ij")
            rr.append(r.ravel()); cc.append(c.ravel()); vv.append(self.t[p][r - self.bi[p] * b, c - self.bj[p] * b].ravel())
        cat = lambda a, dt: np.concatenate(a).astype(dt) if a else np.zeros(0, dt)
        return po.from_coo(po.OrcMatrix, b, self.rows, self.cols, cat(rr, np.int64), cat(cc, np.int64), cat(vv, self.dtype), self.dtype)

    def op(self, t):
        return self.D.T if t else self.D


def random_operand(dtype, b, rows, cols, kind, rng, fill=0.5):
    """about `fill` of the tiles, with an empty block row and an empty block column where there is more than one, and at
    least one tile.  int: integers in [-4, 4] with exact zeros; real: U[-1, 1) times a per-tile scale 10^-U(0, 6)"""
    gr, gc = blocks(rows, b), blocks(cols, b)
    free = np.ones((gr, gc), bool)
    if gr > 1:
        free[rng.integers(gr), :] = False
    if gc > 1:
        free[:, rng.integers(gc)] = False
    mask = free & (rng.random((gr, gc)) < fill)
    if not mask.any():
        mask[tuple(np.argwhere(free)[0])] = True
    bi, bj = np.nonzero(mask)
    n = len(bi)
    if kind == "int":
        t = rng.integers(-4, 5, (n, b, b)).astype(np.float64)
    else:
        t = rng.uniform(-1, 1, (n, b, b)) * (10.0 ** -rng.uniform(0, 6, n))[:, None, None]
    return Operand(dtype, b, rows, cols, bi, bj, t)


def operand_pair(dtype, b, name, tA, tB, kind, tag=""):
    M, K, N = shape(name, b)
    (ar, ac), (br, bc) = stored(M, K, N, tA, tB)
    rng = np.random.default_rng(zlib.crc32(("%s-%d-%d%d-%s%s" % (name, b, tA, tB, kind, tag)).encode()))
    if kind == "int":   # every partial sum is an integer below 2^24: exact in fp64, fp32 and split TF32
        assert 16 * blocks(K, b) * b < 2 ** 24
    return random_operand(dtype, b, ar, ac, kind, rng), random_operand(dtype, b, br, bc, kind, rng)


def grid(*dims_and_b):
    *dims, b = dims_and_b
    return max(1, max(blocks(d, b) for d in dims))


def pick_tau(A, tA, B, tB):
    """a tau between two candidate levels fl(nA * nB) in the middle of their range (the widest gap there): the prune
    drops some products and keeps others; None when there are fewer than two levels"""
    lv = Ref(A, tA, B, tB).levels().astype(np.float64)
    lv = lv[lv > 0]
    if len(lv) < 2:
        return None
    lo, hi = max(1, len(lv) // 3), max(2, 2 * len(lv) // 3 + 1)
    i = lo + int(np.argmax(lv[lo:hi] / lv[lo - 1:hi - 1]))
    return float(np.sqrt(np.sqrt(lv[i - 1] * lv[i])))


def splitmix64(x):
    m = (1 << 64) - 1
    x = (x + 0x9E3779B97F4A7C15) & m
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & m
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & m
    return x ^ (x >> 31)


def checksum(tasks):
    return sum(splitmix64(int(i) << 42 | int(j) << 21 | int(k)) for i, j, k in tasks) & ((1 << 64) - 1)


def klist_reference(a, tA, bop, tB, tasks, ci, cj):
    """per C tile (ci, cj): the float64 sum over its k-list of op(A)(i,k) op(B)(k,j) (r), of |op(A)(i,k)| |op(B)(k,j)| (s),
    and K = b * (length of the k-list); from the numpy operands, padding included"""
    b = a.b
    DA, DB = a.op(tA), bop.op(tB)
    r = np.zeros((len(ci), b, b))
    s = np.zeros_like(r)
    K = np.zeros(len(ci), np.int64)
    pos = {(i, j): p for p, (i, j) in enumerate(zip(ci.tolist(), cj.tolist()))}
    ks = {}
    for i, j, k in np.asarray(tasks).tolist():
        ks.setdefault(pos[(i, j)], []).append(k)
    for p, kl in ks.items():
        idx = (np.asarray(kl)[:, None] * b + np.arange(b)[None, :]).ravel()
        x = DA[ci[p] * b:(ci[p] + 1) * b][:, idx]
        y = DB[idx][:, cj[p] * b:(cj[p] + 1) * b]
        r[p] = x @ y
        s[p] = np.abs(x) @ np.abs(y)
        K[p] = b * len(kl)
    return r, s, K


def check_shape(Cm, M, N, b):
    """dims, depth (get_depth is the deepest existing leaf: 0 without tiles, H:496), consistency (a sized, childless
    non-leaf is not consistent, H:1809), and no tile outside ceil(M/b) x ceil(N/b)"""
    L = Cm.get_n_blocks()
    assert (Cm.get_n_rows(), Cm.get_n_cols()) == (M, N)
    assert Cm.expected_depth() == depth_rule(M, N, b)
    assert Cm.get_depth() == (depth_rule(M, N, b) if L else 0)
    assert Cm.check_if_matrix_is_consistent() == (L > 0)
    ci, cj, _, _ = Cm.export_leaves(tiles=False, norms=False)
    assert (ci < blocks(M, b)).all() and (cj < blocks(N, b)).all(), "a C tile outside ceil(M/b) x ceil(N/b)"


def expected_tiles(tasks, M, N, b):
    """C's tile set: the tiles with executed products, and the zero leaf of a single-leaf C without any"""
    t = {(int(i), int(j)) for i, j, _ in tasks}
    if not t and depth_rule(M, N, b) == 0:
        t = {(0, 0)}
    return t


@pytest.fixture(scope="module")
def engine(oracle_built):
    hb.init(0)


def run(A, tA, B, tB, tau, updated):
    Cm = HM(A.dtype)
    if tau is None:
        nm, nr = HM.multiply(A, tA, B, tB, Cm)
    else:
        nm, nr = HM.spamm(A, tA, B, tB, Cm, tau, updated)
    return Cm, nm, nr, hb.stage_times()["gemm_kernel"]


# ---------------------------------------------------------------------------------------------------
# multiply and SpAMM: every shape x transpose x kernel x operand kind
# ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", SHAPES)
@pytest.mark.parametrize("dtype,b,variant", KERNELS, ids=KIDS)
def test_multiply_and_spamm(engine, dtype, b, variant, name):
    M, K, N = shape(name, b)
    S = max(M, K, N)
    g = grid(M, K, N, b)
    kernel = promised_kernel(dtype, b, variant)
    with_oracle = b in (32, 64) and variant == 0
    ran = 0
    hb.set_gemm_variant(variant)
    try:
        for tA, tB in TRANS:
            for kind in ("int", "real"):
                a, bo = operand_pair(dtype, b, name, tA, tB, kind)
                A, B = a.gpu(), bo.gpu()
                As, Bs = a.gpu(S, S), bo.gpu(S, S)
                tau = pick_tau(A, tA, B, tB)
                calls = [(None, True)] + ([(tau, True), (tau, False)] if tau is not None else [])
                if with_oracle:
                    Ao, Bo = a.oracle(), bo.oracle()
                n_all = None
                for tau_, updated in calls:
                    what = "t%d%d %s tau=%s updated=%d" % (tA, tB, kind, tau_, updated)
                    Cm, nm, nr, kern = run(A, tA, B, tB, tau_, updated)
                    check_shape(Cm, M, N, b)
                    want = sort_tasks(flat_rule_tasks(A, tA, B, tB, tau_, g))
                    got = Cm.export_tasks()
                    assert np.array_equal(sort_tasks(got), want), what
                    assert nm == len(want) == Cm.get_n_block_multiplications(), what
                    ci, cj, ct = tiles_rc(Cm)
                    assert set(zip(ci.tolist(), cj.tolist())) == expected_tiles(want, M, N, b), what
                    assert nr == len(ci) == Cm.get_n_blocks(), what
                    assert Cm.task_checksum() == checksum(want), what
                    if nm:
                        assert kern == kernel, what
                        ran += 1
                    if tau_ is None:
                        n_all = nm
                    else:
                        assert 0 < nm < n_all, "tau must prune some products but not all: " + what
                    if with_oracle:
                        Co, onm, onb, ot = po.OrcMatrix.product(Ao, tA, Bo, tB, spamm=tau_ is not None,
                                                                tau=tau_ or 0.0, want_tasks=True)
                        assert (onm, onb) == (nm, nr), what
                        assert np.array_equal(sort_tasks(ot), want), what
                        assert Co.depth() == Cm.get_depth() and Co.consistent() == Cm.check_if_matrix_is_consistent(), what
                    r, s, Kk = klist_reference(a, tA, bo, tB, got, ci, cj)
                    if kind == "int":
                        check_exact(ct, r)
                        continue
                    Q, qnm, qnr, _ = run(As, tA, Bs, tB, tau_, updated)
                    assert np.array_equal(sort_tasks(Q.export_tasks()), want), what
                    qi, qj, qt = tiles_rc(Q)
                    live = Kk > 0   # (the zero leaf of a single-leaf C without products has no tile in the embedding)
                    assert np.array_equal(qi, ci[live]) and np.array_equal(qj, cj[live]), what
                    assert np.array_equal(bits(qt), bits(ct[live])), "differs from the square embedding: " + what
                    assert not ct[~live].any()
                    if dtype == np.float64:   # |c - exact| and |r - exact| are both below gamma_K |A||B|
                        u = 2.0 ** -53
                        gam = (Kk * u / (1 - Kk * u))[:, None, None]
                        assert (np.abs(ct - r) <= 2 * gam * s).all(), what
    finally:
        hb.set_gemm_variant(0)
    if name not in ("one_element", "one_element_long_k"):
        assert ran > 0, "the promised kernel never ran"


# ---------------------------------------------------------------------------------------------------
# the accumulating product
# ---------------------------------------------------------------------------------------------------
ACC_KERNELS = [(np.float64, 32), (np.float64, 64), (np.float32, 32), (np.float32, 64), (np.float64, 128), (np.float32, 256),
               (np.float64, 48)]
AB = [(1.0, 1.0), (-0.75, 0.5), (2.0, 0.0)]


def old_c(P, M, N, b, dtype, rng):
    """C_old, M x N: some tiles inside P's pattern, some outside"""
    pi, pj, _, _ = P.export_leaves(tiles=False, norms=False)
    gi, gj = np.meshgrid(np.arange(blocks(M, b)), np.arange(blocks(N, b)), indexing="ij")
    gi, gj = gi.ravel(), gj.ravel()
    inP = np.isin(gi * (1 << 21) + gj, pi * (1 << 21) + pj)
    keep = rng.random(len(gi)) < np.where(inP, 0.5, 0.3)
    keep[np.flatnonzero(inP)[:1]] = True
    keep[np.flatnonzero(~inP)[:1]] = True
    return Operand(dtype, b, M, N, gi[keep], gj[keep], rng.uniform(-1, 1, (int(keep.sum()), b, b))).gpu(update=False)


@gpu
@pytest.mark.parametrize("name", SHAPES)
@pytest.mark.parametrize("dtype,b", ACC_KERNELS, ids=["%s-b%d" % ("f64" if d == np.float64 else "f32", b) for d, b in ACC_KERNELS])
def test_multiply_accumulate(engine, dtype, b, name):
    M, K, N = shape(name, b)
    for tA, tB in TRANS:
        a, bo = operand_pair(dtype, b, name, tA, tB, "real", "acc")
        A, B = a.gpu(), bo.gpu()
        P = HM(dtype, b)
        HM.multiply(A, tA, B, tB, P)
        Cold = old_c(P, M, N, b, dtype, np.random.default_rng(tA * 2 + tB))
        tau = pick_tau(A, tA, B, tB)
        for spamm in ((None, tau) if tau is not None else (None,)):
            for alpha, beta in AB:
                check_call(A, tA, B, tB, Cold, alpha, beta, spamm=spamm)
        if name == "single_leaf_c":   # SpAMM skips every product: C is the zero leaf, scaled, plus beta C_old
            for alpha, beta in AB:
                Cm, _ = check_call(A, tA, B, tB, Cold, alpha, beta, spamm=1e30)
                assert len(Cm.export_tasks()) == 0 and Cm.get_n_blocks() == 1


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32)])
def test_multiply_accumulate_in_place_rectangular(engine, dtype, b):
    """X <- alpha X Y + beta X, C is A, with X M x K (M != K and a different number of blocks) and Y K x K"""
    rng = np.random.default_rng(17)
    for M, K in ((LONG[b] * b - 5, 2 * b + 3), (2 * b + 3, LONG[b] * b - 5), (b - 7, 3 * b + 1)):
        X = random_operand(dtype, b, M, K, "real", rng).gpu()
        for tB in (0, 1):
            Y = random_operand(dtype, b, K, K, "real", rng).gpu()
            for alpha, beta in AB:
                for spamm in (None, 1e-4):
                    what = "M=%d K=%d tB=%d alpha=%g beta=%g spamm=%s" % (M, K, tB, alpha, beta, spamm)
                    want, P = composition(X, 0, Y, tB, X, alpha, beta, spamm)
                    Z = copy_of(X)
                    Z.update_internal_info()   # (copy does not carry the leaf norms, H:1490)
                    if spamm is None:
                        nm, nr = HM.multiply_accumulate(Z, 0, Y, tB, Z, alpha, beta)
                    else:
                        nm, nr = HM.spamm_accumulate(Z, 0, Y, tB, Z, alpha, beta, spamm)
                    assert np.array_equal(Z.export_tasks(), P.export_tasks()), what
                    assert_bitwise(Z, want)
                    assert nm == len(P.export_tasks()) and nr == want.get_n_blocks(), what
                    assert (Z.get_n_rows(), Z.get_n_cols()) == (M, K)


# ---------------------------------------------------------------------------------------------------
# hbsm_product_to_host
# ---------------------------------------------------------------------------------------------------
def pinned(n_tiles, b, dtype, fill=np.nan):
    import torch
    h = torch.full((max(n_tiles, 1), b * b), fill, dtype=torch.float64 if dtype == np.float64 else torch.float32, pin_memory=True)
    return h, h.numpy()


def to_host(A, tA, B, tB, tau, n_tiles):
    """hbsm_product_to_host into a NaN-filled pinned buffer of n_tiles tiles; returns (C, n_mults, n_resizes, buffer)"""
    b = A.get_params().blocksize
    h, host = pinned(n_tiles, b, A.dtype)
    Cm = HM(A.dtype)
    nm, nr = C.c_size_t(0), C.c_size_t(0)
    _capi.check(_capi.lib().hbsm_product_to_host(A._h, tA, B._h, tB, Cm._h, int(tau is not None), float(tau or 0.0), 1,
                                                 C.c_void_p(h.data_ptr()), n_tiles, C.byref(nm), C.byref(nr)))
    return Cm, nm.value, nr.value, host.copy()


@gpu
@pytest.mark.parametrize("name", SHAPES)
@pytest.mark.parametrize("dtype,b", [(np.float64, 32), (np.float64, 64), (np.float32, 32), (np.float32, 64)])
def test_product_to_host(engine, dtype, b, name):
    for tA, tB in TRANS:
        for kind in ("int", "real"):
            a, bo = operand_pair(dtype, b, name, tA, tB, kind)
            A, B = a.gpu(), bo.gpu()
            tau = pick_tau(A, tA, B, tB)
            for tau_ in ((None, tau) if tau is not None else (None,)):
                R, rnm, rnr, _ = run(A, tA, B, tB, tau_, True)
                X, nm, nr, host = to_host(A, tA, B, tB, tau_, rnr + 2)
                assert (nm, nr) == (rnm, rnr)
                assert_bitwise(X, R)
                assert np.array_equal(X.export_tasks(), R.export_tasks())
                _, _, _, xt = X.export_leaves(norms=False)
                assert np.array_equal(bits(host[:nr]), bits(xt)), "the host tiles differ from C"
                assert np.isnan(host[nr:]).all()


@gpu
@pytest.mark.parametrize("dtype,b,kind", [(np.float32, 32, "int"), (np.float64, 64, "real")])
def test_product_to_host_outer_product_in_eight_chunks(engine, dtype, b, kind):
    """an outer product with more than 8192 C tiles: the leaf GEMM runs in 8 ranges of C's table"""
    rng = np.random.default_rng(3)
    M = N = 100 * b - 5
    a = random_operand(dtype, b, M, b - 7, kind, rng, fill=0.99)
    bo = random_operand(dtype, b, b - 7, N, kind, rng, fill=0.99)
    A, B = a.gpu(), bo.gpu()
    R, rnm, rnr, _ = run(A, 0, B, 0, None, True)
    assert rnr > 8 * 1024, "8 chunks need more than 8192 C tiles"
    X, nm, nr, host = to_host(A, 0, B, 0, None, rnr + 1)
    assert (nm, nr) == (rnm, rnr) and hb.stage_times()["gemm_kernel"] == promised_kernel(dtype, b, 0)
    assert np.array_equal(X.export_tasks(), R.export_tasks())
    xi, xj, xt = tiles_rc(X)
    assert np.array_equal(bits(host[:nr]), bits(X.export_leaves(norms=False)[3]))
    assert np.isnan(host[nr:]).all()
    r, _, _ = klist_reference(a, 0, bo, 0, X.export_tasks(), xi, xj)
    if kind == "int":   # (the fp32 32-leaf 2 x 2 groups are cut at range boundaries: exact values, not R's bits)
        check_exact(xt, r)
    else:
        assert_bitwise(X, R)


# ---------------------------------------------------------------------------------------------------
# hbsm_product_from_host: the slab path (both operands deep) and the bulk path (a single-leaf operand)
# ---------------------------------------------------------------------------------------------------
def from_host(a, tA, bo, tB, tau, n_slabs, cap, perm=None):
    """hbsm_product_from_host through the C ABI, NaN-filled host tiles and -1-filled coordinates"""
    A2, B2, Cm = HM(a.dtype, a.b), HM(a.dtype, a.b), HM(a.dtype)
    A2.resize(a.rows, a.cols)
    B2.resize(bo.rows, bo.cols)
    pa = perm[0] if perm else np.arange(len(a.bi))
    pb = perm[1] if perm else np.arange(len(bo.bi))
    abi, abj = (np.ascontiguousarray(x[pa], np.int32) for x in (a.bi, a.bj))
    bbi, bbj = (np.ascontiguousarray(x[pb], np.int32) for x in (bo.bi, bo.bj))
    at, bt = a.colmajor()[pa], bo.colmajor()[pb]
    h, host = pinned(cap, a.b, a.dtype)
    cbi, cbj = np.full(max(cap, 1), -1, np.int32), np.full(max(cap, 1), -1, np.int32)
    nm, nr = C.c_size_t(0), C.c_size_t(0)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    _capi.check(_capi.lib().hbsm_product_from_host(A2._h, len(abi), p(abi), p(abj), p(at), tA, B2._h, len(bbi), p(bbi), p(bbj),
                                                   p(bt), tB, Cm._h, int(tau is not None), float(tau or 0.0), n_slabs,
                                                   C.c_void_p(h.data_ptr()), cap, p(cbi), p(cbj), C.byref(nm), C.byref(nr)))
    return A2, B2, Cm, nm.value, nr.value, host.copy(), cbi, cbj


def same_operand(X, Y):
    xi, xj, xn, xt = X.export_leaves()
    yi, yj, yn, yt = Y.export_leaves()
    assert np.array_equal(xi, yi) and np.array_equal(xj, yj) and np.array_equal(bits(xn), bits(yn)) and np.array_equal(bits(xt), bits(yt))
    assert X.get_frob_norm_squared_internal() == Y.get_frob_norm_squared_internal()


@gpu
@pytest.mark.parametrize("name", SHAPES)
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float64, 32), (np.float32, 32), (np.float32, 64)])
def test_product_from_host(engine, dtype, b, name):
    slabs = [(0, False), (1, False), (4, False), (16, False), (4, True)] if name in DEEP_OPERANDS else [(0, False), (4, True)]
    grouped = dtype == np.float32 and b in GROUPED
    for tA, tB in TRANS:
        a, bo = operand_pair(dtype, b, name, tA, tB, "int", "fh")
        A, B = a.gpu(), bo.gpu()
        tau = pick_tau(A, tA, B, tB)
        for tau_ in ((None, tau) if tau is not None else (None,)):
            R, rnm, rnr, _ = run(A, tA, B, tB, tau_, True)
            ri, rj, rt = tiles_rc(R)
            for n_slabs, shuffled in slabs:
                rng = np.random.default_rng(n_slabs)
                perm = (rng.permutation(len(a.bi)), rng.permutation(len(bo.bi))) if shuffled else None
                A2, B2, Cm, nm, nr, host, cbi, cbj = from_host(a, tA, bo, tB, tau_, n_slabs, rnr + 2, perm)
                what = "t%d%d tau=%s slabs=%d shuffled=%d" % (tA, tB, tau_, n_slabs, shuffled)
                assert (nm, nr) == (rnm, rnr), what
                same_operand(A2, A)
                same_operand(B2, B)
                ci, cj, ct = tiles_rc(Cm)
                assert np.array_equal(ci, ri) and np.array_equal(cj, rj), what
                if grouped:   # slabs of one block row cut the 2 x 2 groups: exact integers, signs of zeros aside
                    check_exact(ct, rt.astype(np.float64))
                else:
                    assert np.array_equal(bits(ct), bits(rt)), what
                # the host tiles, labelled by (c_bi, c_bj), are C's
                assert np.isnan(host[nr:]).all() and (cbi[nr:] == -1).all()
                pos = {(i, j): p for p, (i, j) in enumerate(zip(ci.tolist(), cj.tolist()))}
                order = [pos[(i, j)] for i, j in zip(cbi[:nr].tolist(), cbj[:nr].tolist())]
                assert sorted(order) == list(range(nr)), what
                _, _, _, cm = Cm.export_leaves(norms=False)
                assert np.array_equal(bits(host[:nr]), bits(cm[order])), what


# ---------------------------------------------------------------------------------------------------
# a single-leaf C whose product executes nothing is delivered to the host as its zero leaf
# ---------------------------------------------------------------------------------------------------
def disjoint_pair(dtype, b, name):
    """int operands whose tiles never meet on k: A's in even k blocks, B's in odd ones (one k block: B has no tiles)"""
    a, bo = operand_pair(dtype, b, name, 0, 0, "int", "disjoint")
    return a.subset(a.bj % 2 == 0), bo.subset(bo.bi % 2 == 1)


@gpu
@pytest.mark.parametrize("name", ["single_leaf_c", "one_element", "one_element_long_k"])   # slab, bulk, slab path
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32), (np.float64, 48)])
def test_single_leaf_c_without_products_reaches_the_host(engine, dtype, b, name):
    M, K, N = shape(name, b)
    assert depth_rule(M, N, b) == 0
    cases = [("skip", operand_pair(dtype, b, name, 0, 0, "int", "skip"), 1e30)]
    if blocks(K, b) > 1:
        cases.append(("disjoint", disjoint_pair(dtype, b, name), None))
    zero = np.zeros(b * b, dtype)
    for what, (a, bo), tau in cases:
        A, B = a.gpu(), bo.gpu()
        R, rnm, rnr, _ = run(A, 0, B, 0, tau, True)
        assert (rnm, rnr) == (0, 1), what
        X, nm, nr, host = to_host(A, 0, B, 0, tau, 4)
        assert (nm, nr) == (0, 1), what
        assert np.array_equal(bits(host[0]), bits(zero)), "product_to_host left C's zero leaf undelivered: " + what
        assert np.isnan(host[1:]).all()
        for n_slabs in (0, 4):
            _, _, Cm, nm, nr, host, cbi, cbj = from_host(a, 0, bo, 0, tau, n_slabs, 4)
            assert (nm, nr) == (0, 1), what
            assert np.array_equal(bits(host[0]), bits(zero)), "product_from_host left C's zero leaf undelivered: " + what
            assert (cbi[0], cbj[0]) == (0, 0), what
            assert np.isnan(host[1:]).all() and (cbi[1:] == -1).all()
            assert_bitwise(Cm, R)


# ---------------------------------------------------------------------------------------------------
# the symmetric family on rectangular operands
# ---------------------------------------------------------------------------------------------------
def block_triu_mask(n, b):
    i, j = np.arange(n)[:, None], np.arange(n)[None, :]
    return (i // b < j // b) | ((i // b == j // b) & (i <= j))


def symmetric_upper(dtype, b, n, seed, nan=False):
    """upper storage of an integer symmetric n x n matrix (tiles with bi <= bj, diagonal tiles upper triangular) and the
    dense symmetric matrix it stands for; with nan, NaN in the parts the symmetric family ignores: the strict lower part
    of the diagonal tiles, and three tiles below the diagonal"""
    rng = np.random.default_rng(seed)
    g = blocks(n, b)
    V = rng.integers(-4, 5, (g * b, g * b)).astype(np.float64)
    V[n:, :] = 0.0
    V[:, n:] = 0.0
    bi, bj = np.nonzero(np.triu(rng.random((g, g)) < 0.6) | np.eye(g, dtype=bool))
    U = np.zeros_like(V)
    tiles = []
    for i, j in zip(bi, bj):
        t = V[i * b:(i + 1) * b, j * b:(j + 1) * b]
        t = np.triu(t) if i == j else t.copy()
        U[i * b:(i + 1) * b, j * b:(j + 1) * b] = t
        if nan and i == j:
            t = t.copy()
            t[np.tril(np.ones((b, b), bool), -1)] = np.nan
        tiles.append(t)
    below = [(j, i) for i, j in zip(bi, bj) if i < j][:3] if nan else []
    tiles += [np.full((b, b), np.nan) for _ in below]
    bi = np.concatenate([bi, [p[0] for p in below]]).astype(np.int64)
    bj = np.concatenate([bj, [p[1] for p in below]]).astype(np.int64)
    X = HM(dtype, b)
    X.resize(n, n)
    X.assign_tiles(bi, bj, np.stack(tiles).transpose(0, 2, 1).reshape(len(bi), -1).astype(dtype))
    return X, (U + np.triu(U, 1).T)[:n, :n]


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32), (np.float32, 128), (np.float64, 48)])
def test_symmetric_family(engine, dtype, b):
    """symm_rk of a rectangular A: triu(A A^T) and triu(A^T A), diagonal tiles masked; symm_multiply with a rectangular
    non-symmetric operand on either side, and the same with NaN where the upper storage is ignored"""
    rng = np.random.default_rng(b)
    x, s = LONG[b] * b - 5, 2 * b + 3
    for M, K in ((x, s), (s, x)):
        a = random_operand(dtype, b, M, K, "int", rng)
        A = a.gpu()
        D = a.D[:M, :K]
        for transposed, full in ((0, D @ D.T), (1, D.T @ D)):
            Cm = HM(dtype)
            HM.symm_rk(A, transposed, Cm)
            n = full.shape[0]
            assert (Cm.get_n_rows(), Cm.get_n_cols()) == (n, n)
            ci, cj, _, _ = Cm.export_leaves(tiles=False, norms=False)
            assert (ci <= cj).all()
            check_exact(Cm.to_dense(), full * block_triu_mask(n, b))
        U, Sd = symmetric_upper(dtype, b, K, 7 * b + M)
        Un, _ = symmetric_upper(dtype, b, K, 7 * b + M, nan=True)
        for left in (True, False):
            other = random_operand(dtype, b, K, M, "int", rng) if left else a
            O = other.gpu()
            Do = other.D[:other.rows, :other.cols]
            outs = []
            for Sym in (U, Un):
                Cm = HM(dtype)
                if left:
                    HM.symm_multiply(Sym, 1, O, 0, Cm)
                else:
                    HM.symm_multiply(O, 0, Sym, 1, Cm)
                outs.append(Cm)
            check_exact(outs[0].to_dense(), Sd @ Do if left else Do @ Sd)
            assert not np.isnan(outs[1].export_leaves(norms=False)[3]).any(), "an ignored part of the upper storage was read"
            assert_bitwise(outs[1], outs[0])


# ---------------------------------------------------------------------------------------------------
# SpAMM error bounds, worth_to_*, refusals
# ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", ["long_contraction", "outer_product"])
def test_spamm_error_bounds(engine, dtype, name):
    b = 32
    for tA, tB in TRANS:
        a, bo = operand_pair(dtype, b, name, tA, tB, "real", "bounds")
        A, B = a.gpu(), bo.gpu()
        ref = Ref(A, tA, B, tB)
        taus = taus_for(ref)
        bounds, ns = HM.spamm_error_bounds(A, tA, B, tB, taus)
        exp = np.array([ref.bound(t) for t in taus])
        assert np.array_equal(ns, [int(ref.skipped(t).sum()) for t in taus])
        assert np.all(np.abs(bounds - exp) <= 1e-12 * exp)
        scale = float(np.linalg.norm(a.D) * np.linalg.norm(bo.D))
        for rel in (0.0, 1e-8, 1e-4, 1e-2, 10.0):
            info = HM.spamm_tau_for_error(A, tA, B, tB, rel * scale)
            Cm, nm, _, _ = run(A, tA, B, tB, info["tau"], True)
            check_choice(ref, info, rel * scale, Cm.export_tasks(), nm)


@gpu
@pytest.mark.parametrize("name", SHAPES)
def test_worth(engine, name):
    for dtype, b in ((np.float64, 32), (np.float32, 64)):
        M, K, N = shape(name, b)
        g = grid(M, K, N, b)
        for tA, tB in TRANS:
            pairs = [operand_pair(dtype, b, name, tA, tB, "real")] + ([disjoint_pair(dtype, b, name)] if (tA, tB) == (0, 0) else [])
            for a, bo in pairs:
                A, B = a.gpu(), bo.gpu()
                assert HM.worth_to_multiply(A, tA, B, tB) == (len(flat_rule_tasks(A, tA, B, tB, None, g)) > 0)
                for tau in (0.0, pick_tau(A, tA, B, tB) or 1.0, 1e18):
                    assert HM.worth_to_spamm(A, tA, B, tB, tau) == (len(flat_rule_tasks(A, tA, B, tB, tau, g)) > 0)


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 32), (np.float32, 64)])
def test_inner_dims_off_by_one_are_refused(engine, dtype, b):
    """op(A) M x K times op(B) (K + 1) x N, K and K + 1 covering the same blocks: "bad sizes", C stays empty"""
    rng = np.random.default_rng(1)
    for M, K, N in ((2 * b + 3, LONG[b] * b - 5, b - 7), (b - 7, b - 3, 3 * b), (4 * b, 4 * b + 1, 8 * b)):
        assert blocks(K, b) == blocks(K + 1, b)
        for tA, tB in TRANS:
            (ar, ac), _ = stored(M, K, N, tA, tB)
            _, (br, bc) = stored(M, K + 1, N, tA, tB)
            A = random_operand(dtype, b, ar, ac, "int", rng).gpu()
            B = random_operand(dtype, b, br, bc, "int", rng).gpu()
            for spamm in (False, True):
                Cm = HM(dtype)
                with pytest.raises(hb.HbsmError, match="matrices have bad sizes!"):
                    if spamm:
                        HM.spamm(A, tA, B, tB, Cm, 1e-3, True)
                    else:
                        HM.multiply(A, tA, B, tB, Cm)
                assert Cm.empty()


# ---------------------------------------------------------------------------------------------------
# CPU: the shape table, the flat rule, the integer bound
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("b", sorted(LONG))
def test_shape_table_has_the_depth_relations_it_claims(b):
    for name in SHAPES:
        M, K, N = shape(name, b)
        assert min(M, K, N) >= 1
        assert depth_claims(name, M, K, N, b), (name, b, (M, K, N))
    assert set(DEEP_OPERANDS) == {"long_contraction", "outer_product", "a_deep_b_shallow", "a_shallow_b_deep", "single_leaf_c",
                                  "depth_boundary", "one_element_long_k"}


def test_depth_rule_is_the_engines():
    for (m, n, b), d in {(32, 32, 32): 0, (33, 1, 32): 1, (64, 64, 32): 1, (65, 3, 32): 2, (128, 1, 32): 2, (129, 1, 32): 3,
                         (1, 1, 1): 0, (763, 40, 32): 5, (2043, 2043, 256): 3}.items():
        assert depth_rule(m, n, b) == d, (m, n, b)


@pytest.mark.parametrize("b", sorted(LONG))
def test_integer_operands_stay_exact(b):
    for name in SHAPES:
        M, K, N = shape(name, b)
        assert 16 * blocks(K, b) * b < 2 ** 24   # |a b| <= 16 per term: every partial sum an integer below 2^24


class _Leaves:
    """export_leaves of a structure without tiles (the flat rule reads coordinates and norms only)"""

    def __init__(self, bi, bj, norms):
        self.l = (np.asarray(bi, np.int64), np.asarray(bj, np.int64), np.asarray(norms), None)

    def export_leaves(self, tiles=True, norms=True):
        return self.l


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_flat_rule_matches_a_brute_force_loop(dtype):
    rng = np.random.default_rng(4)
    for trial in range(40):
        ga, gk, gb = rng.integers(1, 7, 3)
        tA, tB = TRANS[trial % 4]
        def structure(r, c):
            m = rng.random((r, c)) < rng.uniform(0.2, 0.9)
            bi, bj = np.nonzero(m)
            return bi, bj, (10.0 ** rng.uniform(-6, 2, len(bi))).astype(dtype)
        abi, abj, an = structure(*((gk, ga) if tA else (ga, gk)))
        bbi, bbj, bn = structure(*((gb, gk) if tB else (gk, gb)))
        levels = np.array([x * y for x in an for y in bn], dtype)
        for tau in (None, 0.0, float(np.sqrt(np.median(levels))) if len(levels) else 1.0, 1e9):
            want = []
            for p in range(len(abi)):
                i, k = (abj[p], abi[p]) if tA else (abi[p], abj[p])
                for q in range(len(bbi)):
                    k2, j = (bbj[q], bbi[q]) if tB else (bbi[q], bbj[q])
                    if k == k2 and (tau is None or an[p] * bn[q] > dtype(tau) * dtype(tau)):
                        want.append((i, j, k))
            got = flat_rule_tasks(_Leaves(abi, abj, an), tA, _Leaves(bbi, bbj, bn), tB, tau, int(max(ga, gk, gb)))
            assert np.array_equal(sort_tasks(got), sort_tasks(np.array(want, np.int64))), (trial, tau)
