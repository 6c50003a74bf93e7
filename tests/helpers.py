"""Shared helpers for the parity tests: build the same matrix in the CUDA engine (through the C ABI) and in the CPU
oracle from one set of COO triplets, and compare results."""
import ctypes as C

import numpy as np

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import _capi
from hierarchical_block_sparse_lib_b200 import generators as G
from oracle import pyoracle as po

HBSM = hb.HierarchicalBlockSparseMatrix


def morton(bi, bj):
    key = 0
    for bit in range(21):
        key |= ((int(bi) >> bit) & 1) << (2 * bit) | ((int(bj) >> bit) & 1) << (2 * bit + 1)
    return key


def commit_halo(X, bi, bj, seed=0, tiles=None, norms=None, nan_tiles=False, capacity=0):
    """hbsm_halo_reserve / hbsm_halo_commit: len(bi) halo tiles at (bi, bj) on X, written in the given order.  The tiles
    are `tiles` (rows of b*b, column-major) or random values from `seed`; the norms are `norms` or the tiles' leaf norms.
    nan_tiles: the keys and norms as above, but every tile NaN (tiles still in transit).  The reserve has room for
    max(capacity, len(bi)) tiles.  Returns the device address of the first halo tile."""
    b = X.get_params().blocksize
    n = len(bi)
    if tiles is None:
        tiles = np.random.default_rng(seed).uniform(-1, 1, (n, b * b))
    tiles = np.ascontiguousarray(tiles, X.dtype).reshape(n, b * b)
    if norms is None:
        norms = (tiles.astype(np.float64) ** 2).sum(1)
    norms = np.ascontiguousarray(norms, X.dtype)
    keys = np.array([morton(i, j) for i, j in zip(bi, bj)], np.uint64)
    written = np.full_like(tiles, np.nan) if nan_tiles else tiles
    dk, dn, dt = C.c_void_p(), C.c_void_p(), C.c_void_p()
    _capi.check(_capi.lib().hbsm_halo_reserve(X._h, max(n, capacity), C.byref(dk), C.byref(dn), C.byref(dt)))
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuCtxSynchronize() == 0   # the reserve's copies on the engine stream are done
    for ptr, arr in ((dk, keys), (dn, norms), (dt, written)):
        if arr.nbytes:
            assert cu.cuMemcpyHtoD_v2(C.c_uint64(ptr.value), arr.ctypes.data_as(C.c_void_p), C.c_size_t(arr.nbytes)) == 0
    _capi.check(_capi.lib().hbsm_halo_commit(X._h, n))
    return dt.value


def gpu_from_coo(b, m, n, r, c, v, dtype=np.float64, update=True):
    A = HBSM(dtype, b)
    A.resize(m, n)
    A.assign_from_vectors(r, c, v)
    if update:
        A.update_internal_info()
    return A


def both_from_coo(b, m, n, r, c, v, dtype=np.float64, cls=None):
    cls = cls or po.OrcMatrix
    return gpu_from_coo(b, m, n, r, c, v, dtype), po.from_coo(cls, b, m, n, r, c, v, dtype)


def both_from_dense(b, D, dtype=np.float64, cls=None):
    D = np.asarray(D, dtype)
    m, n = D.shape
    r, c = np.meshgrid(np.arange(m), np.arange(n), indexing="ij")
    return both_from_coo(b, m, n, r.ravel(), c.ravel(), D.ravel(), dtype, cls)


def sort_tasks(t):
    t = np.asarray(t, np.int64).reshape(-1, 3)
    return t[np.lexsort((t[:, 2], t[:, 1], t[:, 0]))]


def rel_frob(x, y):
    d = np.linalg.norm(np.asarray(x, np.float64) - np.asarray(y, np.float64))
    s = np.linalg.norm(np.asarray(y, np.float64))
    return d / s if s > 0 else d


def leaves_equal_structure(g, o):
    gbi, gbj, _, _ = g.export_leaves(tiles=False)
    obi, obj, _, _ = o.leaves(tiles=False)
    return np.array_equal(gbi, obi) and np.array_equal(gbj, obj)


def decay_pair(n, lam, dtype=np.float64, seeds=(1, 2), eps=1e-12):
    W = min(G.decay_width(lam, eps), n - 1)
    return G.decay_coo(n, lam, W, seeds[0], dtype=dtype), G.decay_coo(n, lam, W, seeds[1], dtype=dtype)


# ---------------------------------------------------------------------------------------------------
# backend adapters: one scenario (tests/known_answers.py, the golden fixtures) runs through the CPU oracle port,
# the unmodified reference (oracle/_ref) or the CUDA engine with the same calls
# ---------------------------------------------------------------------------------------------------
class OracleBackend:
    """OrcMatrix (plain-C port) or RefMatrix (unmodified reference compiled in place)."""

    def __init__(self, cls, dtype=np.float64):
        self.cls = cls
        self.dtype = np.dtype(dtype)
        self.name = cls.kind

    def sized(self, b, m, n):
        A = self.cls(b, self.dtype); A.resize(m, n); return A

    def coo(self, b, m, n, r, c, v, update=True):
        return po.from_coo(self.cls, b, m, n, r, c, np.asarray(v, self.dtype), self.dtype, update)

    def dense(self, b, D, update=True):
        return po.from_dense(self.cls, b, D, self.dtype, True, update)

    def to_dense(self, A): return A.to_dense()
    def depth(self, A): return A.depth()
    def shape(self, A): return tuple(A.shape())
    def consistent(self, A): return A.consistent()
    def n_blocks(self, A): return A.n_blocks()
    def n_mults(self, A): return A.n_mults()
    def nnz(self, A): return A.nnz()
    def frob_sq(self, A): return float(A.frob_sq())
    def get(self, A, r, c): return A.get(r, c)
    def get_all(self, A): return A.get_all()
    def leaves(self, A, tiles=True): return A.leaves(tiles)
    def update(self, A): A.update()

    def product(self, A, tA, B, tB, spamm=False, tau=0.0, want_tasks=False):
        return self.cls.product(A, tA, B, tB, spamm=spamm, tau=tau, want_tasks=want_tasks)

    def worth_to_multiply(self, A, tA, B, tB): return self.cls.worth(A, tA, B, tB)
    def worth_to_spamm(self, A, tA, B, tB, tau): return self.cls.worth(A, tA, B, tB, True, tau)
    def add(self, A, B): return self.cls.add(A, B)
    def transpose(self, A): return self.cls.transpose(A)
    def upper(self, A): return self.cls.upper(A)
    def rescale(self, A, alpha): return self.cls.rescale(A, alpha)
    def copy(self, A): return self.cls.copy(A)
    def trunc(self, A, t): return self.cls.trunc(A, t)
    def can_estimate(self): return hasattr(self.cls, "count_skips")
    def count_skips(self, A, tA, B, tB, taus, tr, sp): return self.cls.count_skips(A, tA, B, tB, taus, int(tr), int(sp))
    def spamm_errors(self, A, tA, B, tB, taus): return self.cls.spamm_errors(A, tA, B, tB, taus)
    def can_serialize(self): return hasattr(self.cls, "write_to_buffer")
    def serialize(self, A): return A.write_to_buffer()
    def deserialize(self, b, data): A = self.cls(b, self.dtype); A.assign_from_buffer(data); return A
    def symm_multiply(self, A, sA, B, sB): return self.cls.symm_multiply(A, int(sA), B, int(sB))
    def symm_square(self, A): return self.cls.symm_square(A)
    def symm_rk(self, A, transposed): return self.cls.symm_rk(A, int(transposed))


class GpuBackend:
    """The CUDA engine through the C ABI (Python mirror of the reference class)."""
    name = "cuda"

    def __init__(self, dtype=np.float64):
        self.dtype = np.dtype(dtype)

    def sized(self, b, m, n):
        A = HBSM(self.dtype, b); A.resize(m, n); return A

    def coo(self, b, m, n, r, c, v, update=True):
        return gpu_from_coo(b, m, n, r, c, np.asarray(v, self.dtype), self.dtype, update)

    def dense(self, b, D, update=True):
        D = np.asarray(D, self.dtype)
        m, n = D.shape
        r, c = np.meshgrid(np.arange(m), np.arange(n), indexing="ij")
        return self.coo(b, m, n, r.ravel(), c.ravel(), D.ravel(), update)

    def to_dense(self, A): return A.to_dense()
    def depth(self, A): return A.get_depth()
    def shape(self, A): return (A.get_n_rows(), A.get_n_cols())
    def consistent(self, A): return A.check_if_matrix_is_consistent()
    def n_blocks(self, A): return A.get_n_blocks()
    def n_mults(self, A): return A.get_n_block_multiplications()
    def nnz(self, A): return A.get_nnz()
    def frob_sq(self, A): return float(A.get_frob_squared())
    def get(self, A, r, c): return A.get_values(r, c)
    def get_all(self, A): return A.get_all_values()
    def update(self, A): A.update_internal_info()

    def leaves(self, A, tiles=True):
        return A.export_leaves(tiles=tiles)

    def product(self, A, tA, B, tB, spamm=False, tau=0.0, want_tasks=False):
        Cm = HBSM(self.dtype)
        if spamm:
            nm, nb = HBSM.spamm(A, tA, B, tB, Cm, tau, True)
        else:
            nm, nb = HBSM.multiply(A, tA, B, tB, Cm)
        return Cm, nm, nb, (Cm.export_tasks() if want_tasks else None)

    def worth_to_multiply(self, A, tA, B, tB): return HBSM.worth_to_multiply(A, tA, B, tB)
    def worth_to_spamm(self, A, tA, B, tB, tau): return HBSM.worth_to_spamm(A, tA, B, tB, tau)

    def _out(self, fn, *args):
        Cm = HBSM(self.dtype); fn(*args, Cm); return Cm

    def add(self, A, B): return self._out(HBSM.add, A, B)
    def transpose(self, A): return self._out(HBSM.transpose, A)
    def upper(self, A): Cm = HBSM(self.dtype); A.get_upper_triangle(Cm); return Cm
    def rescale(self, A, alpha): Cm = HBSM(self.dtype); Cm.rescale(A, alpha); return Cm
    def copy(self, A): Cm = HBSM(self.dtype); Cm.copy(A); return Cm
    def trunc(self, A, t): Cm = HBSM(self.dtype); r = A.frob_block_trunc(Cm, t); return Cm, r
    def can_estimate(self): return True
    def count_skips(self, A, tA, B, tB, taus, tr, sp): return HBSM.count_skips(A, tA, B, tB, taus, tr, sp)
    def spamm_errors(self, A, tA, B, tB, taus): return HBSM.get_spamm_errors(A, tA, B, tB, taus)
    def can_serialize(self): return True
    def serialize(self, A): return A.write_to_buffer()
    def deserialize(self, b, data): A = HBSM(self.dtype); A.assign_from_buffer(data); return A
    def symm_multiply(self, A, sA, B, sB): return self._out(HBSM.symm_multiply, A, sA, B, sB)
    def symm_square(self, A): return self._out(HBSM.symm_square, A)
    def symm_rk(self, A, transposed): return self._out(HBSM.symm_rk, A, transposed)


# ---------------------------------------------------------------------------------------------------
# products checked tile by tile: exact and error-bounded references, the flat rule, the accumulating composition
# ---------------------------------------------------------------------------------------------------
def tiles_rc(X):
    """C's tiles as (n, b, b) arrays indexed (row, col), with their block coordinates"""
    b = X.get_params().blocksize
    bi, bj, _, t = X.export_leaves(norms=False)
    return bi, bj, t.reshape(-1, b, b).transpose(0, 2, 1)


def bits(x):
    return x.view(np.uint64 if x.dtype == np.float64 else np.uint32)


def klist_sums(A, tA, Bf, tB, Cref):
    """per C tile of Cref, the float64 sums over its exported k-list of op(A)(i,k) op(B)(k,j) (r) and of
    |op(A)(i,k)| |op(B)(k,j)| (s), and K = b * (length of the k-list); computed with torch on the device"""
    import torch
    b = A.get_params().blocksize
    dev = torch.device("cuda")

    def stack(X):
        bi, bj, _, t = X.export_leaves(norms=False)
        g = int(max(bi.max(initial=0), bj.max(initial=0))) + 1
        where = np.full((g, g), -1, np.int64)
        where[bi, bj] = np.arange(len(bi))
        return where, torch.from_numpy(t.astype(np.float64).reshape(-1, b, b)).to(dev).transpose(1, 2)

    wa, ta = stack(A)
    wb, tb = stack(Bf)
    ci, cj, _ = tiles_rc(Cref)
    tasks = Cref.export_tasks()
    pos = {(i, j): p for p, (i, j) in enumerate(zip(ci.tolist(), cj.tolist()))}
    ct = np.array([pos[(i, j)] for i, j in zip(tasks[:, 0].tolist(), tasks[:, 1].tolist())], np.int64)
    ti, tj, tk = tasks[:, 0], tasks[:, 1], tasks[:, 2]
    ia = wa[tk, ti] if tA else wa[ti, tk]
    ib = wb[tj, tk] if tB else wb[tk, tj]
    assert (ia >= 0).all() and (ib >= 0).all()
    r = torch.zeros((len(ci), b, b), dtype=torch.float64, device=dev)
    s = torch.zeros_like(r)
    step = max(1, (1 << 27) // (b * b * 8))
    for lo in range(0, len(tasks), step):
        a = ta[torch.from_numpy(ia[lo:lo + step]).to(dev)]
        bb = tb[torch.from_numpy(ib[lo:lo + step]).to(dev)]
        if tA:
            a = a.transpose(1, 2)
        if tB:
            bb = bb.transpose(1, 2)
        idx = torch.from_numpy(ct[lo:lo + step]).to(dev)
        r.index_add_(0, idx, a @ bb)
        s.index_add_(0, idx, a.abs() @ bb.abs())
    K = b * np.bincount(ct, minlength=len(ci))
    return r.cpu().numpy(), s.cpu().numpy(), K


def grouped_bound(s, K):
    """|c - r| <= bound, element by element, for the fp32 grouped kernels (r, s: klist_sums).
    Operands: x = hi + lo exactly, hi = x with 13 mantissa bits cleared, |lo| < 2^-10 |x|; the tensor core reads lo with
    13 mantissa bits cleared too, an error below 2^-21 |x|.  The 32-leaf kernel multiplies all four of hi/lo x hi/lo, the
    64-leaf kernel drops lo*lo (< 2^-20 |a b|), so one product a*b is off by at most (2^-20 + 2 * 2^-21 + 2^-42) |a b|
    <= 2^-19 (1 + 2^-22) |a b|; summed, at most 2^-19 (1 + 2^-22) s.
    Sums: every addition, truncating in the tensor core or rounding in the epilogue, errs by less than 2^-23 times the sum
    of the magnitudes of the terms under it, at most s (1 + 2^-8) (the hi/lo parts of a b add up to at most
    (1 + 2^-10)^2 |a b|).  A term passes through at most 2b + 2n + 1 <= 3K additions (n = K / b products in the k-list,
    b >= 32): at most 2b in one accumulator (two super-products of b k's, or hi and lo rows of one), two epilogue adds
    per stage and one final add.  So the sums add less than 3K 2^-23 s (1 + 2^-8) (1 + 2^-23)^(3K), and the float64
    reference is within 3K 2^-53 s of the exact sum.  Total: below (2^-19 + 3.3 K 2^-23) s for K < 2^18.  The bound
    doubles the first term and takes 4K for 3.3K."""
    assert (K < 2 ** 18).all()
    return (2.0 ** -18 + 4.0 * K[:, None, None] * 2.0 ** -23) * s


def check_exact(c, r):
    """integer operands: every element is the exact integer (signs of zeros aside, so compared after adding +0)"""
    assert np.array_equal(bits(c + c.dtype.type(0)), bits(r.astype(c.dtype) + c.dtype.type(0))), \
        "max |c - r| = %g" % np.abs(c.astype(np.float64) - r).max()


def flat_rule_tasks(A, tA, B, tB, tau, g, upper_only=False):
    """{(ci,cj,k)}: both tiles exist and fl(nsq(A_tile) * nsq(B_tile)) > fl(tau*tau) in Treal (tau None = exact multiply)."""
    abi, abj, an, _ = A.export_leaves(tiles=False)
    bbi, bbj, bn, _ = B.export_leaves(tiles=False)
    if tA: abi, abj = abj, abi          # op(A): ci = abi, k = abj
    if tB: bbi, bbj = bbj, bbi          # op(B): k = bbi, cj = bbj
    T = an.dtype.type
    tau2 = None if tau is None else T(tau) * T(tau)
    oa = np.argsort(abj, kind="stable"); ob = np.argsort(bbi, kind="stable")
    a_ci, a_k, a_n = abi[oa], abj[oa], an[oa]
    b_k, b_cj, b_n = bbi[ob], bbj[ob], bn[ob]
    sa = np.searchsorted(a_k, np.arange(g + 1)); sb = np.searchsorted(b_k, np.arange(g + 1))
    out = []
    for k in range(g):
        ia = slice(sa[k], sa[k + 1]); ib = slice(sb[k], sb[k + 1])
        if ia.start == ia.stop or ib.start == ib.stop:
            continue
        keep = np.ones((ia.stop - ia.start, ib.stop - ib.start), bool) if tau2 is None else (a_n[ia][:, None] * b_n[ib][None, :]) > tau2
        if upper_only:
            keep &= a_ci[ia][:, None] <= b_cj[ib][None, :]
        x, y = np.nonzero(keep)
        out.append(np.stack([a_ci[ia][x], b_cj[ib][y], np.full(len(x), k)], 1))
    return np.concatenate(out) if out else np.zeros((0, 3), np.int64)


def copy_of(X):
    Y = HBSM(X.dtype, X.get_params().blocksize)
    if not X.empty():
        Y.copy(X)
    return Y


def composition(A, tA, B, tB, Cold, alpha, beta, spamm=None, updated=True):
    """add(rescale(P, alpha), rescale(C_old, beta)) on copies, with its P"""
    b = A.get_params().blocksize
    P = HBSM(A.dtype, b)
    if spamm is None:
        HBSM.multiply(A, tA, B, tB, P)
    else:
        HBSM.spamm(A, tA, B, tB, P, spamm, updated)
    P1 = HBSM(A.dtype, b)
    P1.rescale(P, alpha)
    if beta == 0.0 or Cold.empty():
        return P1, P
    C1 = HBSM(A.dtype, b)
    C1.rescale(Cold, beta)
    R = HBSM(A.dtype, b)
    HBSM.add(P1, C1, R)
    return R, P


def assert_bitwise(X, Y):
    xi, xj, _, xt = X.export_leaves(norms=False)
    yi, yj, _, yt = Y.export_leaves(norms=False)
    assert np.array_equal(xi, yi) and np.array_equal(xj, yj)
    it = np.uint64 if X.dtype == np.float64 else np.uint32
    assert X.dtype == Y.dtype and np.array_equal(xt.view(it), yt.view(it))
    assert (X.get_n_rows(), X.get_n_cols()) == (Y.get_n_rows(), Y.get_n_cols())


def check_call(A, tA, B, tB, Cold, alpha, beta, spamm=None, updated=True):
    want, P = composition(A, tA, B, tB, Cold, alpha, beta, spamm, updated)
    Cm = copy_of(Cold)
    old_mults = Cm.get_n_block_multiplications() if not Cm.empty() else 0
    if spamm is None:
        nm, nr = HBSM.multiply_accumulate(A, tA, B, tB, Cm, alpha, beta)
    else:
        nm, nr = HBSM.spamm_accumulate(A, tA, B, tB, Cm, alpha, beta, spamm, updated)
    assert_bitwise(Cm, want)
    assert nm == len(P.export_tasks())
    assert nr == Cm.get_n_blocks()
    assert Cm.get_n_block_multiplications() == nm + (old_mults if beta != 0.0 else 0)
    assert np.array_equal(Cm.export_tasks(), P.export_tasks())
    assert Cm.task_checksum() == P.task_checksum()
    return Cm, P
