"""-m gpu: SpAMM with error control (hbsm_spamm_error_bounds / hbsm_spamm_tau_for_error) against a numpy reference of the
bound built from export_leaves / hbsm_leaf_norms, against the products hbsm_spamm and hbsm_symm_square_spamm run at the
chosen tau, and against the a-priori estimator hbsm_spamm_errors; plus the C++ drop-in's two statics."""
import ctypes as C
import os
import subprocess
import tempfile
from collections import defaultdict

import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import _capi
from hierarchical_block_sparse_lib_b200 import generators as G
from helpers import commit_halo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HM = hb.HierarchicalBlockSparseMatrix
DTYPES = [np.float64, np.float32]
U = {np.float64: 2.0 ** -53, np.float32: 2.0 ** -24}
GEMM_TOL = {np.float64: 1e-12, np.float32: 1e-5}   # executed leaf GEMMs, relative to ||A||_F ||B||_F (DESIGN section 4)


@pytest.fixture(scope="module", autouse=True)
def engine():
    hb.init(0)


def leaf_norms(A):
    n = C.c_size_t(0)
    _capi.check(_capi.lib().hbsm_leaf_norms(A._h, 0, None, C.byref(n)))
    out = np.zeros(n.value, A.dtype)
    if n.value:
        _capi.check(_capi.lib().hbsm_leaf_norms(A._h, n.value, out.ctypes.data_as(C.c_void_p), C.byref(n)))
    return out


def random_tiles(dtype, b, n, seed, upper=False, density=0.4):
    """~40 % of the tiles, entries U[-1,1) times a per-tile scale 10^-U(0,8), three zero tiles; zero outside n x n"""
    rng = np.random.default_rng(seed)
    g = -(-n // b)
    bi, bj = np.meshgrid(np.arange(g), np.arange(g), indexing="ij")
    bi, bj = bi.ravel(), bj.ravel()
    keep = rng.random(len(bi)) < density
    if upper:
        keep &= bi <= bj
    bi, bj = bi[keep], bj[keep]
    t = rng.uniform(-1, 1, (len(bi), b, b)) * (10.0 ** -rng.uniform(0, 8, len(bi)))[:, None, None]
    t[rng.choice(len(bi), min(3, len(bi)), replace=False)] = 0.0
    r = np.arange(b)
    for k in range(len(bi)):   # t[k] is (col, row): column-major tile
        t[k][:, bi[k] * b + r >= n] = 0.0
        t[k][bj[k] * b + r >= n, :] = 0.0
    A = HM(dtype, b)
    A.resize(n, n)
    A.assign_tiles(bi, bj, t.reshape(len(bi), b * b).astype(dtype))
    A.update_internal_info()
    return A


def decay(dtype, b, n, seed, sym=False):
    lam = 8.0 / b
    W = min(G.decay_width(lam), n - 1)
    r, c, v = G.decay_coo(n, lam, W, seed, symmetric=sym, dtype=dtype)
    A = HM(dtype, b)
    A.resize(n, n)
    A.assign_from_vectors(r, c, v)
    if sym:
        U_ = HM(dtype, b)
        A.get_upper_triangle(U_)
        A = U_
    A.update_internal_info()
    return A


def make(dtype, b, kind, seed, n=None):
    n = n or 7 * b + 5
    return random_tiles(dtype, b, n, seed) if kind == "random" else decay(dtype, b, n, seed)


# ---------------------------------------------------------------------------------------------------
# numpy reference of the bound
# ---------------------------------------------------------------------------------------------------
class Ref:
    """The candidates of op(A)*op(B) (C tiles with ci <= cj only when upper), their levels p = fl(nA*nB) in the dtype and
    s = sqrt(nA) sqrt(nB) / (1 - gamma) in float64; `extra_b` = (bi, bj, norms) of committed halo tiles of B"""

    def __init__(self, A, tA, B, tB, updated=True, upper=False, w=1.0, extra_b=None):
        self.dtype = A.dtype
        b = A.get_params().blocksize
        abi, abj, an, _ = A.export_leaves(tiles=False)
        bbi, bbj, bn, _ = B.export_leaves(tiles=False)
        if not updated:
            an, bn = leaf_norms(A), leaf_norms(B)
        if extra_b is not None:
            bbi, bbj, bn = (np.concatenate([x, np.asarray(y, x.dtype)]) for x, y in zip((bbi, bbj, bn), extra_b))
        ai, ak = (abj, abi) if tA else (abi, abj)
        bk, bj = (bbj, bbi) if tB else (bbi, bbj)
        rows = defaultdict(list)
        for t, k in enumerate(bk):
            rows[int(k)].append(t)
        ci, cj, kk, na, nb = [], [], [], [], []
        for t, (i, k) in enumerate(zip(ai, ak)):
            for u in rows.get(int(k), []):
                if upper and i > bj[u]:
                    continue
                ci.append(int(i)); cj.append(int(bj[u])); kk.append(int(k)); na.append(an[t]); nb.append(bn[u])
        self.ci, self.cj, self.k = np.array(ci, np.int64), np.array(cj, np.int64), np.array(kk, np.int64)
        na, nb = np.array(na, self.dtype), np.array(nb, self.dtype)
        self.p = na * nb
        nu = b * b * U[self.dtype.type]
        self.s = np.sqrt(na.astype(np.float64)) * np.sqrt(nb.astype(np.float64)) / (1.0 - nu / (1.0 - nu))
        self.tile = self.ci * (1 << 21) + self.cj
        self.w = w
        self.q = len(self.p)

    def tau2(self, tau):
        t = self.dtype.type(tau)
        return t * t

    def skipped(self, tau):
        with np.errstate(invalid="ignore"):
            return ~(self.p > self.tau2(tau))

    def bound(self, tau):
        sk = self.skipped(tau)
        if not sk.any():
            return 0.0
        _, inv = np.unique(self.tile[sk], return_inverse=True)
        S = np.bincount(inv, weights=self.s[sk])
        return float(np.sqrt(self.w * np.sum(S * S)))

    def bound_at_level(self, v):
        sk = self.p <= v
        if not sk.any():
            return 0.0
        _, inv = np.unique(self.tile[sk], return_inverse=True)
        S = np.bincount(inv, weights=self.s[sk])
        return float(np.sqrt(self.w * np.sum(S * S)))

    def levels(self):
        return np.unique(self.p)

    def executed(self, tau):
        keep = ~self.skipped(tau)
        return sort_tasks(np.stack([self.ci[keep], self.cj[keep], self.k[keep]], 1))


def sort_tasks(t):
    t = np.asarray(t, np.int64).reshape(-1, 3)
    return t[np.lexsort((t[:, 2], t[:, 1], t[:, 0]))]


def taus_for(ref):
    """0, every level exactly (as a tau), values between levels, above the top level"""
    lv = ref.levels().astype(np.float64)
    lv = lv[np.isfinite(lv)]
    pick = lv[np.linspace(0, len(lv) - 1, min(len(lv), 12)).astype(int)] if len(lv) else lv
    taus = [0.0] + [float(np.sqrt(v)) for v in pick]
    taus += [float(np.sqrt(np.sqrt(a * c))) for a, c in zip(lv[:-1:max(1, len(lv) // 8)], lv[1::max(1, len(lv) // 8)])]
    if len(lv):
        taus.append(float(np.sqrt(lv[-1])) * 2.0)
    return sorted(taus)


def hits(dtype, v, v_next):
    """is there a tau >= 0 with v <= fl(tau*tau) < v_next in the dtype?  fl(t*t) is non-decreasing in t, so the smallest t
    with fl(t*t) >= v decides"""
    T = np.dtype(dtype).type
    v = T(v)
    t = T(np.sqrt(np.float64(v)))
    while t > 0 and np.nextafter(t, T(0)) * np.nextafter(t, T(0)) >= v:
        t = np.nextafter(t, T(0))
    while t * t < v:
        t = np.nextafter(t, T(np.inf))
    return v_next is None or t * t < T(v_next)


# ---------------------------------------------------------------------------------------------------
# 1. bounds against numpy
# ---------------------------------------------------------------------------------------------------
CASES = [(d, b, k) for d in DTYPES for b in (7, 32, 64, 80) for k in ("random", "decay")]
IDS = ["%s-b%d-%s" % ("f64" if d == np.float64 else "f32", b, k) for d, b, k in CASES]


@pytest.mark.parametrize("dtype,b,kind", CASES, ids=IDS)
def test_bounds_match_numpy(dtype, b, kind):
    A = make(dtype, b, kind, 11 + b)
    B = make(dtype, b, kind, 12 + b)
    for tA in (0, 1):
        for tB in (0, 1):
            ref = Ref(A, tA, B, tB)
            taus = taus_for(ref)
            bounds, ns = HM.spamm_error_bounds(A, tA, B, tB, taus)
            exp = np.array([ref.bound(t) for t in taus])
            nexp = np.array([int(ref.skipped(t).sum()) for t in taus])
            assert np.array_equal(ns, nexp), (tA, tB)
            assert np.all(np.abs(bounds - exp) <= 1e-12 * exp), (tA, tB, bounds, exp)
            assert np.all(np.diff(bounds) >= 0)
            assert ns[-1] == ref.q and ns[0] == int((ref.p <= 0).sum())


# ---------------------------------------------------------------------------------------------------
# 2. the chosen tau does what it says
# ---------------------------------------------------------------------------------------------------
def check_choice(ref, info, eps, tasks, nm):
    dtype = ref.dtype
    v = info["level"]
    assert info["n_candidates"] == ref.q and info["n_levels"] == len(ref.levels())
    sk = ref.skipped(info["tau"])
    assert np.array_equal(sk, ref.p <= v) if v >= 0 else not sk.any()
    assert info["n_skipped"] == int(sk.sum()) and nm == ref.q - info["n_skipped"]
    assert np.array_equal(sort_tasks(tasks), ref.executed(info["tau"]))
    assert info["bound"] <= eps
    assert abs(info["bound"] - ref.bound(info["tau"])) <= 1e-12 * info["bound"]
    lv = ref.levels()
    above = lv[lv > v] if v >= 0 else lv
    if len(above):   # maximality: the next level is over budget, or no tau singles it out (and so on upwards)
        j = 0
        while ref.bound_at_level(above[j]) <= eps * (1 - 1e-12):   # (a level at the budget's edge counts as over it)
            assert not hits(dtype, above[j], above[j + 1] if j + 1 < len(above) else None), (v, above[j], eps)
            j += 1
            if j == len(above):
                break


def measured_error(A, tA, B, tB, Cm):
    Da = A.to_dense().astype(np.float64)
    Db = B.to_dense().astype(np.float64)
    P = (Da.T if tA else Da) @ (Db.T if tB else Db)
    return float(np.linalg.norm(P - Cm.to_dense().astype(np.float64))), float(np.linalg.norm(Da) * np.linalg.norm(Db))


@pytest.mark.parametrize("dtype,b,kind", [c for c in CASES if c[1] in (7, 32, 64)], ids=[i for c, i in zip(CASES, IDS) if c[1] in (7, 32, 64)])
def test_chosen_tau_does_what_it_says(dtype, b, kind):
    A = make(dtype, b, kind, 21 + b)
    B = make(dtype, b, kind, 22 + b)
    for tA, tB in ((0, 0), (1, 0), (0, 1)):
        ref = Ref(A, tA, B, tB)
        scale = float(np.linalg.norm(A.to_dense().astype(np.float64)) * np.linalg.norm(B.to_dense().astype(np.float64)))
        for rel in (0.0, 1e-12, 1e-8, 1e-5, 1e-3, 1e-1, 10.0):
            eps = rel * scale
            info = HM.spamm_tau_for_error(A, tA, B, tB, eps)
            Cm = HM(dtype)
            nm, _ = HM.spamm(A, tA, B, tB, Cm, info["tau"], True)
            check_choice(ref, info, eps, Cm.export_tasks(), nm)
            err, ab = measured_error(A, tA, B, tB, Cm)
            assert err <= info["bound"] + GEMM_TOL[dtype] * ab, (rel, err, info)
        assert info["n_skipped"] >= ref.q // 2   # eps = 10 ||A|| ||B|| skips almost everything


# ---------------------------------------------------------------------------------------------------
# 3. symm_square on upper storage
# ---------------------------------------------------------------------------------------------------
def full_symmetric(A):
    """a matrix holding sym_expand(A)'s tiles (triu(A) + striu(A)^T), norms refreshed, and that dense matrix"""
    b = A.get_params().blocksize
    n = A.get_n_rows()
    D = A.to_dense().astype(np.float64)
    F = np.triu(D) + np.triu(D, 1).T
    bi, bj, _, _ = A.export_leaves(tiles=False, norms=False)
    pos = sorted(set(zip(bi.tolist(), bj.tolist())) | set(zip(bj.tolist(), bi.tolist())))
    g = -(-n // b)
    Fp = np.zeros((g * b, g * b))
    Fp[:n, :n] = F
    ti = np.array([p[0] for p in pos]); tj = np.array([p[1] for p in pos])
    tiles = np.stack([Fp[i * b:(i + 1) * b, j * b:(j + 1) * b].T.ravel() for i, j in pos]).astype(A.dtype)
    S = HM(A.dtype, b)
    S.resize(n, n)
    S.assign_tiles(ti, tj, tiles)
    S.update_internal_info()
    return S, F


@pytest.mark.parametrize("dtype,b,kind", [(d, b, k) for d in DTYPES for b in (7, 32, 64) for k in ("random", "decay")],
                         ids=["%s-b%d-%s" % ("f64" if d == np.float64 else "f32", b, k) for d in DTYPES for b in (7, 32, 64)
                              for k in ("random", "decay")])
def test_symm_square(dtype, b, kind):
    n = 7 * b + 5
    A = random_tiles(dtype, b, n, 31 + b, upper=True) if kind == "random" else decay(dtype, b, n, 31 + b, sym=True)
    S, F = full_symmetric(A)
    ref = Ref(S, 0, S, 0, upper=True, w=2.0)
    taus = taus_for(ref)
    bounds, ns = HM.spamm_error_bounds(A, 0, A, 0, taus, symm_square=True)
    assert np.array_equal(ns, [int(ref.skipped(t).sum()) for t in taus])
    exp = np.array([ref.bound(t) for t in taus])
    assert np.all(np.abs(bounds - exp) <= 1e-12 * exp) and np.all(np.diff(bounds) >= 0)
    P = F @ F
    scale = float(np.linalg.norm(F) ** 2)
    for rel in (0.0, 1e-10, 1e-6, 1e-3, 1.0):
        eps = rel * scale
        info = HM.spamm_tau_for_error(A, 0, A, 0, eps, symm_square=True)
        Cm = HM(dtype)
        nm, _ = HM.symm_square_spamm(A, Cm, info["tau"])
        check_choice(ref, info, eps, Cm.export_tasks(), nm)
        E = np.triu(P) - Cm.to_dense().astype(np.float64)
        E = np.triu(E) + np.triu(E, 1).T
        assert float(np.linalg.norm(E)) <= info["bound"] + GEMM_TOL[dtype] * scale, (rel, info)


# ---------------------------------------------------------------------------------------------------
# 4. updated = 0
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_updated_false_uses_fresh_norms_and_leaves_the_caches(dtype):
    b = 32
    A = make(dtype, b, "random", 41)
    B = make(dtype, b, "decay", 42)
    Sa, Sb = HM(dtype), HM(dtype)   # stale caches: rescale leaves zero norms behind
    Sa.rescale(A, 2.0)
    Sb.rescale(B, 0.5)
    taus = taus_for(Ref(A, 0, B, 0))
    before = [(X.get_frob_norm_squared_internal(), X.export_leaves(tiles=False)[2].copy()) for X in (Sa, Sb)]
    b0, n0 = HM.spamm_error_bounds(Sa, 0, Sb, 1, taus, updated=False)
    i0 = HM.spamm_tau_for_error(Sa, 0, Sb, 1, 1e-6, updated=False)
    s0, m0 = HM.spamm_error_bounds(Sa, 1, Sa, 0, taus, updated=False)   # B is A
    for X, (f, nr) in zip((Sa, Sb), before):
        assert X.get_frob_norm_squared_internal() == f and np.array_equal(X.export_leaves(tiles=False)[2], nr)
    Sa.update_internal_info()
    Sb.update_internal_info()
    b1, n1 = HM.spamm_error_bounds(Sa, 0, Sb, 1, taus)
    assert np.array_equal(b0, b1) and np.array_equal(n0, n1)
    assert i0 == HM.spamm_tau_for_error(Sa, 0, Sb, 1, 1e-6)
    s1, m1 = HM.spamm_error_bounds(Sa, 1, Sa, 0, taus)
    assert np.array_equal(s0, s1) and np.array_equal(m0, m1)


# ---------------------------------------------------------------------------------------------------
# 5. tighter than the a-priori estimator
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,b", [(np.float64, 32), (np.float64, 64)], ids=["f64-b32", "f64-b64"])
def test_tighter_than_spamm_errors(dtype, b):
    """(fp64: the bound's 1/(1 - gamma) is below 1e-12 there; at fp32 it is 6e-5 at b = 32, which a C tile with a single
    skipped pair, where the two estimates coincide, would show)"""
    A = decay(dtype, b, 16 * b, 51)
    B = decay(dtype, b, 16 * b, 52)
    ref = Ref(A, 0, B, 0)
    lv = ref.levels().astype(np.float64)
    lv = lv[lv > 0]
    idx = np.linspace(0, len(lv) - 2, 10).astype(int)
    taus = [float(np.sqrt(np.sqrt(lv[i] * lv[i + 1]))) for i in idx]
    bounds, _ = HM.spamm_error_bounds(A, 0, B, 0, taus)
    old = HM.get_spamm_errors(A, 0, B, 0, taus).astype(np.float64)
    assert np.all(bounds <= old * (1 + 1e-12)), (bounds, old)
    assert np.any(bounds > 0)


# ---------------------------------------------------------------------------------------------------
# 6. edges
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_edges(dtype):
    b = 32
    A = make(dtype, b, "random", 61)   # three zero tiles
    B = make(dtype, b, "random", 62)
    ref = Ref(A, 0, B, 0)
    zero = int((ref.p == 0).sum())
    assert zero > 0
    info = HM.spamm_tau_for_error(A, 0, B, 0, 0.0)   # eps = 0 skips exactly the zero-level pairs
    assert info["tau"] == 0.0 and info["level"] == 0.0 and info["n_skipped"] == zero and info["bound"] == 0.0

    one = HM(dtype, b)   # a single-leaf product
    one.resize(20, 20)
    one.assign_from_vectors(np.arange(20, dtype=np.int32), np.arange(20, dtype=np.int32), np.linspace(1, 2, 20).astype(dtype))
    one.update_internal_info()
    r1 = Ref(one, 0, one, 0)
    bounds, ns = HM.spamm_error_bounds(one, 0, one, 0, [0.0, 1.0, 100.0])
    assert list(ns) == [0, 0, 1] and bounds[2] == pytest.approx(r1.bound(100.0), rel=1e-12) and bounds[0] == 0.0
    info = HM.spamm_tau_for_error(one, 0, one, 0, 1.01 * r1.bound(100.0))
    assert info["n_skipped"] == 1 and info["n_candidates"] == 1 and info["n_levels"] == 1

    L_ = HM(dtype, b)   # no candidates: A's tiles in block column 0, B's in block row 1
    L_.resize(4 * b, 4 * b)
    L_.assign_tiles(np.array([0, 1]), np.array([0, 0]), np.ones((2, b * b), dtype))
    L_.update_internal_info()
    R_ = HM(dtype, b)
    R_.resize(4 * b, 4 * b)
    R_.assign_tiles(np.array([1]), np.array([2]), np.ones((1, b * b), dtype))
    R_.update_internal_info()
    bounds, ns = HM.spamm_error_bounds(L_, 0, R_, 0, [0.0, 1.0])
    assert list(bounds) == [0.0, 0.0] and list(ns) == [0, 0]
    assert HM.spamm_tau_for_error(L_, 0, R_, 0, 1.0) == {"tau": 0.0, "bound": 0.0, "level": -1.0, "n_candidates": 0,
                                                         "n_skipped": 0, "n_levels": 0}

    bi, bj, _, t = A.export_leaves(norms=False)   # a NaN tile
    t = t.copy()
    t[len(t) // 2, 5] = np.nan
    N_ = HM(dtype, b)
    N_.resize(A.get_n_rows(), A.get_n_cols())
    N_.assign_tiles(bi, bj, t)
    N_.update_internal_info()
    bounds, _ = HM.spamm_error_bounds(N_, 0, B, 0, [0.0, 1e-3, 1e3])
    assert np.all(np.isposinf(bounds))
    with pytest.raises(_capi.HbsmError) as e:
        HM.spamm_tau_for_error(N_, 0, B, 0, 1.0)
    assert e.value.code == _capi.HBSM_E_ARG


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_committed_halo_takes_part(dtype):
    b = 32
    n = 8 * b
    A = random_tiles(dtype, b, n, 71)
    Bf = random_tiles(dtype, b, n, 72)
    bi, bj, nrm, t = Bf.export_leaves()
    halo = bi >= 5   # B's block rows 5.. arrive as a halo
    Bo = HM(dtype, b)
    Bo.resize(n, n)
    Bo.assign_tiles(bi[~halo], bj[~halo], t[~halo])
    Bo.update_internal_info()
    commit_halo(Bo, bi[halo], bj[halo], tiles=t[halo], norms=nrm[halo])
    ref = Ref(A, 0, Bo, 0, extra_b=(bi[halo], bj[halo], nrm[halo]))
    full = Ref(A, 0, Bf, 0)
    assert ref.q == full.q
    taus = taus_for(ref)
    bounds, ns = HM.spamm_error_bounds(A, 0, Bo, 0, taus)
    assert np.array_equal(ns, [int(ref.skipped(x).sum()) for x in taus])
    exp = np.array([ref.bound(x) for x in taus])
    assert np.all(np.abs(bounds - exp) <= 1e-12 * exp)
    eps = 1e-6 * float(np.linalg.norm(A.to_dense().astype(np.float64)) * np.linalg.norm(Bf.to_dense().astype(np.float64)))
    info = HM.spamm_tau_for_error(A, 0, Bo, 0, eps)
    Cm = HM(dtype)
    nm, _ = HM.spamm(A, 0, Bo, 0, Cm, info["tau"], True)
    check_choice(ref, info, eps, Cm.export_tasks(), nm)
    with pytest.raises(_capi.HbsmError) as e:   # updated = 0 is refused with a committed halo, as hbsm_spamm refuses it
        HM.spamm_error_bounds(A, 0, Bo, 0, [1.0], updated=False)
    assert e.value.code == _capi.HBSM_E_ARG


# ---------------------------------------------------------------------------------------------------
# 7. determinism and argument errors
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_two_calls_are_bitwise_equal(dtype):
    A = make(dtype, 64, "decay", 81, n=20 * 64)
    taus = taus_for(Ref(A, 0, A, 1))
    b1, n1 = HM.spamm_error_bounds(A, 0, A, 1, taus)
    b2, n2 = HM.spamm_error_bounds(A, 0, A, 1, taus)
    assert np.array_equal(b1.view(np.uint64), b2.view(np.uint64)) and np.array_equal(n1, n2)
    assert HM.spamm_tau_for_error(A, 0, A, 1, 1e-7) == HM.spamm_tau_for_error(A, 0, A, 1, 1e-7)


def test_every_argument_error_returns_before_any_launch():
    L = _capi.lib()
    b = 32
    A = make(np.float64, b, "random", 91)
    A32 = make(np.float32, b, "random", 92)
    A16 = make(np.float64, 16, "random", 93, n=A.get_n_rows())
    R = HM(np.float64, b)
    R.resize(100, 60)
    R.assign_tiles(np.array([0]), np.array([0]), np.ones((1, b * b)))
    unsized = HM(np.float64, b)
    H_ = make(np.float64, b, "random", 94)
    commit_halo(H_, [7], [7], seed=1)
    taus = np.array([1.0]); out = np.zeros(1); ns = np.zeros(1, np.uint64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    info = _capi.SpammTolInfo()
    refusals = [  # (A, tA, B, tB, symm_square, updated)
        (None, 0, A._h, 0, 0, 1), (A._h, 0, None, 0, 0, 1), (unsized._h, 0, A._h, 0, 0, 1), (A._h, 0, A32._h, 0, 0, 1),
        (A._h, 0, A16._h, 0, 0, 1), (A._h, 0, H_._h, 0, 0, 0), (A._h, 0, A32._h, 0, 1, 1), (A._h, 1, A._h, 0, 1, 1),
        (A._h, 0, A._h, 1, 1, 1), (R._h, 0, R._h, 0, 1, 1), (unsized._h, 0, unsized._h, 0, 1, 1)]
    for a, ta, bb, tb, sq, up in refusals:
        l0 = hb.kernel_launch_count()
        assert L.hbsm_spamm_error_bounds(a, ta, bb, tb, sq, up, 1, p(taus), p(out), p(ns)) == _capi.HBSM_E_ARG, (ta, tb, sq, up)
        assert L.hbsm_last_error()
        assert L.hbsm_spamm_tau_for_error(a, ta, bb, tb, sq, up, 1.0, C.byref(info)) == _capi.HBSM_E_ARG
        assert hb.kernel_launch_count() == l0
    for eps in (-1.0, float("nan"), float("inf")):
        l0 = hb.kernel_launch_count()
        assert L.hbsm_spamm_tau_for_error(A._h, 0, A._h, 0, 0, 1, eps, C.byref(info)) == _capi.HBSM_E_ARG
        assert hb.kernel_launch_count() == l0
    for t, o in ((None, p(out)), (p(taus), None)):
        l0 = hb.kernel_launch_count()
        assert L.hbsm_spamm_error_bounds(A._h, 0, A._h, 0, 0, 1, 1, t, o, None) == _capi.HBSM_E_ARG
        assert hb.kernel_launch_count() == l0
    # bad sizes: hbsm_spamm's own code and message
    Cm = HM(np.float64)
    rc = L.hbsm_spamm(R._h, 0, R._h, 0, Cm._h, 1.0, 1, None, None)
    msg = L.hbsm_last_error()
    l0 = hb.kernel_launch_count()
    assert L.hbsm_spamm_error_bounds(R._h, 0, R._h, 0, 0, 1, 1, p(taus), p(out), None) == rc != 0
    assert L.hbsm_last_error() == msg
    assert hb.kernel_launch_count() == l0
    assert L.hbsm_spamm_error_bounds(A._h, 0, A._h, 0, 0, 1, 0, None, None, None) == 0   # n == 0: nothing to do


# ---------------------------------------------------------------------------------------------------
# 8. the C++ statics
# ---------------------------------------------------------------------------------------------------
CPP = r"""
#include "hbsm/hierarchical_block_sparse_lib.h"
#include <cmath>
#include <cstdio>
#include <vector>
typedef hbsm::HierarchicalBlockSparseMatrix<double> M;
int main() {
    M A;
    M::Params p; p.blocksize = 8; A.set_params(p);
    const int n = 61;
    A.resize(n, n);
    std::vector<int> r, c; std::vector<double> v;
    for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) if (std::abs(i - j) <= 20) { r.push_back(i); c.push_back(j); v.push_back(std::ldexp(1.0 + i / 64.0, -std::abs(j - i))); }
    A.assign_from_vectors(r, c, v);
    A.update_internal_info();
    std::vector<double> taus(3), bounds;
    std::vector<size_t> ns;
    taus[0] = 1e-4; taus[1] = 1e-2; taus[2] = 1e-1;
    M::spamm_error_bounds(A, false, A, true, taus, bounds, ns);
    hbsm_spamm_tol_info info = M::spamm_tau_for_error(A, false, A, true, 1e-3);
    std::printf("bounds %.17g %.17g %.17g\n", bounds[0], bounds[1], bounds[2]);
    std::printf("skipped %zu %zu %zu\n", ns[0], ns[1], ns[2]);
    std::printf("tau %.17g %.17g %.17g %zu %zu %zu\n", info.tau, info.bound, info.level, info.n_candidates, info.n_skipped, info.n_levels);
    return 0;
}
"""


def test_cpp_statics_match_python():
    libdir = os.path.join(ROOT, "hierarchical_block_sparse_lib_b200", "lib")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "t.cc"), os.path.join(d, "t")
        open(src, "w").write(CPP)
        r = subprocess.run(["/usr/bin/g++", "-std=c++11", "-Wall", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                            "-L", libdir, "-lhbsm_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
    lines = dict(l.split(" ", 1) for l in r.stdout.strip().splitlines())
    n = 61
    rr, cc, vv = [], [], []
    for i in range(n):
        for j in range(n):
            if abs(i - j) <= 20:
                rr.append(i); cc.append(j); vv.append(np.ldexp(1.0 + i / 64.0, -abs(j - i)))   # exact in both languages
    A = HM(np.float64, 8)
    A.resize(n, n)
    A.assign_from_vectors(np.array(rr, np.int32), np.array(cc, np.int32), np.array(vv))
    A.update_internal_info()
    bounds, ns = HM.spamm_error_bounds(A, 0, A, 1, [1e-4, 1e-2, 1e-1])
    assert [float(x) for x in lines["bounds"].split()] == list(bounds)
    assert [int(x) for x in lines["skipped"].split()] == list(ns)
    info = HM.spamm_tau_for_error(A, 0, A, 1, 1e-3)
    got = lines["tau"].split()
    assert [float(x) for x in got[:3]] == [info["tau"], info["bound"], info["level"]]
    assert [int(x) for x in got[3:]] == [info["n_candidates"], info["n_skipped"], info["n_levels"]]
    assert 0 < info["n_skipped"] < info["n_candidates"]
