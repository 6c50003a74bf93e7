"""-m gpu: truncation with spectral-norm error control (hbsm_spectral_block_trunc) and spectral norms of truncation error
matrices (hbsm_truncation_spectral_errors) against numpy on to_dense(), against hbsm_spectral_norm on a matrix holding
exactly the dropped tiles, and against hbsm_frob_block_trunc; plus the C++ drop-in's two extras."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import _capi
from hierarchical_block_sparse_lib_b200 import generators as G

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HM = hb.HierarchicalBlockSparseMatrix
BS = [7, 32, 64, 80, 200]
DTYPES = [np.float64, np.float32]
RTOL = {np.float64: 1e-10, np.float32: 1e-6}   # Lanczos rel_tol of the full-convergence runs
TOL = {np.float64: 1e-7, np.float32: 1e-3}     # against numpy


@pytest.fixture(scope="module", autouse=True)
def engine():
    hb.init(0)


def leaf_norms(A):
    """fresh leaf ||.||_F^2 through hbsm_leaf_norms, in A's dtype"""
    n = C.c_size_t(0)
    _capi.check(_capi.lib().hbsm_leaf_norms(A._h, 0, None, C.byref(n)))
    out = np.zeros(n.value, A.dtype)
    if n.value:
        _capi.check(_capi.lib().hbsm_leaf_norms(A._h, n.value, out.ctypes.data_as(C.c_void_p), C.byref(n)))
    return out


def random_tiles(dtype, b, n, seed, upper):
    """random block-sparse: ~40 % of the tiles, entries U[-1,1) times a per-tile scale 10^-U(0,8), a few zero tiles;
    entries outside the n x n matrix are zero"""
    rng = np.random.default_rng(seed)
    g = -(-n // b)
    bi, bj = np.meshgrid(np.arange(g), np.arange(g), indexing="ij")
    bi, bj = bi.ravel(), bj.ravel()
    keep = rng.random(len(bi)) < 0.4
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
    return A


def decay(dtype, b, n, sym):
    lam = 8.0 / b
    W = min(G.decay_width(lam), n - 1)
    r, c, v = G.decay_coo(n, lam, W, 5 + b, symmetric=sym, dtype=dtype)
    A = HM(dtype, b)
    A.resize(n, n)
    A.assign_from_vectors(r, c, v)
    if not sym:
        return A
    U = HM(dtype, b)   # symmetric law, stored as its upper triangle
    A.get_upper_triangle(U)
    return U


_CACHE = {}


def matrix(dtype, b, kind, sym):
    key = (dtype, b, kind, sym)
    if key not in _CACHE:
        n = 7 * b + 5
        A = random_tiles(dtype, b, n, 100 + b, sym) if kind == "random" else decay(dtype, b, n, sym)
        _CACHE[key] = A
    return _CACHE[key]


def op_norm(D, sym):
    D = np.asarray(D, np.float64)
    if sym:
        return float(np.abs(np.linalg.eigvalsh(np.triu(D) + np.triu(D, 1).T)).max()) if D.size else 0.0
    return float(np.linalg.norm(D, 2)) if D.size else 0.0


def subset(A, mask):
    """a matrix of A's shape holding exactly A's tiles where mask"""
    bi, bj, _, t = A.export_leaves(norms=False)
    E = HM(A.dtype, A.get_params().blocksize)
    E.resize(A.get_n_rows(), A.get_n_cols())
    if mask.any():
        E.assign_tiles(bi[mask], bj[mask], t[mask])
    return E


def eligible(A, sym):
    bi, bj, _, _ = A.export_leaves(tiles=False, norms=False)
    return (bi <= bj) if sym else np.ones(len(bi), bool)


CASES = [(d, b, k, s) for d in DTYPES for b in BS for k in ("decay", "random") for s in (True, False)]
IDS = ["%s-b%d-%s-%s" % ("f64" if d == np.float64 else "f32", b, k, "sym" if s else "gen") for d, b, k, s in CASES]


@pytest.mark.parametrize("dtype,b,kind,sym", CASES, ids=IDS)
def test_masked_operator_is_bitwise_the_dropped_tiles_matrix(dtype, b, kind, sym):
    A = matrix(dtype, b, kind, sym)
    nsq = leaf_norms(A)
    levels = np.unique(nsq)
    taus = [float(np.sqrt(levels[int(q * (len(levels) - 1))])) * 1.0001 for q in (0.2, 0.5, 0.8)]
    norms, its = A.truncation_spectral_errors(taus, symmetric_upper=sym, max_iter=1000, rel_tol=RTOL[dtype])
    for tau, nrm, it in zip(taus, norms, its):
        t = np.asarray(tau, dtype)
        mask = nsq < t * t   # the frob_block_trunc rule, in the matrix's dtype
        E = subset(A, mask)
        ref = E.spectral_norm_estimate(symmetric_upper=sym, max_iter=1000, rel_tol=RTOL[dtype])
        assert nrm == ref[0] and it == ref[3], (tau, nrm, it, ref)
        exact = op_norm(E.to_dense(), sym)
        assert abs(nrm - exact) <= TOL[dtype] * max(exact, 1e-300) or (exact == 0 and nrm == 0), (tau, nrm, exact)


def check_contract(A, sym, eps, dtype, max_iter=1000):
    Cm = HM(dtype)
    info = A.spectral_block_trunc(Cm, eps, symmetric_upper=sym, max_iter=max_iter)
    nsq = leaf_norms(A)
    el = eligible(A, sym)
    v = info["drop_nsq"]
    drop = el & (nsq <= v)
    assert info["n_dropped"] == int(drop.sum())
    assert info["n_dropped"] >= info["n_frob"]
    bi, bj, _, t = A.export_leaves(norms=False)
    cbi, cbj, cn, ct = Cm.export_leaves()
    assert np.array_equal(cbi, bi[~drop]) and np.array_equal(cbj, bj[~drop])
    assert np.array_equal(ct, t[~drop])
    assert not np.any(cn)   # cached norms stale (zero), as after frob_block_trunc
    assert Cm.get_n_block_multiplications() == A.get_n_block_multiplications()
    D = subset(A, drop).to_dense()
    err = op_norm(D, sym)
    tol = TOL[dtype]
    assert err <= eps * (1 + tol) + 1e-300, (err, eps, info)
    rest = np.unique(nsq[el & ~drop])
    if len(rest):
        nxt = rest[0]
        assert op_norm(subset(A, el & (nsq <= nxt)).to_dense(), sym) >= eps * (1 - tol), (eps, info)
    # C equals frob_block_trunc between the chosen level and the next one (which also drops tiles below the diagonal)
    vv = max(float(v), 0.0)
    t2 = (vv + float(rest[0])) / 2 if len(rest) else 2 * vv + 1.0
    tau = np.sqrt(t2)
    tq = np.asarray(tau, dtype)
    if el.all() and (tq * tq > v) and (not len(rest) or tq * tq <= rest[0]):
        F = HM(dtype)
        A.frob_block_trunc(F, tau)
        fbi, fbj, fn, ft = F.export_leaves()
        assert np.array_equal(fbi, cbi) and np.array_equal(fbj, cbj) and np.array_equal(ft, ct) and np.array_equal(fn, cn)
        assert F.get_n_block_multiplications() == Cm.get_n_block_multiplications()
        assert F.get_frob_norm_squared_internal() == Cm.get_frob_norm_squared_internal()
    return info, Cm


@pytest.mark.parametrize("dtype,b,kind,sym", CASES, ids=IDS)
def test_truncation_contract(dtype, b, kind, sym):
    A = matrix(dtype, b, kind, sym)
    scale = op_norm(A.to_dense(), sym)
    rels = (1e-2, 1e-4, 1e-6) if dtype == np.float64 else (1e-2, 1e-4)
    for rel in rels:
        info, _ = check_contract(A, sym, rel * scale, dtype)
        if info["certified_by_lanczos"]:
            assert info["n_decisions"] >= 1 and info["lanczos_steps"] >= 1
            assert info["err_bound"] <= rel * scale
        else:
            assert info["n_dropped"] == info["n_frob"]


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_edges(dtype):
    b = 32
    R = matrix(dtype, b, "random", False)
    nsq = leaf_norms(R)
    info, Cm = check_contract(R, False, 0.0, dtype)   # eps = 0 drops exactly the zero-norm leaves
    assert info["n_dropped"] == int((nsq == 0).sum()) > 0 and info["drop_nsq"] == 0.0
    D = matrix(dtype, b, "decay", True)
    dn = leaf_norms(D)
    eps = 1e-3 * float(np.sqrt(dn.min() / b))
    info, Cm = check_contract(D, True, eps, dtype)   # below every level: nothing goes, C equals A
    assert info["n_dropped"] == 0 and info["drop_nsq"] == -1.0
    assert np.array_equal(Cm.export_leaves()[3], D.export_leaves()[3])
    for M, sym in ((D, True), (R, False)):   # eps >= ||op(A)||_2: everything droppable goes
        info, Cm = check_contract(M, sym, 1.05 * op_norm(M.to_dense(), sym), dtype)
        assert info["n_dropped"] == int(eligible(M, sym).sum()) and Cm.get_n_blocks() == 0
    G_ = matrix(dtype, b, "decay", False)   # symmetric_upper on a full matrix: tiles below the diagonal stay
    info, Cm = check_contract(G_, True, 1.05 * op_norm(G_.to_dense(), True), dtype)
    bi, bj, _, _ = Cm.export_leaves(tiles=False, norms=False)
    assert np.all(bi > bj) and len(bi) == int((~eligible(G_, True)).sum())
    one = HM(dtype, b)   # a single leaf is never truncated
    one.resize(20, 20)
    one.assign_from_vectors(np.arange(20, dtype=np.int32), np.arange(20, dtype=np.int32), np.full(20, 1e-9, dtype))
    Cm = HM(dtype)
    info = one.spectral_block_trunc(Cm, 1.0)
    assert info["n_dropped"] == 0 and np.array_equal(Cm.to_dense(), one.to_dense())
    assert np.array_equal(one.truncation_spectral_errors([1.0])[0], [0.0])
    sized = HM(dtype, b)   # sized, no tiles
    sized.resize(300, 300)
    Cm = HM(dtype)
    info = sized.spectral_block_trunc(Cm, 1.0, symmetric_upper=True)
    assert info["n_dropped"] == 0 and not Cm.empty() and Cm.get_n_blocks() == 0 and Cm.get_n_rows() == 300
    unsized = HM(dtype, b)
    Cm = HM(dtype, b)
    Cm.resize(100, 100)
    info = unsized.spectral_block_trunc(Cm, 1.0)
    assert info["n_dropped"] == 0 and Cm.empty()
    norms, its = unsized.truncation_spectral_errors([1.0, 2.0])
    assert list(norms) == [0.0, 0.0] and list(its) == [0, 0]


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_two_calls_are_bitwise_equal(dtype):
    A = matrix(dtype, 64, "random", True)
    eps = 1e-4 * op_norm(A.to_dense(), True)
    C1, C2 = HM(dtype), HM(dtype)
    i1 = A.spectral_block_trunc(C1, eps, symmetric_upper=True)
    i2 = A.spectral_block_trunc(C2, eps, symmetric_upper=True)
    assert i1 == i2
    e1, e2 = C1.export_leaves(), C2.export_leaves()
    assert all(np.array_equal(x, y) for x, y in zip(e1, e2))
    taus = [1e-6, 1e-4, 1e-2]
    n1, t1 = A.truncation_spectral_errors(taus, symmetric_upper=True)
    n2, t2 = A.truncation_spectral_errors(taus, symmetric_upper=True)
    assert np.array_equal(n1, n2) and np.array_equal(t1, t2)


def test_every_argument_error_returns_before_any_launch():
    L = _capi.lib()
    A = matrix(np.float64, 32, "random", False)
    R = HM(np.float64, 32)
    R.resize(100, 60)
    big = HM(np.float64, 300)
    big.resize(10, 10)
    Cm = HM(np.float64)
    info = _capi.TruncInfo()
    for h, sym, eps, it, c in [(None, 0, 1.0, 10, Cm._h), (A._h, 0, -1.0, 10, Cm._h), (A._h, 0, float("nan"), 10, Cm._h),
                               (A._h, 0, 1.0, 0, Cm._h), (A._h, 0, 1.0, 10, A._h), (R._h, 1, 1.0, 10, Cm._h),
                               (big._h, 0, 1.0, 10, Cm._h)]:
        l0 = hb.kernel_launch_count()
        rc = L.hbsm_spectral_block_trunc(h, sym, eps, it, c, C.byref(info))
        assert rc == _capi.HBSM_E_ARG, (sym, eps, it)
        assert L.hbsm_last_error()
        assert hb.kernel_launch_count() == l0
    taus = np.array([1.0]); out = np.zeros(1); its = np.zeros(1, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for h, sym, n, t, it, tol, o, i in [(None, 0, 1, p(taus), 10, 1e-8, p(out), p(its)),
                                        (A._h, 0, 1, p(taus), 0, 1e-8, p(out), p(its)),
                                        (A._h, 0, 1, p(taus), 10, 0.0, p(out), p(its)),
                                        (A._h, 0, 1, p(taus), 10, -1.0, p(out), p(its)),
                                        (R._h, 1, 1, p(taus), 10, 1e-8, p(out), p(its)),
                                        (big._h, 0, 1, p(taus), 10, 1e-8, p(out), p(its)),
                                        (A._h, 0, 1, None, 10, 1e-8, p(out), p(its)),
                                        (A._h, 0, 1, p(taus), 10, 1e-8, None, p(its)),
                                        (A._h, 0, 1, p(taus), 10, 1e-8, p(out), None)]:
        l0 = hb.kernel_launch_count()
        rc = L.hbsm_truncation_spectral_errors(h, sym, n, t, it, tol, o, i)
        assert rc == _capi.HBSM_E_ARG, (sym, n, it, tol)
        assert L.hbsm_last_error()
        assert hb.kernel_launch_count() == l0
    assert L.hbsm_truncation_spectral_errors(A._h, 0, 0, None, 10, 1e-8, None, None) == 0   # n == 0: nothing to do


CPP = r"""
#include "hbsm/hierarchical_block_sparse_lib.h"
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <vector>
typedef hbsm::HierarchicalBlockSparseMatrix<double> M;
int main() {
    M A;
    M::Params p; p.blocksize = 8; A.set_params(p);
    const int n = 61;
    A.resize(n, n);
    std::vector<int> r, c; std::vector<double> v;
    for (int i = 0; i < n; ++i) for (int j = i; j < n; ++j) if (j - i <= 20) { r.push_back(i); c.push_back(j); v.push_back(std::ldexp(1.0 + i / 64.0, -(j - i))); }
    A.assign_from_vectors(r, c, v);
    std::vector<double> taus(3), out;
    taus[0] = 1e-4; taus[1] = 1e-2; taus[2] = 1e-1;
    A.get_spectral_errors_of_truncation(out, taus, true, 1000, 1e-10);
    M Cm; Cm.set_params(p);
    hbsm_trunc_info info;
    A.spectral_block_trunc(Cm, 1e-3, true, 1000, &info);
    bool threw = false;
    try { std::vector<double> o; A.get_spectral_squared_of_error_matrix(o, taus, 10, true); } catch (std::runtime_error&) { threw = true; }
    if (!threw) { std::printf("get_spectral_squared_of_error_matrix did not throw\n"); return 1; }
    std::printf("errors %.17g %.17g %.17g\n", out[0], out[1], out[2]);
    std::printf("trunc %zu %.17g %zu %d %zu\n", info.n_dropped, info.drop_nsq, info.n_frob, info.n_decisions, Cm.get_n_blocks());
    return 0;
}
"""


def test_cpp_dropin_extras_match_python():
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
        for j in range(i, min(n, i + 21)):
            rr.append(i); cc.append(j); vv.append(np.ldexp(1.0 + i / 64.0, -(j - i)))   # exact in both languages
    A = HM(np.float64, 8)
    A.resize(n, n)
    A.assign_from_vectors(np.array(rr, np.int32), np.array(cc, np.int32), np.array(vv))
    norms, _ = A.truncation_spectral_errors([1e-4, 1e-2, 1e-1], symmetric_upper=True, max_iter=1000, rel_tol=1e-10)
    assert [float(x) for x in lines["errors"].split()] == list(norms)
    Cm = HM(np.float64)
    info = A.spectral_block_trunc(Cm, 1e-3, symmetric_upper=True, max_iter=1000)
    got = lines["trunc"].split()
    assert (int(got[0]), float(got[1]), int(got[2]), int(got[3]), int(got[4])) == \
        (info["n_dropped"], info["drop_nsq"], info["n_frob"], info["n_decisions"], Cm.get_n_blocks())
    assert info["n_dropped"] > 0
