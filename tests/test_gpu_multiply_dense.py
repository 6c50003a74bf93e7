"""-m gpu: Y = alpha*op(A)*X + beta*Y (hbsm_multiply_dense / _device) and the Lanczos spectral-norm estimate
(hbsm_spectral_norm) against numpy on A.to_dense(), plus the C++ drop-in's multiply_dense / spectral_norm_estimate."""
import ctypes as C
import math
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
TOL = {np.float64: 1e-12, np.float32: 1e-5}
OPS = ["N", "T", "SYM_UPPER"]


@pytest.fixture(scope="module", autouse=True)
def engine():
    hb.init(0)


def make(dtype, b, M, N, r, c, v):
    A = HM(dtype, b)
    A.resize(M, N)
    keep = (r < M) & (c < N)
    A.assign_from_vectors(r[keep], c[keep], v[keep])
    return A


def op_dense(D, op):
    D = D.astype(np.float64)
    if op == "N":
        return D
    if op == "T":
        return D.T
    return np.triu(D) + np.triu(D, 1).T


_CACHE = {}


def matrix(dtype, b, kind, sym):
    """The matrix of the product tests (cached): M = 7b+5, N = 5b+3 (square 7b+5 for SYM_UPPER)."""
    key = (dtype, b, kind, sym)
    if key not in _CACHE:
        M = 7 * b + 5
        N = M if sym else 5 * b + 3
        n = max(M, N)
        if kind == "random":
            r, c, v = G.random_block_sparse_coo(n, b, 0.3, 11 + b, dtype)
            A = make(dtype, b, M, N, r, c, v)
        else:
            lam = 8.0 / b
            W = min(G.decay_width(lam), n - 1)
            r, c, v = G.decay_coo(n, lam, W, 5 + b, symmetric=sym, dtype=dtype)
            A = make(dtype, b, M, N, r, c, v)
            if sym:   # symmetric law, stored as its upper triangle
                U = HM(dtype, b)
                A.get_upper_triangle(U)
                A = U
        _CACHE[key] = A
    return _CACHE[key]


def check_cols(Y, ref, dtype):
    Y = np.asarray(Y, np.float64).reshape(ref.shape)
    assert np.all(np.isfinite(Y))
    for j in range(ref.shape[1]):
        den = np.linalg.norm(ref[:, j])
        err = np.linalg.norm(Y[:, j] - ref[:, j]) / (den if den > 0 else 1.0)
        assert err <= TOL[dtype], (j, err)


@pytest.mark.parametrize("kind", ["random", "decay"])
@pytest.mark.parametrize("m", [1, 5, 8, 12, 33])   # column chunks MC = 8, 16 and 32
@pytest.mark.parametrize("b", [7, 32, 64, 80, 128, 200, 256])   # 80 .. 256: tiles streamed in K-chunks
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_product_against_dense(dtype, op, b, m, kind):
    A = matrix(dtype, b, kind, op == "SYM_UPPER")
    opD = op_dense(A.to_dense(), op)
    Mo, K = opD.shape
    rng = np.random.default_rng(b * 100 + m)
    X = rng.standard_normal((K, m)).astype(dtype)
    if m == 1:
        X = X[:, 0]   # the 1-D path
    X64 = X.astype(np.float64).reshape(K, m)
    for beta in (0.0, 1.0, 0.5):
        Y0 = rng.standard_normal((Mo, m)).astype(dtype)
        Y = np.asfortranarray(np.full_like(Y0, np.nan) if beta == 0.0 else Y0)
        if m == 1:
            Y = Y[:, 0].copy()
        out = A.multiply_dense(X, op=op, alpha=-2.0, beta=beta, Y=Y)
        assert out is Y
        ref = -2.0 * (opD @ X64) + (beta * Y0.astype(np.float64) if beta != 0.0 else 0.0)
        check_cols(out, ref, dtype)


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_leading_dimension_padding_is_never_touched(dtype, op):
    A = matrix(dtype, 32, "decay", op == "SYM_UPPER")
    opD = op_dense(A.to_dense(), op)
    Mo, K = opD.shape
    m = 5
    rng = np.random.default_rng(3)
    X = rng.standard_normal((K, m)).astype(dtype)
    Xbig = np.full((K + 3, m), 1e30, dtype, order="F")   # a read of the padding would show in the result
    Xbig[:K] = X
    Y0 = rng.standard_normal((Mo, m)).astype(dtype)
    Ybig = np.full((Mo + 5, m), 12345.0, dtype, order="F")
    Ybig[:Mo] = Y0
    A.multiply_dense(Xbig[:K], op=op, alpha=1.5, beta=0.5, Y=Ybig[:Mo])
    assert np.all(Ybig[Mo:] == 12345.0)
    check_cols(Ybig[:Mo], 1.5 * opD @ X.astype(np.float64) + 0.5 * Y0.astype(np.float64), dtype)


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_empty_block_rows_and_tileless_and_single_leaf(dtype, op):
    b, n = 16, 6 * 16
    rng = np.random.default_rng(4)
    # tiles only in block rows 0 and 3 (and, by symmetry of the pattern, block columns 0 and 3)
    rr, cc, vv = [], [], []
    for bi, bj in [(0, 0), (0, 3), (3, 3), (0, 5), (3, 4)]:
        i, j = np.meshgrid(np.arange(b), np.arange(b), indexing="ij")
        rr.append((bi * b + i).ravel()); cc.append((bj * b + j).ravel()); vv.append(rng.standard_normal(b * b))
    A = make(dtype, b, n, n, np.concatenate(rr), np.concatenate(cc), np.concatenate(vv).astype(dtype))
    opD = op_dense(A.to_dense(), op)
    X = rng.standard_normal((n, 3)).astype(dtype)
    Y0 = rng.standard_normal((n, 3)).astype(dtype)
    Y = A.multiply_dense(X, op=op, alpha=1.0, beta=0.5, Y=np.asfortranarray(Y0.copy()))
    check_cols(Y, opD @ X.astype(np.float64) + 0.5 * Y0.astype(np.float64), dtype)
    # a sized matrix without tiles: Y = beta * Y, and beta = 0 gives zeros even over NaN
    E = HM(dtype, b)
    E.resize(n, n)
    assert E.get_n_blocks() == 0
    Y = E.multiply_dense(X, op=op, beta=0.5, Y=np.asfortranarray(Y0.copy()))
    assert np.array_equal(Y, (np.float64(0.5) * Y0.astype(np.float64)).astype(dtype))
    Y = E.multiply_dense(X, op=op, beta=0.0, Y=np.full((n, 3), np.nan, dtype, order="F"))
    assert np.array_equal(Y, np.zeros((n, 3), dtype))
    # a single leaf (M, N <= b)
    Mi, Ni = (13, 13) if op == "SYM_UPPER" else (13, 9)
    i, j = np.meshgrid(np.arange(Mi), np.arange(Ni), indexing="ij")
    S = make(dtype, b, Mi, Ni, i.ravel().astype(np.int32), j.ravel().astype(np.int32),
             rng.standard_normal(Mi * Ni).astype(dtype))
    opS = op_dense(S.to_dense(), op)
    Xs = rng.standard_normal((opS.shape[1], 2)).astype(dtype)
    check_cols(S.multiply_dense(Xs, op=op), opS @ Xs.astype(np.float64), dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_two_calls_are_bitwise_equal(dtype):
    for op in OPS:
        for b in (7, 64, 256):
            A = matrix(dtype, b, "decay", op == "SYM_UPPER")
            K = A.get_n_rows() if op == "T" else A.get_n_cols()
            X = np.random.default_rng(9).standard_normal((K, 8)).astype(dtype)
            assert np.array_equal(A.multiply_dense(X, op=op), A.multiply_dense(X, op=op)), (op, b)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_sym_upper_of_triu_matches_full_and_ignores_lower_tiles(dtype):
    b, n = 32, 7 * 32 + 5
    W = min(G.decay_width(0.1), n - 1)
    r, c, v = G.decay_coo(n, 0.1, W, 21, symmetric=True, dtype=dtype)
    S = make(dtype, b, n, n, r, c, v)
    U = HM(dtype, b)
    S.get_upper_triangle(U)
    X = np.random.default_rng(2).standard_normal((n, 8)).astype(dtype)
    y_sym = U.multiply_dense(X, op="SYM_UPPER")
    y_full = S.multiply_dense(X, op="N")
    check_cols(y_sym, y_full.astype(np.float64), dtype)
    # S has the lower tiles and the lower halves of the diagonal tiles: SYM_UPPER must not see them
    assert np.array_equal(S.multiply_dense(X, op="SYM_UPPER"), y_sym)


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_device_path_on_a_side_stream_equals_host_path(dtype, op):
    import torch
    A = matrix(dtype, 64, "random", op == "SYM_UPPER")
    opD = op_dense(A.to_dense(), op)
    Mo, K = opD.shape
    rng = np.random.default_rng(12)
    X = np.asfortranarray(rng.standard_normal((K, 8)).astype(dtype))
    Y0 = np.asfortranarray(rng.standard_normal((Mo, 8)).astype(dtype))
    y_host = A.multiply_dense(X, op=op, alpha=0.75, beta=0.5, Y=Y0.copy(order="F"))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        Xt = torch.from_numpy(np.ascontiguousarray(X.T)).cuda().t()          # column-major view, stride (1, K)
        Yt = torch.from_numpy(np.ascontiguousarray(Y0.T)).cuda().t()
        out = A.multiply_dense(Xt, op=op, alpha=0.75, beta=0.5, Y=Yt)
        assert out is Yt
        y_dev = Yt.cpu().numpy()   # ordered on s
        v = A.multiply_dense(Xt[:, 0], op=op)                                 # 1-D, Y allocated
        v_host = A.multiply_dense(X[:, 0], op=op)
        assert np.array_equal(v.cpu().numpy(), v_host)
    s.synchronize()
    assert np.array_equal(y_dev, y_host)
    with pytest.raises(ValueError):   # a row-major CUDA matrix is refused, not copied
        A.multiply_dense(torch.zeros((K, 8), dtype=Xt.dtype, device="cuda"), op=op)


def test_every_argument_error_raises_before_any_launch():
    L = _capi.lib()
    A = matrix(np.float64, 32, "random", False)   # 229 x 163
    S = matrix(np.float64, 32, "random", True)    # 229 x 229
    X = np.zeros((400, 4)); Y = np.zeros((400, 4))
    x, y = X.ctypes.data_as(C.c_void_p), Y.ctypes.data_as(C.c_void_p)
    unsized = HM(np.float64, 32)
    big = HM(np.float64, 300)   # leaf sizes above 256 have no kernel
    big.resize(10, 10)
    cases = [
        (None, 0, 1, x, 163, y, 229),
        (unsized._h, 0, 1, x, 1, y, 1),
        (A._h, 3, 1, x, 163, y, 229),
        (A._h, -1, 1, x, 163, y, 229),
        (A._h, 0, -1, x, 163, y, 229),
        (A._h, 0, 2, x, 162, y, 229),
        (A._h, 0, 2, x, 163, y, 228),
        (A._h, 1, 2, x, 228, y, 163),
        (A._h, 1, 2, x, 229, y, 162),
        (A._h, 2, 1, x, 229, y, 229),      # SYM_UPPER of a non-square A
        (big._h, 0, 1, x, 10, y, 10),
    ]
    for args in cases:
        l0 = hb.kernel_launch_count()
        with pytest.raises(hb.HbsmError) as e:
            _capi.check(L.hbsm_multiply_dense(*args, 1.0, 0.0))
        assert e.value.code == _capi.HBSM_E_ARG, args
        with pytest.raises(hb.HbsmError) as e:
            _capi.check(L.hbsm_multiply_dense_device(*args, 1.0, 0.0, None))
        assert e.value.code == _capi.HBSM_E_ARG, args
        assert hb.kernel_launch_count() == l0, args
    assert L.hbsm_multiply_dense(S._h, 2, 0, x, 229, y, 229, 1.0, 0.0) == 0   # m == 0: a no-op
    for h, sym, it, tol in [(None, 0, 10, 1e-8), (unsized._h, 0, 10, 1e-8), (A._h, 1, 10, 1e-8), (S._h, 0, 0, 1e-8),
                            (S._h, 1, 10, 0.0), (S._h, 1, 10, -1.0), (big._h, 0, 10, 1e-8)]:
        d = C.c_double(); i = C.c_int()
        l0 = hb.kernel_launch_count()
        with pytest.raises(hb.HbsmError) as e:
            _capi.check(L.hbsm_spectral_norm(h, sym, it, tol, C.byref(d), None, None, C.byref(i)))
        assert e.value.code == _capi.HBSM_E_ARG, (sym, it, tol)
        assert hb.kernel_launch_count() == l0


# ---- spectral norm ----
def random_matrix(dtype, n=1000, b=32):
    r, c, v = G.random_block_sparse_coo(n, b, 0.3, 17, dtype)
    return make(dtype, b, n, n, r, c, v)


@pytest.mark.parametrize("dtype,rel_tol,tol", [(np.float64, 1e-10, 1e-9), (np.float32, 1e-6, 1e-4)], ids=["f64", "f32"])
def test_spectral_norm_of_random_block_sparse(dtype, rel_tol, tol):
    A = random_matrix(dtype)
    ref = np.linalg.norm(A.to_dense().astype(np.float64), 2)
    nrm, lo, hi, it = A.spectral_norm_estimate(max_iter=400, rel_tol=rel_tol)
    assert lo <= hi and abs(math.sqrt(hi) - nrm) <= 1e-12 * nrm   # extreme Ritz values of A^T A
    assert 1 <= it <= 400
    assert abs(nrm - ref) / ref <= tol, (nrm, ref, it)
    assert A.spectral_norm_estimate(max_iter=400, rel_tol=rel_tol) == (nrm, lo, hi, it)   # bitwise repeatable
    nrm5, _, _, it5 = A.spectral_norm_estimate(max_iter=5, rel_tol=rel_tol)
    assert it5 <= 5 and nrm5 <= ref * (1 + tol)   # Ritz values never exceed the extreme eigenvalue


@pytest.mark.parametrize("dtype,rel_tol,tol", [(np.float64, 1e-10, 1e-9), (np.float32, 1e-6, 1e-4)], ids=["f64", "f32"])
def test_spectral_bounds_of_symmetric_decay(dtype, rel_tol, tol):
    n, b, lam = 4096, 64, 0.05
    W = min(G.decay_width(lam), n - 1)
    r, c, v = G.decay_coo(n, lam, W, 8, symmetric=True, dtype=dtype)
    S = make(dtype, b, n, n, r, c, v)
    U = HM(dtype, b)
    S.get_upper_triangle(U)
    ev = np.linalg.eigvalsh(S.to_dense().astype(np.float64))
    scale = np.abs(ev).max()
    nrm, lo, hi, it = U.spectral_norm_estimate(symmetric_upper=True, max_iter=1000, rel_tol=rel_tol)
    assert 1 <= it <= 1000
    assert abs(hi - ev[-1]) <= tol * scale, (hi, ev[-1], it)
    assert abs(lo - ev[0]) <= tol * scale, (lo, ev[0], it)
    assert abs(nrm - scale) <= tol * scale
    assert U.spectral_norm_estimate(symmetric_upper=True, max_iter=1000, rel_tol=rel_tol) == (nrm, lo, hi, it)


@pytest.mark.parametrize("b", [80, 200])   # leaf sizes whose tiles stream in K-chunks
@pytest.mark.parametrize("dtype,rel_tol,tol", [(np.float64, 1e-10, 1e-9), (np.float32, 1e-6, 1e-4)], ids=["f64", "f32"])
def test_spectral_estimates_at_chunked_leaf_sizes(dtype, rel_tol, tol, b):
    n, lam = 1000, 0.05
    W = min(G.decay_width(lam), n - 1)
    r, c, v = G.decay_coo(n, lam, W, 3, symmetric=True, dtype=dtype)
    S = make(dtype, b, n, n, r, c, v)
    U = HM(dtype, b)
    S.get_upper_triangle(U)
    D = S.to_dense().astype(np.float64)
    ev = np.linalg.eigvalsh(D)
    scale = np.abs(ev).max()
    nrm, lo, hi, it = U.spectral_norm_estimate(symmetric_upper=True, max_iter=1000, rel_tol=rel_tol)
    assert abs(hi - ev[-1]) <= tol * scale and abs(lo - ev[0]) <= tol * scale, (lo, hi, ev[0], ev[-1], it)
    nrm, _, _, it = S.spectral_norm_estimate(max_iter=1000, rel_tol=rel_tol)
    assert abs(nrm - scale) <= tol * scale, (nrm, scale, it)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_spectral_norm_of_zero_rank_one_and_one_by_one(dtype):
    tol = 1e-12 if dtype == np.float64 else 1e-5
    E = HM(dtype, 32)
    E.resize(300, 200)
    assert E.spectral_norm_estimate() == (0.0, 0.0, 0.0, 0)
    Z = make(dtype, 32, 300, 200, np.arange(100, dtype=np.int32), np.arange(100, dtype=np.int32), np.zeros(100, dtype))
    nrm, _, _, it = Z.spectral_norm_estimate()
    assert nrm == 0.0 and it <= 1
    rng = np.random.default_rng(6)
    u = rng.standard_normal(300); w = rng.standard_normal(200)
    i, j = np.meshgrid(np.arange(300), np.arange(200), indexing="ij")
    R = make(dtype, 32, 300, 200, i.ravel().astype(np.int32), j.ravel().astype(np.int32), np.outer(u, w).ravel().astype(dtype))
    ref = np.linalg.norm(R.to_dense().astype(np.float64), 2)
    nrm, _, _, it = R.spectral_norm_estimate(rel_tol=1e-8)
    assert abs(nrm - ref) <= tol * ref and it <= 3, (nrm, ref, it)
    i, j = np.meshgrid(np.arange(300), np.arange(300), indexing="ij")
    Sr = make(dtype, 32, 300, 300, i.ravel().astype(np.int32), j.ravel().astype(np.int32), np.outer(u, u).ravel().astype(dtype))
    lam = float(np.dot(u.astype(dtype).astype(np.float64), u.astype(dtype).astype(np.float64)))
    nrm, lo, hi, it = Sr.spectral_norm_estimate(symmetric_upper=True, rel_tol=1e-8)
    assert abs(hi - lam) <= tol * lam and abs(lo) <= tol * lam and it <= 3, (hi, lo, lam, it)
    One = make(dtype, 4, 1, 1, np.array([0], np.int32), np.array([0], np.int32), np.array([-3.0], dtype))
    nrm, _, _, it = One.spectral_norm_estimate()
    assert abs(nrm - 3.0) <= 3.0 * tol and it == 1
    nrm, lo, hi, it = One.spectral_norm_estimate(symmetric_upper=True)
    assert abs(nrm - 3.0) <= 3.0 * tol and abs(lo + 3.0) <= 3.0 * tol and lo == hi and it == 1


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
    const int n = 20;
    A.resize(n, n);
    std::vector<int> r, c; std::vector<double> v;
    for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) if (std::abs(i - j) <= 2) { r.push_back(i); c.push_back(j); v.push_back(1.0 + i + 0.5 * j); }
    A.assign_from_vectors(r, c, v);
    std::vector<double> X(n, 1.0), Y(n, 0.0), ref(n, 0.0);
    for (size_t t = 0; t < v.size(); ++t) ref[r[t]] += v[t];
    M::multiply_dense(A, HBSM_OP_N, 1, X.data(), n, Y.data(), n, 1.0, 0.0);
    for (int i = 0; i < n; ++i) if (std::fabs(Y[i] - ref[i]) > 1e-12 * std::fabs(ref[i])) { std::printf("row %d: %g vs %g\n", i, Y[i], ref[i]); return 1; }
    int it = 0; double lo = 0, hi = 0;
    const double s = A.spectral_norm_estimate(false, 100, 1e-10, &it);
    M U; U.set_params(p);
    A.get_upper_triangle(U);
    const double s2 = U.spectral_norm_estimate(true, 100, 1e-10, &it, &lo, &hi);
    if (!(s > 0) || !(s2 > 0) || it < 1 || it > 100 || hi < lo) { std::printf("bad estimates %g %g %d\n", s, s2, it); return 1; }
    bool threw = false;
    try { A.spectral_norm(); } catch (std::runtime_error& e) { threw = true; }
    if (!threw) { std::printf("spectral_norm() did not throw\n"); return 1; }
    std::printf("cpp dense ok %.6f %.6f\n", s, s2);
    return 0;
}
"""


def test_cpp_dropin_multiply_dense_and_spectral_norm_estimate():
    libdir = os.path.join(ROOT, "hierarchical_block_sparse_lib_b200", "lib")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "t.cc"), os.path.join(d, "t")
        open(src, "w").write(CPP)
        r = subprocess.run(["/usr/bin/g++", "-std=c++11", "-Wall", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                            "-L", libdir, "-lhbsm_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "cpp dense ok" in r.stdout
