"""Inverse Cholesky factor (inv_chol, H:3110) at the engine's leaf sizes: the device leaf kernel hbsm_leaf_inv_chol, the
quadrant re-keying hbsm_extract_quadrant / hbsm_assemble_quadrants (both through the C ABI), and the C++ drop-in's block
recursion (tests/cpp/test_inv_chol.cc, one process per dtype and leaf size) against a high-precision reference.

What Z is.  For an n x n matrix A with a factorisation A = L U without pivoting and positive pivots, Z = U^-1 where U is
balanced (diag(L) = diag(U)).  The leaf recurrence computes exactly this factor: it makes column i of A Z vanish above
the diagonal, so A Z is lower triangular with diag(A Z) = 1 / diag(Z).  For symmetric positive definite A it is the
inverse Cholesky factor, Z = R^-1 with R = chol(A)^T, the unique upper-triangular Z with positive diagonal and
Z^T A Z = I.  The leaf inputs are asymmetric by rounding (as the Schur complements the recursion hands to the leaf kernel
are), so the reference factors the stored matrix as it is.

Bounds (u = 2^-53 in fp64, 2^-24 in fp32; kappa = kappa_2(A); ||.|| = max-abs entry).  Each is a random-walk estimate:
an n-term sum in precision u carries an error of about sqrt(n) u, and a triangular factor R of A amplifies it by
kappa(R) = sqrt(kappa).

  REF   ||Z - Z_ref||    <= 4 sqrt(n) sqrt(kappa) u ||Z||   Z_ref is computed in long double for fp64 results (the
                                                            recursion's up to n = 600, see rec_ref) and in float64
                                                            otherwise.
  EMUL  ||Z - Z_emul||   <= 2 sqrt(n) sqrt(kappa) u ||Z||   leaf only: Z_emul runs the kernel's own column recurrence in
                                                            the kernel's dtype and differs from it only in the order of
                                                            the A-inner-product sums.
  RESID ||Z^T A Z - I||  <= 4 sqrt(n) sqrt(kappa) u ||Z||^2 ||A||   recursion, evaluated in float64 from the exported Z.

The recursion's fp32 products are split-TF32 on the tensor cores, accurate to fp32, so u is the same there.  The unmarked
tests below check every bar on the CPU: a numpy emulation of the leaf recurrence (and of the recursion over it) passes
it, and three broken emulations fail it on the kappa ~ 2 inputs -- one projection skipped, A(k, j) read where the
recurrence reads A(j, k), and the column normalised with its un-projected norm.  Largest error / bound ratios seen on
the CPU emulations are about 0.1; the tests print the GPU's per dtype and leaf size (pytest -s).
"""
import ctypes as C
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROG = os.path.join(ROOT, "tests", "cpp", "_build", "test_inv_chol")
gpu = pytest.mark.gpu
U = {np.float64: 2.0 ** -53, np.float32: 2.0 ** -24}
DTYPES = [np.float64, np.float32]
KINDS = ["k2", "k1e2", "band", "ident"]


# ---------------------------------------------------------------------------------------------------------------------
# inputs, references, emulations (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def leaf_input(kind, n, dtype, seed):
    """n x n SPD input rounded to dtype: Q diag(d) Q^T with kappa ~ 2 or ~ 1e2, made asymmetric by a relative 16 n u (the
    level a Schur complement computed in dtype can carry); a diagonally dominant band; 3 I"""
    rng = np.random.default_rng(seed)
    if kind == "ident":
        return np.eye(n, dtype=dtype) * dtype(3)
    if kind == "band":
        A = np.zeros((n, n))
        for d in range(1, min(4, n)):
            v = rng.uniform(-0.5, 0.5, n - d) / (1 + d)
            A += np.diag(v, d) + np.diag(v, -d)
        return (A + np.diag(2 + rng.random(n))).astype(dtype)
    kappa = 2.0 if kind == "k2" else 1e2
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    d = np.geomspace(1.0, 1.0 / kappa, n)
    A = (Q * d) @ Q.T
    A = (A + A.T) / 2
    return (A * (1 + 16 * n * U[dtype] * rng.uniform(-1, 1, (n, n)))).astype(dtype)


def kappa_of(A):
    A = np.asarray(A, np.float64)
    if np.array_equal(A, A.T):
        w = np.linalg.eigvalsh(A)
        return float(w[-1] / w[0])
    return float(np.linalg.cond(A))


def inv_factor_ref(A, prec):
    """Z = U^-1 of the balanced A = L U (Doolittle without pivoting, row-oriented, in `prec`); for symmetric A, U = R"""
    a = np.array(A, dtype=prec)
    n = a.shape[0]
    for k in range(n):
        a[k + 1:, k] /= a[k, k]
        a[k + 1:, k + 1:] -= np.outer(a[k + 1:, k], a[k, k + 1:])
    Ub = np.triu(a) / np.sqrt(np.diag(a).copy())[:, None]
    Z = np.zeros((n, n), prec)
    for i in range(n - 1, -1, -1):   # U Z = I, back substitution row by row
        Z[i] = -(Ub[i, i + 1:] @ Z[i + 1:])
        Z[i, i] += 1
        Z[i] /= Ub[i, i]
    return Z


def ref_prec(dtype):
    return np.longdouble if dtype == np.float64 else np.float64


def tree_sum(p):
    """the kernel's reduction order: a shuffle tree inside each 32-lane warp, then the 8 warp sums in order"""
    v = np.zeros(256, p.dtype)
    v[:len(p)] = p
    v = v.reshape(8, 32)
    for d in (16, 8, 4, 2, 1):
        v = v[:, :d] + v[:, d:2 * d]
    s = p.dtype.type(0)
    for w in v[:, 0]:
        s += w
    return s


def emulate_leaf(A, dtype, broken=None, order="dot"):
    """the kernel's column recurrence (matrix.cu, k_leaf_inv_chol) in dtype: column i starts as e_i, loses its component
    along each finished column j < i in order (R = A(j, :) z_i * Z(j, j)), then is scaled by sqrt(1 / A(i, :) z_i).
    broken: "skip" drops the projection of the last column on column 0, "triangle" reads A(k, j) for A(j, k), "norm"
    normalises with the un-projected A(i, i)."""
    a = np.array(A, dtype)
    n = a.shape[0]
    if broken == "triangle":
        a = a.T.copy()
    dot = (lambda x, y: tree_sum(x * y)) if order == "tree" else (lambda x, y: x @ y)
    one = dtype(1)
    Z = np.zeros((n, n), dtype)
    for i in range(n):
        zi = np.zeros(n, dtype)
        zi[i] = one
        for j in range(i):
            if broken == "skip" and i == n - 1 and j == 0:
                continue
            R = dot(a[j], zi) * Z[j, j]
            zi = zi - Z[:, j] * R
        R = a[i, i] if broken == "norm" else dot(a[i], zi)
        Z[:, i] = zi * np.sqrt(one / R)
    return Z


def amax(X):
    return float(np.max(np.abs(X))) if X.size else 0.0


def ref_ratio(Z, Zref, kappa, dtype):
    """REF error / bound"""
    return amax(np.asarray(Z, np.float64) - np.asarray(Zref, np.float64)) / (4 * np.sqrt(len(Z) * kappa) * U[dtype] * amax(Zref))


def emul_ratio(Z, Ze, kappa, dtype):
    """EMUL error / bound"""
    return amax(np.asarray(Z, np.float64) - np.asarray(Ze, np.float64)) / (2 * np.sqrt(len(Z) * kappa) * U[dtype] * amax(Ze))


def resid_ratio(Z, A, kappa, dtype):
    """RESID error / bound"""
    Z = np.asarray(Z, np.float64)
    A = np.asarray(A, np.float64)
    R = Z.T @ A @ Z - np.eye(len(Z))
    return amax(R) / (4 * np.sqrt(len(Z) * kappa) * U[dtype] * amax(Z) ** 2 * amax(A))


def emulate_rec(A, b, dtype, broken=None):
    """the drop-in's inv_chol_rec on dense arrays in dtype (leaves by emulate_leaf); A is n x n, padded to its virtual size"""
    n = len(A)
    v = b
    while v < n:
        v *= 2
    Av = np.zeros((v, v), dtype)
    Av[:n, :n] = A

    def rec(A, valid):
        v = len(A)
        Z = np.zeros((v, v), dtype)
        if v == b:
            Z[:valid, :valid] = emulate_leaf(A[:valid, :valid], dtype, broken)
            return Z
        h = v // 2
        Z00 = rec(A[:h, :h], min(valid, h))
        X = -(Z00 @ (Z00.T @ A[:h, h:]))
        Z[:h, :h] = Z00
        if valid > h:
            Z11 = rec(A[h:, :h] @ X + A[h:, h:], valid - h)
            Z[h:, h:] = Z11
            Z[:h, h:] = X @ Z11
        return Z

    return rec(Av, n)[:n, :n]


def recursion_tiles(P, valid, b, hits=None):
    """the tile pattern of Z that inv_chol_rec produces from A's g x g tile pattern P (g a power of two): every product
    makes the tiles its operands' patterns reach, every leaf factor is one tile, absent quadrants take the branches of
    the header.  `hits` (a set) collects the branches taken: absent A01 / A10 / A11, valid <= half (Z11 skipped) and a
    leaf factor of a ragged valid < b."""
    hits = set() if hits is None else hits
    g = len(P)
    if g == 1:
        if valid < b:
            hits.add("ragged_leaf")
        return np.ones((1, 1), bool)
    h = g // 2
    mm = lambda X, Y: (X.astype(np.int64) @ Y.astype(np.int64)) > 0
    P00, P10, P01, P11 = P[:h, :h], P[h:, :h], P[:h, h:], P[h:, h:]
    for name, part in (("absent_A01", P01), ("absent_A10", P10), ("absent_A11", P11)):
        if not part.any():
            hits.add(name)
    if valid <= h * b:
        hits.add("valid_le_half")
    Z = np.zeros((g, g), bool)
    Z00 = recursion_tiles(P00, min(valid, h * b), b, hits)
    Z[:h, :h] = Z00
    X = mm(Z00, mm(Z00.T, P01)) if P01.any() else None
    if P10.any() and X is not None:
        Q = mm(P10, X) | P11
    elif P11.any():
        Q = P11
    else:
        Q = None
    if Q is not None and valid > h * b:
        Z11 = recursion_tiles(Q, valid - h * b, b, hits)
        Z[h:, h:] = Z11
        if X is not None:
            Z[:h, h:] = mm(X, Z11)
    return Z


def rec_input(kind, n, b, seed):
    """n x n SPD float64 inputs of the recursion: "band", a block-banded matrix whose leaves are coupled only across the
    splits between tile 2m - 1 and 2m (so A01 / A10 are absent at the lowest inner level and present above it); "bdiag",
    one SPD block per diagonal leaf (A01 / A10 absent at every level); "dense", Q diag(d) Q^T with kappa ~ 1e2"""
    rng = np.random.default_rng(seed)
    g = -(-n // b)
    if kind == "dense":
        Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
        A = (Q * np.geomspace(1.0, 1e-2, n)) @ Q.T
        return (A + A.T) / 2
    A = np.zeros((g * b, g * b))
    for t in range(g):
        S = rng.uniform(-1, 1, (b, b)) / b
        A[t * b:(t + 1) * b, t * b:(t + 1) * b] = S + S.T
        if kind == "band" and t % 2 == 1 and t + 1 < g:
            C = rng.uniform(-1, 1, (b, b)) / b
            A[t * b:(t + 1) * b, (t + 1) * b:(t + 2) * b] = C
            A[(t + 1) * b:(t + 2) * b, t * b:(t + 1) * b] = C.T
    A = A[:n, :n]
    return A + np.diag(np.abs(A).sum(axis=1) + rng.uniform(0.5, 1.5, n))   # diagonally dominant


def chol_inv_ref(A):
    """R^-1 with R = chol(A)^T, in float64 (LAPACK)"""
    import scipy.linalg as sl
    R = sl.cholesky(A, lower=False)
    return sl.solve_triangular(R, np.eye(len(A)), lower=False)


def stored(dtype):
    return np.uint64 if dtype == np.float64 else np.uint32


# ---------------------------------------------------------------------------------------------------------------------
# the bars on the CPU: the emulations pass them, broken emulations fail them
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("n", [7, 32, 100, 256])
@pytest.mark.parametrize("kind", KINDS)
def test_leaf_bars_hold_for_the_emulated_recurrence(dtype, n, kind):
    A = leaf_input(kind, n, dtype, n)
    k = kappa_of(A)
    Zr = inv_factor_ref(A, ref_prec(dtype))
    Zd = emulate_leaf(A, dtype)
    Zt = emulate_leaf(A, dtype, order="tree")   # the kernel's summation order
    assert ref_ratio(Zd, Zr, k, dtype) <= 1 and ref_ratio(Zt, Zr, k, dtype) <= 1
    assert emul_ratio(Zt, Zd, k, dtype) <= 1


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("n", [32, 100])
@pytest.mark.parametrize("kind", ["k2", "k1e2"])
@pytest.mark.parametrize("broken", ["skip", "triangle", "norm"])
def test_leaf_bars_reject_broken_recurrences(dtype, n, kind, broken):
    A = leaf_input(kind, n, dtype, n)
    k = kappa_of(A)
    Zb = emulate_leaf(A, dtype, broken)
    assert emul_ratio(Zb, emulate_leaf(A, dtype), k, dtype) > 1
    if broken != "triangle":   # reading the other triangle changes Z by the asymmetry only: EMUL's job
        assert ref_ratio(Zb, inv_factor_ref(A, ref_prec(dtype)), k, dtype) > 1


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("b", [32, 64])
@pytest.mark.parametrize("kind", ["band", "bdiag", "dense"])
def test_recursion_bars_hold_for_the_emulated_recursion(dtype, b, kind):
    for n in (b - 3, 3 * b + 5, 8 * b - 1):
        A = rec_input(kind, n, b, n + b)
        k = kappa_of(A)
        Z = emulate_rec(A.astype(dtype), b, dtype)
        assert ref_ratio(Z, rec_ref(A, dtype), k, dtype) <= 1 and resid_ratio(Z, A, k, dtype) <= 1
        g = -(-n // b)
        E = recursion_tiles(tile_pattern(A, b), n, b)
        nz = np.zeros_like(E)
        for i in range(g):
            for j in range(g):
                nz[i, j] = Z[i * b:(i + 1) * b, j * b:(j + 1) * b].any()
        assert np.array_equal(nz, E)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("broken", ["skip", "norm"])
def test_recursion_bars_reject_broken_leaves(dtype, broken):
    b, n = 32, 101
    A = rec_input("dense", n, b, 7)
    k = kappa_of(A)
    Z = emulate_rec(A.astype(dtype), b, dtype, broken)
    assert ref_ratio(Z, rec_ref(A, dtype), k, dtype) > 1 and resid_ratio(Z, A, k, dtype) > 1


def rec_ref(A, dtype):
    """the reference of a recursion result: long double for fp64 up to n = 600 (its O(n^3) cost without BLAS is about 1 s
    there and grows past a minute at n = 2047), float64 LAPACK otherwise.  Above n = 600 the fp64 bar is unchanged and
    so also holds the float64 reference's own error, of the same form: measured ratios stay below 0.1."""
    return inv_factor_ref(A, np.longdouble) if dtype == np.float64 and len(A) <= 600 else chol_inv_ref(A)


def tile_pattern(A, b):
    """A's tile pattern, padded to the virtual grid side (a power of two)"""
    g = -(-len(A) // b)
    P = np.zeros((g, g), bool)
    for i in range(g):
        for j in range(g):
            P[i, j] = A[i * b:(i + 1) * b, j * b:(j + 1) * b].any()
    return pad_pattern(P)


def pad_pattern(P):
    g = 1
    while g < len(P):
        g *= 2
    out = np.zeros((g, g), bool)
    out[:len(P), :len(P)] = P
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the leaf kernel through the C ABI (GPU)
# ---------------------------------------------------------------------------------------------------------------------
RATIOS = {}   # (part, dtype, b) -> largest error / bound seen


def note(part, dtype, b, r):
    key = (part, np.dtype(dtype).name, b)
    RATIOS[key] = max(RATIOS.get(key, 0.0), r)


@pytest.fixture(scope="module")
def engine():
    import hierarchical_block_sparse_lib_b200 as hb
    hb.init(0)
    yield hb
    if RATIOS:
        print("\nlargest error / bound per (check, dtype, leaf size):")
        for k in sorted(RATIOS):
            print("  %-6s %-8s b=%-4d %.3g" % (k + (RATIOS[k],)))


def lib():
    from hierarchical_block_sparse_lib_b200 import _capi
    return _capi.lib()


def E_ARG():
    from hierarchical_block_sparse_lib_b200 import _capi
    return _capi.HBSM_E_ARG


def single_leaf(hb, dtype, b, T):
    """a single-leaf b x b matrix whose tile is T (row, col)"""
    A = hb.HierarchicalBlockSparseMatrix(dtype, b)
    A.resize(b, b)
    A.assign_tiles(np.zeros(1, np.int64), np.zeros(1, np.int64), np.ascontiguousarray(T.T, dtype).reshape(1, b * b))
    return A


def leaf_factor(hb, A, dtype, b, zdim, valid):
    Z = hb.HierarchicalBlockSparseMatrix(dtype, b)
    assert lib().hbsm_leaf_inv_chol(A._h, Z._h, zdim, valid) == 0, lib().hbsm_last_error()
    bi, bj, _, t = Z.export_leaves(norms=False)
    assert (Z.get_n_rows(), Z.get_n_cols()) == (zdim, zdim)
    assert len(bi) == 1 and bi[0] == 0 and bj[0] == 0
    return t[0].reshape(b, b).T.copy()


def snapshot(X):
    bi, bj, nrm, t = X.export_leaves()
    return X.get_n_rows(), X.get_n_cols(), bi, bj, nrm.view(stored(X.dtype)), t.view(stored(X.dtype))


def same(s1, s2):
    return s1[:2] == s2[:2] and all(np.array_equal(x, y) for x, y in zip(s1[2:], s2[2:]))


LEAF_B = [1, 2, 7, 31, 32, 33, 64, 100, 128, 255, 256]


def valids(b):
    return sorted({b, max(b - 1, 1), 1, max(b // 2 + 1, 1)})


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("b", LEAF_B)
def test_leaf_kernel_against_reference_and_emulation(engine, dtype, b):
    """every valid in {b, b - 1, 1, b/2 + 1}, zdim in {b, valid}, the four input kinds; padding rows / columns hold NaN, so
    any read of them (even one multiplied by zero) shows in Z"""
    hb = engine
    for valid in valids(b):
        for kind in KINDS:
            Av = leaf_input(kind, valid, dtype, 1000 * b + valid)
            T = np.full((b, b), np.nan, dtype)
            T[:valid, :valid] = Av
            A = single_leaf(hb, dtype, b, T)
            k = kappa_of(Av)
            Zr = inv_factor_ref(Av, ref_prec(dtype))
            Ze = emulate_leaf(Av, dtype)
            for zdim in sorted({b, valid}):
                Z = leaf_factor(hb, A, dtype, b, zdim, valid)
                Zv = Z[:valid, :valid]
                ctx = (kind, valid, zdim)
                assert np.all(np.isfinite(Zv)), ctx
                assert not np.any(np.tril(Z, -1).view(stored(dtype))), ctx   # +0 bit patterns below the diagonal
                assert not np.any(Z[valid:].view(stored(dtype))) and not np.any(Z[:, valid:].view(stored(dtype))), ctx
                assert np.all(np.diag(Zv) > 0), ctx
                if kind == "ident":   # one nonzero product per sum: exact
                    want = np.diag(np.full(valid, np.sqrt(dtype(1) / dtype(3)), dtype))
                    assert np.array_equal(Zv.view(stored(dtype)), want.view(stored(dtype))), ctx
                r_ref, r_emu = ref_ratio(Zv, Zr, k, dtype), emul_ratio(Zv, Ze, k, dtype)
                note("REF", dtype, b, r_ref)
                note("EMUL", dtype, b, r_emu)
                assert r_ref <= 1, (ctx, r_ref)
                assert r_emu <= 1, (ctx, r_emu)
                Z2 = leaf_factor(hb, A, dtype, b, zdim, valid)
                assert np.array_equal(Z.view(stored(dtype)), Z2.view(stored(dtype))), ctx


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_leaf_kernel_argument_errors_leave_z_untouched(engine, dtype):
    hb = engine
    b = 8
    A = single_leaf(hb, dtype, b, leaf_input("k2", b, dtype, 1))
    Z = hb.HierarchicalBlockSparseMatrix(dtype, b)
    assert lib().hbsm_leaf_inv_chol(A._h, Z._h, b, b) == 0
    before = snapshot(Z)
    two = hb.HierarchicalBlockSparseMatrix(dtype, b)   # two leaves
    two.resize(2 * b, 2 * b)
    two.assign_tiles(np.array([0, 1]), np.array([0, 1]), np.tile(np.eye(b, dtype=dtype).ravel(), (2, 1)))
    unsized = hb.HierarchicalBlockSparseMatrix(dtype, b)
    bad = [(two, b, b), (unsized, b, b), (A, 0, b), (A, -1, b), (A, b + 1, b), (A, b - 1, b), (A, 3, 4)]   # valid > zdim
    for big in (257, 512):
        bad.append((single_leaf(hb, dtype, big, np.eye(big, dtype=dtype)), big, big))
    for X, zdim, valid in bad:
        assert lib().hbsm_leaf_inv_chol(X._h, Z._h, zdim, valid) == E_ARG(), (X.get_n_rows(), zdim)
        assert same(snapshot(Z), before)


# ---------------------------------------------------------------------------------------------------------------------
# quadrant extraction / assembly through the C ABI (GPU)
# ---------------------------------------------------------------------------------------------------------------------
QUAD_CASES = [(12, 9, 8, 0), (16, 16, 8, 1), (20, 30, 8, 2), (37, 53, 8, 3), (300, 200, 32, 1), (1000, 1000, 64, 0),
              (1000, 1000, 64, None)]   # rows, cols, b, root quadrant left empty


def quad_matrix(hb, dtype, m, n, b, empty_q, seed):
    """random tiles (about half of them), values zero outside m x n, root quadrant empty_q without tiles"""
    rng = np.random.default_rng(seed)
    gm, gn = -(-m // b), -(-n // b)
    v = b
    while v < max(m, n):
        v *= 2
    h = v // (2 * b)
    bi, bj = [x.ravel() for x in np.meshgrid(np.arange(gm), np.arange(gn), indexing="ij")]
    keep = rng.random(len(bi)) < 0.5
    if empty_q is not None:
        keep &= ~(((bi >= h) == (empty_q in (1, 3))) & ((bj >= h) == (empty_q in (2, 3))))
    keep[0] = keep[0] or empty_q != 0
    bi, bj = bi[keep], bj[keep]
    dense = np.zeros((v, v), dtype)
    tiles = np.zeros((len(bi), b * b), dtype)
    for t in range(len(bi)):
        T = rng.uniform(-1, 1, (b, b)).astype(dtype)
        T[m - bi[t] * b:, :] = 0
        T[:, n - bj[t] * b:] = 0
        dense[bi[t] * b:(bi[t] + 1) * b, bj[t] * b:(bj[t] + 1) * b] = T
        tiles[t] = T.T.ravel()
    A = hb.HierarchicalBlockSparseMatrix(dtype, b)
    A.resize(m, n)
    A.assign_tiles(bi, bj, tiles)
    A.update_internal_info()
    return A, dense, v


def extract(hb, A, q, dtype, b):
    Cq = hb.HierarchicalBlockSparseMatrix(dtype, b)
    e = C.c_int(-1)
    assert lib().hbsm_extract_quadrant(A._h, q, Cq._h, C.byref(e)) == 0, lib().hbsm_last_error()
    return Cq, e.value


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("case", QUAD_CASES, ids=lambda c: "%dx%d_b%d_q%s" % c)
def test_extract_and_assemble_quadrants(engine, dtype, case):
    hb = engine
    m, n, b, empty_q = case
    A, dense, v = quad_matrix(hb, dtype, m, n, b, empty_q, m + n + b)
    h = v // 2
    ai, aj, an, at = A.export_leaves()
    parts = []
    for q in range(4):
        Cq, e = extract(hb, A, q, dtype, b)
        r0, c0 = (h if q in (1, 3) else 0), (h if q in (2, 3) else 0)
        inq = (ai * b >= r0) & (ai * b < r0 + h) & (aj * b >= c0) & (aj * b < c0 + h)
        assert e == int(inq.any()), q
        assert (Cq.get_n_rows(), Cq.get_n_cols()) == (h, h)
        want = dense[r0:r0 + h, c0:c0 + h]
        assert np.array_equal(Cq.to_dense().view(stored(dtype)), want.view(stored(dtype))), q
        ci, cj, cn, ct = Cq.export_leaves()
        if e and h > b:
            assert np.array_equal(ci, ai[inq] - r0 // b) and np.array_equal(cj, aj[inq] - c0 // b)
            assert np.array_equal(cn.view(stored(dtype)), an[inq].view(stored(dtype)))
            assert np.array_equal(ct.view(stored(dtype)), at[inq].view(stored(dtype)))
        elif e:   # the child is one leaf
            assert len(ci) == 1 and ci[0] == 0 and cj[0] == 0
            assert np.array_equal(cn.view(stored(dtype)), an[inq].view(stored(dtype)))
            assert np.array_equal(ct.view(stored(dtype)), at[inq].view(stored(dtype)))
        elif h > b:
            assert len(ci) == 0
        else:     # an absent leaf child keeps its zero tile
            assert len(ci) == 1 and not np.any(ct)
        parts.append(Cq if e else (None if q % 2 == 0 else hb.HierarchicalBlockSparseMatrix(dtype, b)))
    R = hb.HierarchicalBlockSparseMatrix(dtype, b)
    hs = [p._h if p is not None else None for p in parts]
    assert lib().hbsm_assemble_quadrants(R._h, m, n, *hs) == 0, lib().hbsm_last_error()
    ri, rj, _, rt = R.export_leaves(norms=False)
    assert (R.get_n_rows(), R.get_n_cols()) == (m, n)
    assert np.array_equal(ri, ai) and np.array_equal(rj, aj)
    assert np.array_equal(rt.view(stored(dtype)), at.view(stored(dtype)))


@gpu
def test_quadrant_argument_errors(engine):
    hb = engine
    dt, b = np.float64, 8
    A, _, _ = quad_matrix(hb, dt, 37, 53, b, None, 3)
    leaf = single_leaf(hb, dt, b, np.eye(b))
    Cq = hb.HierarchicalBlockSparseMatrix(dt, b)
    e = C.c_int(0)
    L = lib()
    assert L.hbsm_extract_quadrant(A._h, 0, A._h, C.byref(e)) == E_ARG()
    for q in (-1, 4):
        assert L.hbsm_extract_quadrant(A._h, q, Cq._h, C.byref(e)) == E_ARG()
    assert L.hbsm_extract_quadrant(leaf._h, 0, Cq._h, C.byref(e)) == E_ARG()
    assert L.hbsm_extract_quadrant(hb.HierarchicalBlockSparseMatrix(dt, b)._h, 0, Cq._h, C.byref(e)) == E_ARG()
    q0, _ = extract(hb, A, 0, dt, b)                                 # 32 x 32 at b = 8: depth 2, fits a 37 x 53 target
    q3, _ = extract(hb, A, 3, dt, b)
    shallow, _ = extract(hb, q0, 0, dt, b)                           # depth 1
    f32, _, _ = quad_matrix(hb, np.float32, 32, 32, b, None, 4)
    b4 = hb.HierarchicalBlockSparseMatrix(dt, 4)
    b4.resize(16, 16)                                                # depth 2 as well
    b4.assign_tiles(np.array([0]), np.array([0]), np.eye(4).reshape(1, 16))
    R = hb.HierarchicalBlockSparseMatrix(dt, b)
    R.copy(A)
    before = snapshot(R)
    for args in [(R, 37, 53, R, None, None, q3),       # target aliases a quadrant
                 (R, 37, 53, None, None, None, None),  # all four absent
                 (R, 37, 53, hb.HierarchicalBlockSparseMatrix(dt, b), None, None, hb.HierarchicalBlockSparseMatrix(dt, b)),
                 (R, 8, 8, leaf, None, None, None),    # a single-leaf target
                 (R, 37, 53, q0, None, None, shallow),   # wrong depth
                 (R, 37, 53, q0, None, None, f32),       # wrong dtype
                 (R, 37, 53, q0, None, None, b4)]:       # wrong leaf size
        hs = [x._h if x is not None else None for x in args[3:]]
        assert L.hbsm_assemble_quadrants(args[0]._h, args[1], args[2], *hs) == E_ARG(), args[1:3]
        assert same(snapshot(R), before)


# ---------------------------------------------------------------------------------------------------------------------
# the C++ drop-in's recursion, M::inv_chol (tests/cpp/test_inv_chol.cc, one process per dtype and leaf size) (GPU)
# ---------------------------------------------------------------------------------------------------------------------
REC_B = [32, 64, 128, 256]
REC_KINDS = ["band", "bdiag", "dense"]


def rec_sizes(b):
    """n = 2b + 5 leaves valid = 5 <= half in the Schur complement one level down (Z11 skipped, A11 absent)"""
    return [b, b - 3, 2 * b + 5, 3 * b + 5, 8 * b - 1, 1000]


REC_SIZE_IDS = ["n=b", "n=b-3", "n=2b+5", "n=3b+5", "n=8b-1", "n=1000"]


_runs = {}


def run_program(dtype, b):
    """writes every (n, kind) case of this dtype and leaf size, runs the program once, returns {(n, kind): (A, result)}"""
    key = (np.dtype(dtype).name, b)
    if key in _runs:
        return _runs[key]
    if not os.path.exists(PROG):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    cases = [(n, kind) for n in rec_sizes(b) for kind in REC_KINDS]
    mats = {}
    with tempfile.TemporaryDirectory() as tmp:
        fin, fout = os.path.join(tmp, "in.bin"), os.path.join(tmp, "out.bin")
        with open(fin, "wb") as f:
            f.write(struct.pack("<i", len(cases)))
            for n, kind in cases:
                A = rec_input(kind, n, b, 31 * n + b)
                mats[(n, kind)] = A
                r, c = np.nonzero(A)
                f.write(struct.pack("<iiiq", 0 if dtype == np.float64 else 1, b, n, len(r)))
                f.write(r.astype("<i4").tobytes() + c.astype("<i4").tobytes() + A[r, c].astype("<f8").tobytes())
        p = subprocess.run([PROG, fin, fout], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        raw = open(fout, "rb").read()
    out, at = {}, 0
    for n, kind in cases:
        nb, kernel, zm, zn, cnt = struct.unpack_from("<qqqqq", raw, at)
        at += 40
        r = np.frombuffer(raw, "<i4", cnt, at); at += 4 * cnt
        c = np.frombuffer(raw, "<i4", cnt, at); at += 4 * cnt
        v = np.frombuffer(raw, "<f8", cnt, at); at += 8 * cnt
        out[(n, kind)] = (mats[(n, kind)], nb, kernel, (zm, zn), r, c, v)
    assert at == len(raw)
    _runs[key] = out
    return out


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("b", REC_B)
@pytest.mark.parametrize("kind", REC_KINDS)
@pytest.mark.parametrize("which", range(6), ids=REC_SIZE_IDS)
def test_dropin_inv_chol_recursion(engine, dtype, b, kind, which):
    n = rec_sizes(b)[which]
    A, n_blocks, kernel, dims, r, c, v = run_program(dtype, b)[(n, kind)]
    assert dims == (n, n)
    Z = np.zeros((n, n))
    Z[r, c] = v
    assert not np.any(v[r > c]), "nonzero below the diagonal"
    k = kappa_of(A)
    r_ref, r_res = ref_ratio(Z, rec_ref(A, dtype), k, dtype), resid_ratio(Z, A, k, dtype)
    note("REC", dtype, b, r_ref)
    note("RESID", dtype, b, r_res)
    assert r_ref <= 1 and r_res <= 1, (r_ref, r_res)
    g = -(-n // b)
    E = recursion_tiles(tile_pattern(A, b), n, b)
    assert not E[g:].any() and not E[:, g:].any() and not np.tril(E, -1).any()
    nz = np.zeros_like(E)
    nz[r // b, c // b] = True
    assert np.array_equal(nz, E) and n_blocks == E.sum(), (n_blocks, int(E.sum()))
    if kind == "bdiag":
        assert n_blocks == g   # Z block diagonal: only the diagonal leaves
    elif n > b:              # the recursion's products: fp64 DMMA, fp32 split-TF32 tcgen05 (grouped at b = 32 / 64)
        assert kernel == (1 if dtype == np.float64 else 3), kernel


def test_recursion_cases_reach_every_branch():
    """the drop-in cases above, replayed over their tile patterns, take every branch of inv_chol_rec at least once in
    each leaf size (dense inputs have every tile)"""
    want = {"single_leaf_root", "absent_A01", "absent_A10", "absent_A11", "valid_le_half", "ragged_leaf"}
    for b in REC_B:
        hits = set()
        for n in rec_sizes(b):
            for kind in REC_KINDS:
                if n <= b:
                    hits.add("single_leaf_root")
                P = tile_pattern(rec_input(kind, n, b, 31 * n + b), b) if kind != "dense" else \
                    pad_pattern(np.ones((-(-n // b),) * 2, bool))
                recursion_tiles(P, n, b, hits)
        assert hits == want, (b, want - hits)
