"""hbsm_multiply_accumulate: C <- alpha*op(A)*op(B) + beta*C in one call, checked bit for bit against the composition of
existing calls on copies, add(rescale(P, alpha), rescale(C_old, beta)) (rescale(P, alpha) when beta == 0 or C is
unsized), with P = multiply / spamm on the same operands; plus the executed set, counters, aliasing, argument errors and
the C++ drop-in's two statics.  Every test but the header syntax check needs the GPU."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import _capi
from hierarchical_block_sparse_lib_b200 import generators as G
from helpers import assert_bitwise, check_call, commit_halo, composition, copy_of

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HM = hb.HierarchicalBlockSparseMatrix
gpu = pytest.mark.gpu
BS = [7, 80, 32, 64, 128, 256]   # generic kernel at 7 / 80, tensor kernels at the others
DTYPES = [np.float64, np.float32]
TRANS = [(0, 0), (0, 1), (1, 0), (1, 1)]
AB = [(1.0, 1.0), (-1.0, 2.0), (0.5, -0.25), (2.0, 0.0), (0.0, 3.0),
      (0.1, 0.3), (1.0 / 3.0, -0.7)]   # both products inexact: an FMA, or alpha / beta not rounded to fp32, changes bits
OLD = ["unsized", "no_tiles", "outside", "subset", "equal"]


@pytest.fixture(scope="module")
def engine():
    hb.init(0)


def random_tiles(dtype, b, n, seed, frac=0.4):
    """random block-sparse n x n: ~frac of the tiles, entries U[-1,1) times a per-tile scale 10^-U(0,4), zero outside"""
    rng = np.random.default_rng(seed)
    g = -(-n // b)
    bi, bj = np.meshgrid(np.arange(g), np.arange(g), indexing="ij")
    bi, bj = bi.ravel(), bj.ravel()
    keep = rng.random(len(bi)) < frac
    return with_tiles(dtype, b, n, n, bi[keep], bj[keep], rng)


def with_tiles(dtype, b, m, n, bi, bj, rng):
    t = rng.uniform(-1, 1, (len(bi), b, b)) * (10.0 ** -rng.uniform(0, 4, len(bi)))[:, None, None]
    r = np.arange(b)
    for k in range(len(bi)):   # t[k] is (col, row): column-major tile
        t[k][:, bi[k] * b + r >= m] = 0.0
        t[k][bj[k] * b + r >= n, :] = 0.0
    A = HM(dtype, b)
    A.resize(m, n)
    if len(bi):
        A.assign_tiles(np.asarray(bi), np.asarray(bj), t.reshape(len(bi), b * b).astype(dtype))
    return A


def decay(dtype, b, n, seed):
    lam = 8.0 / b
    W = min(G.decay_width(lam), n - 1)
    r, c, v = G.decay_coo(n, lam, W, seed, symmetric=False, dtype=dtype)
    A = HM(dtype, b)
    A.resize(n, n)
    A.assign_from_vectors(r, c, v)
    return A


def operands(dtype, b, kind):
    n = 7 * b + 5
    if kind == "random":
        return random_tiles(dtype, b, n, 100 + b), random_tiles(dtype, b, n, 200 + b)
    return decay(dtype, b, n, 5 + b), decay(dtype, b, n, 6 + b)


def old_matrix(case, P, seed):
    """C_old for one of the OLD cases, relative to the pattern of the product P"""
    b = P.get_params().blocksize
    m, n = P.get_n_rows(), P.get_n_cols()
    if case == "unsized":
        return HM(P.dtype, b)
    rng = np.random.default_rng(seed)
    pi, pj, _, _ = P.export_leaves(tiles=False, norms=False)
    g = -(-max(m, n) // b)
    inP = np.zeros((g, g), bool)
    inP[pi, pj] = True
    if case == "no_tiles":
        bi = bj = np.zeros(0, np.int64)
    elif case == "equal":
        bi, bj = pi, pj
    elif case == "subset":   # P has tiles outside C_old's pattern
        keep = rng.random(len(pi)) < 0.5
        bi, bj = pi[keep], pj[keep]
    else:                    # C_old has tiles outside P's pattern (and some inside)
        gi, gj = np.meshgrid(np.arange(-(-m // b)), np.arange(-(-n // b)), indexing="ij")
        gi, gj = gi.ravel(), gj.ravel()
        keep = ~inP[gi, gj] | (rng.random(len(gi)) < 0.3)
        bi, bj = gi[keep], gj[keep]
    return with_tiles(P.dtype, b, m, n, bi, bj, rng)


CASES = [(d, b, t, k) for d in DTYPES for b in BS for t in TRANS for k in ("decay", "random")]
IDS = ["%s-b%d-t%d%d-%s" % ("f64" if d == np.float64 else "f32", b, t[0], t[1], k) for d, b, t, k in CASES]


@gpu
@pytest.mark.parametrize("dtype,b,trans,kind", CASES, ids=IDS)
def test_values_are_the_composition_bitwise(engine, dtype, b, trans, kind):
    A, B = operands(dtype, b, kind)
    tA, tB = trans
    P = HM(dtype, b)
    HM.multiply(A, tA, B, tB, P)
    for i, case in enumerate(OLD):
        Cold = old_matrix(case, P, 7 * b + i)
        for alpha, beta in AB:
            check_call(A, tA, B, tB, Cold, alpha, beta)


@gpu
@pytest.mark.parametrize("variant,dtype,b", [(1, np.float64, 32), (1, np.float32, 64), (1, np.float64, 128),
                                             (3, np.float32, 32), (3, np.float32, 64)])
def test_kernel_variants_match_their_own_composition(engine, variant, dtype, b):
    A, B = operands(dtype, b, "random")
    P = HM(dtype, b)
    HM.multiply(A, 0, B, 0, P)
    hb.set_gemm_variant(variant)
    try:
        for tA, tB in TRANS:
            for case in ("outside", "equal"):
                Cold = old_matrix(case, P, 3)
                for alpha, beta in [(-1.0, 2.0), (0.5, 0.0)]:
                    check_call(A, tA, B, tB, Cold, alpha, beta)
                    assert hb.stage_times()["gemm_kernel"] == (0 if variant == 1 else 3)
    finally:
        hb.set_gemm_variant(0)


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32), (np.float32, 128), (np.float64, 7)])
def test_aliasing(engine, dtype, b):
    A, B = operands(dtype, b, "random")
    for tA, tB in TRANS:
        # C is A
        want, _ = composition(A, tA, B, tB, A, 0.5, -0.25)
        X = copy_of(A)
        HM.multiply_accumulate(X, tA, B, tB, X, 0.5, -0.25)
        assert_bitwise(X, want)
        # C is B
        want, _ = composition(A, tA, B, tB, B, -1.0, 2.0)
        Y = copy_of(B)
        HM.multiply_accumulate(A, tA, Y, tB, Y, -1.0, 2.0)
        assert_bitwise(Y, want)
        # C is A is B: X <- 2X - op(X) op(X) in one call, against the four-call idiom
        X = copy_of(A)
        P = HM(dtype, b)
        HM.multiply(A, tA, A, tB, P)
        P1 = HM(dtype, b)
        P1.rescale(P, -1.0)
        X1 = HM(dtype, b)
        X1.rescale(A, 2.0)
        Xn = HM(dtype, b)
        HM.add(P1, X1, Xn)
        nm, nr = HM.multiply_accumulate(X, tA, X, tB, X, -1.0, 2.0)
        assert_bitwise(X, Xn)
        assert nm == len(P.export_tasks()) and nr == Xn.get_n_blocks()


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32), (np.float64, 80), (np.float32, 256)])
@pytest.mark.parametrize("updated", [True, False])
def test_spamm_executed_set_and_values(engine, dtype, b, updated):
    A, B = operands(dtype, b, "decay")
    A.update_internal_info()
    B.update_internal_info()
    na = A.export_leaves(tiles=False)[2].astype(np.float64)
    nb = B.export_leaves(tiles=False)[2].astype(np.float64)
    tau = float(np.sqrt(np.median(na) * np.median(nb)))
    P = HM(dtype, b)
    HM.multiply(A, 0, B, 0, P)
    for tA, tB in TRANS:
        S = HM(dtype, b)
        HM.spamm(A, tA, B, tB, S, tau, updated)
        Cold = old_matrix("outside", P, 11)
        Cm, Pspamm = check_call(A, tA, B, tB, Cold, -1.0, 2.0, spamm=tau, updated=updated)
        assert np.array_equal(Cm.export_tasks(), S.export_tasks())
        assert 0 < len(S.export_tasks()) < len(HM_tasks(A, tA, B, tB))


def HM_tasks(A, tA, B, tB):
    P = HM(A.dtype, A.get_params().blocksize)
    HM.multiply(A, tA, B, tB, P)
    return P.export_tasks()


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_beta_zero_never_reads_old_c(engine, dtype):
    for b in (7, 32, 64):
        A, B = operands(dtype, b, "random")
        P = HM(dtype, b)
        HM.multiply(A, 0, B, 0, P)
        bi, bj, _, _ = old_matrix("outside", P, 1).export_leaves(tiles=False, norms=False)
        Cm = HM(dtype, b)
        Cm.resize(P.get_n_rows(), P.get_n_cols())
        Cm.assign_tiles(bi, bj, np.full((len(bi), b * b), np.nan, dtype))
        want = HM(dtype, b)
        want.rescale(P, 1.5)
        HM.multiply_accumulate(A, 0, B, 0, Cm, 1.5, 0.0)
        assert_bitwise(Cm, want)
        assert not np.isnan(Cm.export_leaves(norms=False)[3]).any()


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_counters_tile_tasks_and_stage_times(engine, dtype):
    b = 32
    A, B = operands(dtype, b, "random")
    P = HM(dtype, b)
    HM.multiply(A, 0, B, 0, P)
    Cold = old_matrix("outside", P, 5)
    Cold.set_n_block_multiplicaitons(1234)   # (sic, H:220)
    Cm, _ = check_call(A, 0, B, 0, Cold, 1.0, 1.0)
    assert Cm.get_n_block_multiplications() == len(P.export_tasks()) + 1234
    st = hb.stage_times()
    assert st["n_products"] == len(P.export_tasks()) and st["gemm_ms"] > 0 and st["total_ms"] >= st["gemm_ms"]
    pi, pj, _, _ = P.export_leaves(tiles=False, norms=False)
    ci, cj, _, _ = Cm.export_leaves(tiles=False, norms=False)
    inP = set(zip(pi.tolist(), pj.tolist()))
    for i, j in zip(ci.tolist(), cj.tolist()):
        k = Cm.tile_tasks(i, j)
        if (i, j) in inP:
            assert np.array_equal(k, P.tile_tasks(i, j))
        else:
            assert k is not None and len(k) == 0   # a tile only in C_old has no products
    Cm2, _ = check_call(A, 0, B, 0, Cold, 1.0, 0.0)
    assert Cm2.get_n_block_multiplications() == len(P.export_tasks())


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_two_calls_are_bitwise_equal(engine, dtype):
    for b in (32, 64, 80):
        A, B = operands(dtype, b, "random")
        P = HM(dtype, b)
        HM.multiply(A, 0, B, 0, P)
        Cold = old_matrix("outside", P, 9)
        X, Y = copy_of(Cold), copy_of(Cold)
        HM.multiply_accumulate(A, 1, B, 0, X, -0.75, 1.25)
        HM.multiply_accumulate(A, 1, B, 0, Y, -0.75, 1.25)
        assert_bitwise(X, Y)


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_no_executed_products(engine, dtype):
    for b in (32, 64, 7):
        A, B = operands(dtype, b, "random")
        P = HM(dtype, b)
        HM.multiply(A, 0, B, 0, P)
        Cold = old_matrix("outside", P, 4)
        E = HM(dtype, b)   # an operand without tiles
        E.resize(A.get_n_rows(), A.get_n_cols())
        for alpha, beta in [(-1.0, 2.0), (0.1, 0.3), (2.0, 0.0)]:
            check_call(E, 0, B, 0, Cold, alpha, beta)
            check_call(A, 1, E, 0, Cold, alpha, beta)
        A.update_internal_info()
        B.update_internal_info()
        for updated in (True, False):   # SpAMM skips every product
            Cm, _ = check_call(A, 0, B, 0, Cold, -1.0, 2.0, spamm=1e30, updated=updated)
            assert len(Cm.export_tasks()) == 0 and Cm.get_n_blocks() == Cold.get_n_blocks()


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_single_leaf_whose_product_spamm_skips(engine, dtype):
    """hbsm_spamm leaves the zero leaf of a single-leaf C: the accumulating call scales that leaf, signs of zeros included"""
    for b in (7, 32, 64):
        n = b - 3
        A = with_tiles(dtype, b, n, n, [0], [0], np.random.default_rng(b))
        A.update_internal_info()
        P = HM(dtype, b)
        HM.multiply(A, 0, A, 0, P)
        for case in ("unsized", "equal"):
            Cold = old_matrix(case, P, 2)
            for alpha, beta in [(-1.0, 0.0), (-1.0, 2.0), (0.1, -0.3), (float("inf"), 0.0), (2.0, 1.0)]:
                Cm, _ = check_call(A, 0, A, 0, Cold, alpha, beta, spamm=1e30)
                assert Cm.get_n_blocks() == 1
        X = copy_of(A)
        want, _ = composition(A, 0, A, 0, A, -1.0, 0.0, spamm=1e30)
        HM.spamm_accumulate(X, 0, X, 0, X, -1.0, 0.0, 1e30)
        assert_bitwise(X, want)
        assert np.signbit(X.export_leaves(norms=False)[3]).all()   # fl(-1 * +0) = -0, as rescale(P, -1)


@gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_n_mults_and_root_norm_of_a_sized_c(engine, dtype):
    b = 32
    A, B = operands(dtype, b, "random")
    P = HM(dtype, b)
    nm0, _ = HM.multiply(A, 0, B, 0, P)
    for beta, extra in [(2.0, 77), (0.0, 0)]:
        Cm = HM(dtype, b)   # sized, no tiles, a recorded n_mults
        Cm.resize(A.get_n_rows(), A.get_n_cols())
        Cm.set_n_block_multiplicaitons(77)   # (sic, H:220)
        nm, _ = HM.multiply_accumulate(A, 0, B, 0, Cm, 1.0, beta)
        assert nm == nm0 and Cm.get_n_block_multiplications() == nm0 + extra
    Cm = old_matrix("outside", P, 8)
    Cm.update_internal_info()
    assert Cm.get_frob_norm_squared_internal() > 0
    HM.multiply_accumulate(A, 0, B, 0, Cm, 1.0, 1.0)
    assert Cm.get_frob_norm_squared_internal() == P.get_frob_norm_squared_internal() == 0


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32), (np.float32, 128)])
@pytest.mark.parametrize("updated", [True, False])
def test_spamm_in_place_purification(engine, dtype, b, updated):
    """X <- 2X - spamm(op(X), op(X), tau) in one call, C is A is B"""
    A, _ = operands(dtype, b, "decay")
    A.update_internal_info()
    na = A.export_leaves(tiles=False)[2].astype(np.float64)
    tau = float(np.sqrt(np.median(na) * np.quantile(na, 0.7)))
    for tA, tB in TRANS:
        want, P = composition(A, tA, A, tB, A, -1.0, 2.0, spamm=tau, updated=updated)
        X = copy_of(A)
        X.update_internal_info()
        nm, nr = HM.spamm_accumulate(X, tA, X, tB, X, -1.0, 2.0, tau, updated)
        assert_bitwise(X, want)
        assert nm == len(P.export_tasks()) > 0 and nr == want.get_n_blocks()
        assert np.array_equal(X.export_tasks(), P.export_tasks())


@gpu
@pytest.mark.parametrize("dtype,b", [(np.float64, 64), (np.float32, 32), (np.float64, 7)])
def test_halo_of_b_takes_part_and_halo_of_c_is_dropped(engine, dtype, b):
    A, B = operands(dtype, b, "random")
    g = -(-B.get_n_rows() // b)
    bi, bj, _, _ = B.export_leaves(tiles=False, norms=False)
    own = set(zip(bi.tolist(), bj.tolist()))
    free = [(i, j) for i in range(g) for j in range(g) if (i, j) not in own][:5]
    commit_halo(B, [p[0] for p in free], [p[1] for p in free], 1)
    P = HM(dtype, b)
    HM.multiply(A, 0, B, 0, P)
    Q = HM(dtype, b)
    B0 = copy_of(B)   # the own tiles only
    HM.multiply(A, 0, B0, 0, Q)
    assert len(P.export_tasks()) > len(Q.export_tasks())   # the halo tiles are read
    Cold = old_matrix("outside", P, 6)
    check_call(A, 0, B, 0, Cold, -1.0, 2.0)
    # a halo on C: C_old is C's own tiles, and the call drops the halo
    ci, cj, _, _ = Cold.export_leaves(tiles=False, norms=False)
    cown = set(zip(ci.tolist(), cj.tolist()))
    cfree = [(i, j) for i in range(g) for j in range(g) if (i, j) not in cown][:3]
    want, _ = composition(A, 0, B0, 0, Cold, 0.1, 0.3)
    commit_halo(Cold, [p[0] for p in cfree], [p[1] for p in cfree], 2)
    HM.multiply_accumulate(A, 0, B0, 0, Cold, 0.1, 0.3)
    assert_bitwise(Cold, want)
    assert _capi.lib().hbsm_halo_commit(Cold._h, 1) == _capi.HBSM_E_ARG   # nothing reserved any more


@gpu
def test_every_argument_error_returns_before_any_launch(engine):
    L = _capi.lib()
    A, B = operands(np.float64, 32, "random")
    Cold = old_matrix("outside", HM_product(A, B), 2)
    before = Cold.export_leaves()
    nm, nr = C.c_size_t(7), C.c_size_t(7)

    def call(a, ta, bb, tb, c, spamm=0):
        l0 = hb.kernel_launch_count()
        rc = L.hbsm_multiply_accumulate(a, ta, bb, tb, c, -1.0, 2.0, spamm, 0.1, 1, C.byref(nm), C.byref(nr))
        assert hb.kernel_launch_count() == l0
        return rc, last_error()

    def plain(a, ta, bb, tb, spamm=0):
        E = HM(np.float64, 32)
        rc = L.hbsm_spamm(a, ta, bb, tb, E._h, 0.1, 1, None, None) if spamm else L.hbsm_multiply(a, ta, bb, tb, E._h, None, None)
        return rc, last_error()

    unsized = HM(np.float64, 32)
    rect = with_tiles(np.float64, 32, 100, 60, [0], [0], np.random.default_rng(0))
    f32 = operands(np.float32, 32, "random")[0]
    b64 = HM(np.float64, 64)
    b64.resize(A.get_n_rows(), A.get_n_cols())
    for spamm in (0, 1):   # the operand errors of multiply / spamm: same codes, same messages
        for a, ta, bb, tb in [(unsized._h, 0, B._h, 0), (A._h, 0, unsized._h, 0), (A._h, 0, f32._h, 0), (A._h, 0, b64._h, 0),
                              (A._h, 0, rect._h, 0), (rect._h, 1, A._h, 0)]:
            got = call(a, ta, bb, tb, Cold._h, spamm)
            assert got == plain(a, ta, bb, tb, spamm) and got[0] != 0
    assert call(None, 0, B._h, 0, Cold._h)[0] == _capi.HBSM_E_ARG
    assert call(A._h, 0, B._h, 0, None)[0] == _capi.HBSM_E_ARG
    # a sized C of the wrong shape, dtype or leaf size
    wrong_shape = with_tiles(np.float64, 32, A.get_n_rows(), A.get_n_cols() - 40, [0], [0], np.random.default_rng(1))
    wrong_dtype = HM(np.float32, 32)
    wrong_dtype.resize(A.get_n_rows(), A.get_n_cols())
    wrong_b = HM(np.float64, 64)
    wrong_b.resize(A.get_n_rows(), A.get_n_cols())
    for W in (wrong_shape, wrong_dtype, wrong_b):
        w0 = W.export_leaves()
        assert call(A._h, 0, B._h, 0, W._h)[0] == _capi.HBSM_E_ARG
        for x, y in zip(w0, W.export_leaves()):
            assert np.array_equal(x, y)
    # a product in flight on this thread
    F = HM(np.float64, 32)
    _capi.check(L.hbsm_product_begin(A._h, 0, B._h, 0, F._h, 0, 0.0, 1, 0))
    try:
        l0 = hb.kernel_launch_count()
        assert L.hbsm_multiply_accumulate(A._h, 0, B._h, 0, Cold._h, 1.0, 1.0, 0, 0.0, 1, None, None) == _capi.HBSM_E_ARG
        assert hb.kernel_launch_count() == l0
    finally:
        L.hbsm_product_abort()
    for x, y in zip(before, Cold.export_leaves()):   # C untouched by every rejected call
        assert np.array_equal(x, y, equal_nan=True)
    assert Cold.get_n_rows() == A.get_n_rows()


def last_error():
    e = _capi.lib().hbsm_last_error()
    return e.decode() if isinstance(e, bytes) else str(e)


def HM_product(A, B):
    P = HM(A.dtype, A.get_params().blocksize)
    HM.multiply(A, 0, B, 0, P)
    return P


CPP = r"""
#include "hbsm/hierarchical_block_sparse_lib.h"
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>
typedef hbsm::HierarchicalBlockSparseMatrix<double> M;
static bool same(const M& X, const M& Y) {
    std::vector<int> r1, c1, r2, c2; std::vector<double> v1, v2;
    X.get_all_values(r1, c1, v1); Y.get_all_values(r2, c2, v2);
    return r1 == r2 && c1 == c2 && v1.size() == v2.size() && (v1.empty() || std::memcmp(&v1[0], &v2[0], v1.size() * sizeof(double)) == 0);
}
int main() {
    M::Params p; p.blocksize = 8;
    const int n = 61;
    M X; X.set_params(p); X.resize(n, n);
    std::vector<int> r, c; std::vector<double> v;
    for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) if (std::abs(i - j) <= 12) { r.push_back(i); c.push_back(j); v.push_back(std::ldexp(1.0 + (i + 2 * j) / 256.0, -std::abs(i - j))); }
    X.assign_from_vectors(r, c, v);
    // X <- 2X - X*X: one call against the four-call idiom
    M P, P1, X1, Xn; P.set_params(p); P1.set_params(p); X1.set_params(p); Xn.set_params(p);
    M::multiply(X, false, X, false, P);
    P1.rescale(P, -1.0); X1.rescale(X, 2.0); M::add(P1, X1, Xn);
    M Y; Y.set_params(p); Y.copy(X);
    size_t nm = 0, nr = 0;
    M::multiply_accumulate(Y, false, Y, false, Y, -1.0, 2.0, &nm, &nr);
    if (!same(Y, Xn) || nm != P.get_n_block_multiplications() || nr != Xn.get_n_blocks()) { std::printf("multiply_accumulate differs\n"); return 1; }
    // SpAMM: C <- 0.5 spamm(X^T, X, tau) + C
    X.update_internal_info();
    M S, S1, Z, Zn; S.set_params(p); S1.set_params(p); Z.set_params(p); Zn.set_params(p);
    M::spamm(X, true, X, false, S, 1e-3, true);
    S1.rescale(S, 0.5); M::add(S1, X, Zn);
    Z.copy(X);
    M::spamm_accumulate(X, true, X, false, Z, 0.5, 1.0, 1e-3, true, &nm, &nr);
    if (!same(Z, Zn) || nm != S.get_n_block_multiplications()) { std::printf("spamm_accumulate differs\n"); return 1; }
    std::printf("ok %zu %zu\n", nm, nr);
    return 0;
}
"""


def test_header_declares_the_call_and_compiles_cxx11_werror():
    src = ('#include "hbsm/hierarchical_block_sparse_lib.h"\n'
           "template class hbsm::HierarchicalBlockSparseMatrix<double>;\n"
           "template class hbsm::HierarchicalBlockSparseMatrix<float>;\n"
           "int (*f)(hbsm_handle, int, hbsm_handle, int, hbsm_handle, double, double, int, double, int, size_t*, size_t*) = "
           "hbsm_multiply_accumulate;\nint main(){return f == 0;}\n")
    r = subprocess.run(["/usr/bin/g++", "-std=c++11", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                        "-x", "c++", "-"], input=src, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


@gpu
def test_cpp_dropin_statics(engine):
    libdir = os.path.join(ROOT, "hierarchical_block_sparse_lib_b200", "lib")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "t.cc"), os.path.join(d, "t")
        open(src, "w").write(CPP)
        r = subprocess.run(["/usr/bin/g++", "-std=c++11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                            "-L", libdir, "-lhbsm_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.startswith("ok ")
