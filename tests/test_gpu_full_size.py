"""-m gpu: the five BASELINE.json configurations at their FULL sizes through the C ABI, checked with size-independent
properties (the CPU oracle cannot finish these sizes in test time; cfg 1 is small enough and is compared with it directly):
executed-product set == the flat rule recomputed on the host from the exported leaf norms (SURVEY 8c "light oracle"),
transposition identities, triu(A*A) for the symmetric square, linearity, exactness of add."""
import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import generators as G
from oracle import pyoracle as po
from helpers import HBSM, both_from_coo, flat_rule_tasks, sort_tasks, rel_frob

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _built(oracle_built):
    hb.init(0)
    return oracle_built


def test_cfg1_exact_multiply_random_block_sparse_vs_oracle():
    """configs[0]: exact multiply, random block-sparse fp64 N=1024 leaf=32 -- against the CPU oracle port and, where built,
    the unmodified reference: identical executed set, values to 1e-12."""
    n, b = 1024, 32
    ra, ca, va = G.random_block_sparse_coo(n, b, 0.30, 1); rb, cb, vb = G.random_block_sparse_coo(n, b, 0.30, 2)
    Ag, Ao = both_from_coo(b, n, n, ra, ca, va); Bg, Bo = both_from_coo(b, n, n, rb, cb, vb)
    C = HBSM(np.float64); nm, nr = HBSM.multiply(Ag, 0, Bg, 0, C)
    Co, onm, onb, ot = po.OrcMatrix.product(Ao, 0, Bo, 0, want_tasks=True)
    assert (nm, nr) == (onm, onb)
    assert np.array_equal(sort_tasks(C.export_tasks()), sort_tasks(ot))
    assert rel_frob(C.to_dense(), Co.to_dense()) <= 1e-12
    assert rel_frob(C.to_dense(), Ag.to_dense() @ Bg.to_dense()) <= 1e-12
    Cs = HBSM(np.float64); nms, _ = HBSM.spamm(Ag, 0, Bg, 0, Cs, 0.0, True)      # tau = 0 cross-check (SURVEY 8d)
    assert nms == nm and np.array_equal(Cs.export_leaves(norms=False)[3], C.export_leaves(norms=False)[3])
    import os
    if os.path.exists(po.REF_SO):
        Ar = po.from_coo(po.RefMatrix, b, n, n, ra, ca, va); Br = po.from_coo(po.RefMatrix, b, n, n, rb, cb, vb)
        Cr, rnm, rnb, rt = po.RefMatrix.product(Ar, 0, Br, 0, want_tasks=True)
        assert (nm, nr) == (rnm, rnb) and np.array_equal(sort_tasks(C.export_tasks()), sort_tasks(rt))
        assert rel_frob(C.to_dense(), Cr.to_dense()) <= 1e-12


def test_cfg3_symm_square_full_size():
    """configs[2]: symm_square of banded symmetric decay, fp64 N=65536 leaf=64; tau sweep as the SpAMM-pruned symmetric square."""
    n, b, lam = 65536, 64, 0.05
    g = n // b
    W = G.decay_width(lam)
    F = HBSM(np.float64, b); F.generate_decay(n, lam, W, 3, symmetric=True); F.update_internal_info()
    U = HBSM(np.float64); F.get_upper_triangle(U); U.update_internal_info()
    # exact: symm_square(U) == triu(F*F), tile for tile
    C = HBSM(np.float64); HBSM.symm_square(U, C)
    Cf = HBSM(np.float64); nmf, _ = HBSM.multiply(F, 0, F, 0, Cf)
    Cu = HBSM(np.float64); Cf.get_upper_triangle(Cu)
    ci, cj, _, t1 = C.export_leaves(norms=False); ui, uj, _, t2 = Cu.export_leaves(norms=False)
    assert np.array_equal(ci, ui) and np.array_equal(cj, uj) and np.all(ci <= cj)
    assert rel_frob(t1, t2) <= 1e-13
    # F*F of a symmetric F is symmetric: the full product equals its own transpose (same tiles, transposed)
    Ct = HBSM(np.float64); HBSM.transpose(Cf, Ct)
    assert rel_frob(Ct.export_leaves(norms=False)[3], Cf.export_leaves(norms=False)[3]) <= 1e-13
    del Ct, Cu, t1, t2
    for tau in (1e-4, 1e-6, 1e-8, 1e-10):
        Cs = HBSM(np.float64); nm, nr = HBSM.symm_square_spamm(U, Cs, tau)
        want = flat_rule_tasks(F, 0, F, 0, tau, g, upper_only=True)
        assert nm == len(want)
        assert np.array_equal(sort_tasks(Cs.export_tasks()), sort_tasks(want))
        Cfs = HBSM(np.float64); HBSM.spamm(F, 0, F, 0, Cfs, tau, True)
        Cus = HBSM(np.float64); Cfs.get_upper_triangle(Cus)
        assert nr == Cus.get_n_blocks()
        assert rel_frob(Cs.export_leaves(norms=False)[3], Cus.export_leaves(norms=False)[3]) <= 1e-13


def test_cfg4_spamm_n262144_leaf128_task_set():
    """configs[3] on one GPU: fp64 N=262144 leaf=128 tau=1e-6 -- executed set == flat rule, (AB)^T == B^T A^T."""
    n, b, lam, tau = 262144, 128, 0.01, 1e-6
    g = n // b
    W = G.decay_width(lam)
    A = HBSM(np.float64, b); A.generate_decay(n, lam, W, 1); A.update_internal_info()
    B = HBSM(np.float64, b); B.generate_decay(n, lam, W, 2); B.update_internal_info()
    C = HBSM(np.float64); nm, nr = HBSM.spamm(A, 0, B, 0, C, tau, True)
    want = flat_rule_tasks(A, 0, B, 0, tau, g)
    assert nm == len(want) and nr == C.get_n_blocks()
    assert np.array_equal(sort_tasks(C.export_tasks()), sort_tasks(want))
    # a sample of C tiles recomputed in numpy from the operand tiles (SURVEY 8c: sample C tiles, same k order)
    t = sort_tasks(C.export_tasks())
    rng = np.random.default_rng(0)
    ci_all, cj_all, _, _ = C.export_leaves(tiles=False)
    for s in rng.choice(len(ci_all), 4, replace=False):
        ci, cj = int(ci_all[s]), int(cj_all[s])
        ks = t[(t[:, 0] == ci) & (t[:, 1] == cj)][:, 2]
        ref = np.zeros((b, b))
        for k in ks:
            ref += A.get_tile(ci, int(k)) @ B.get_tile(int(k), cj)
        got = C.get_tile(ci, cj)
        assert rel_frob(got, ref) <= 1e-12


@pytest.mark.parametrize("b", [32, 64, 128, 256])
def test_cfg5_fp32_transposed_and_add_full_size(b):
    """configs[4]: fp32 N=65536, A^T*B and A*B^T against the explicitly transposed operand, add against numpy; leaf sweep."""
    n, lam, tau = 65536, 0.02, 1e-6
    g = n // b
    W = G.decay_width(lam)
    A = HBSM(np.float32, b); A.generate_decay(n, lam, W, 1); A.update_internal_info()
    B = HBSM(np.float32, b); B.generate_decay(n, lam, W, 2); B.update_internal_info()
    At = HBSM(np.float32); HBSM.transpose(A, At); At.update_internal_info()
    Bt = HBSM(np.float32); HBSM.transpose(B, Bt); Bt.update_internal_info()
    # A^T * B through the flag == (explicit A^T) * B : same executed set, values within the fp32 tolerance
    C1 = HBSM(np.float32); nm1, nr1 = HBSM.spamm(A, 1, B, 0, C1, tau, True)
    C2 = HBSM(np.float32); nm2, nr2 = HBSM.spamm(At, 0, B, 0, C2, tau, True)
    assert (nm1, nr1) == (nm2, nr2)
    assert np.array_equal(sort_tasks(C1.export_tasks()), sort_tasks(C2.export_tasks()))
    assert rel_frob(C1.export_leaves(norms=False)[3], C2.export_leaves(norms=False)[3]) <= 1e-5
    assert nm1 == len(flat_rule_tasks(A, 1, B, 0, tau, g))
    del C2
    C3 = HBSM(np.float32); nm3, nr3 = HBSM.spamm(A, 0, B, 1, C3, tau, True)
    C4 = HBSM(np.float32); nm4, nr4 = HBSM.spamm(A, 0, Bt, 0, C4, tau, True)
    assert (nm3, nr3) == (nm4, nr4)
    assert rel_frob(C3.export_leaves(norms=False)[3], C4.export_leaves(norms=False)[3]) <= 1e-5
    del C1, C3, C4, At, Bt
    # add: union structure, fl(a+b) bit-exact where both exist (same law, same band => same structure here)
    S = HBSM(np.float32); HBSM.add(A, B, S)
    ai, aj, _, ta = A.export_leaves(norms=False); bi, bj, _, tb = B.export_leaves(norms=False)
    si, sj, _, ts = S.export_leaves(norms=False)
    assert np.array_equal(ai, bi) and np.array_equal(aj, bj) and np.array_equal(si, ai) and np.array_equal(sj, aj)
    assert np.array_equal(ts, ta + tb)
