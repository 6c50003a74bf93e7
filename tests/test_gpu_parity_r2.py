"""-m gpu parity tests, second batch: the tensor-core leaf kernels against the UNMODIFIED reference (oracle/_ref) directly,
for every leaf size and operand orientation; BASELINE config 2 at full size against the reference; the norm fold on
scattered patterns; re-entrancy; the parity hooks used by bench.py --check."""
import os
import threading

import numpy as np
import pytest

import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import generators as G
from oracle import pyoracle as po
from oracle import sampled_check as sc
from helpers import HBSM, both_from_coo, gpu_from_coo, sort_tasks, rel_frob, leaves_equal_structure

pytestmark = pytest.mark.gpu
TOL = {np.float64: 1e-12, np.float32: 1e-5}


@pytest.fixture(scope="module", autouse=True)
def _built(oracle_built):
    hb.init(0)
    return oracle_built


def _ref_cls():
    return sc.checker_class()   # the unmodified reference where its build travelled, else the (pinned) port


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("b", [32, 64, 128, 256])
@pytest.mark.parametrize("tA,tB", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_tensor_core_kernels_against_the_reference(dtype, b, tA, tB):
    """DMMA (fp64) / tcgen05 (fp32) leaf kernels, every leaf size and (tA,tB): executed-product set bit-exact and C within
    the stated tolerance of the reference's own spamm() (hierarchical prune H:6649-6651, leaf gemm H:7273).  tau prunes
    about 40 % of the structurally possible products, so the predicate is exercised, not just the structure."""
    cls = _ref_cls()
    n, lam, tau = 6 * b, 4.0 / b, 1e-3
    W = min(G.decay_width(lam), n - 1)
    ra, ca, va = G.decay_coo(n, lam, W, 1, dtype=dtype)
    rb, cb, vb = G.decay_coo(n, lam, W, 2, dtype=dtype)
    g_a, r_a = both_from_coo(b, n, n, ra, ca, va, dtype, cls)
    g_b, r_b = both_from_coo(b, n, n, rb, cb, vb, dtype, cls)
    Cg = HBSM(dtype)
    nm, nr = HBSM.spamm(g_a, tA, g_b, tB, Cg, tau, True)
    assert hb.stage_times()["gemm_kernel"] == (1 if dtype == np.float64 else 3), "the tensor-core kernel did not run"
    Cr, rnm, rnb, rt = cls.product(r_a, tA, r_b, tB, spamm=True, tau=tau, want_tasks=True)
    assert 0 < rnm < 216, "the test must prune some but not all products"
    assert (nm, nr) == (rnm, rnb)
    assert np.array_equal(sort_tasks(Cg.export_tasks()), sort_tasks(rt))
    assert leaves_equal_structure(Cg, Cr)
    assert rel_frob(Cg.to_dense(), Cr.to_dense()) <= TOL[dtype]
    assert Cg.task_checksum() == G.task_checksum(rt[:, 0], rt[:, 1], rt[:, 2])
    # exact multiply on the same operands: structure-only rule (worth_to_multiply H:1873)
    Ce = HBSM(dtype)
    nme, nre = HBSM.multiply(g_a, tA, g_b, tB, Ce)
    Cre, enm, enb, _ = cls.product(r_a, tA, r_b, tB)
    assert (nme, nre) == (enm, enb) and rel_frob(Ce.to_dense(), Cre.to_dense()) <= TOL[dtype]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_leaf_norms_bit_exact_b256(dtype):
    b, n = 256, 256 * 4
    r, c, v = G.decay_coo(n, 0.01, min(G.decay_width(0.01), n - 1), 4, dtype=dtype)
    g, o = both_from_coo(b, n, n, r, c, v, dtype, _ref_cls())
    _, _, gn, _ = g.export_leaves(tiles=False)
    _, _, on, _ = o.leaves(tiles=False)
    assert np.array_equal(gn, on)
    assert g.get_frob_norm_squared_internal() == o.frob_sq_cached()
    assert g.get_frob_squared() == o.frob_sq()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("case", ["random_1pct_depth8", "diagonal_stride4_depth8", "random_depth13_fallback", "dense_depth3"])
def test_root_norm_on_scattered_patterns(dtype, case):
    """The bottom-up norm refresh (H:3918-3923) on patterns where an upper level has about as many nodes as the leaves
    (scattered tiles: no halving per level), compared bit-for-bit with the oracle's recursive sum."""
    rng = np.random.default_rng(7)
    if case == "random_1pct_depth8":
        b, g = 4, 256
        t = rng.choice(g * g, size=g * g // 100, replace=False)
        bi, bj = t // g, t % g
    elif case == "diagonal_stride4_depth8":
        b, g = 4, 256
        bi = np.arange(0, g, 4); bj = bi.copy()
    elif case == "random_depth13_fallback":
        b, g = 1, 8192
        bi = rng.integers(0, g, 3000); bj = rng.integers(0, g, 3000)
    else:
        b, g = 8, 8
        bi, bj = [x.ravel() for x in np.meshgrid(np.arange(g), np.arange(g), indexing="ij")]
    n = b * g
    r = (bi[:, None] * b + rng.integers(0, b, (len(bi), 3))).ravel()
    c = (bj[:, None] * b + rng.integers(0, b, (len(bi), 3))).ravel()
    v = rng.standard_normal(len(r)).astype(dtype)
    g_m, o_m = both_from_coo(b, n, n, r, c, v, dtype)
    assert g_m.get_n_blocks() == o_m.n_blocks()
    assert g_m.get_frob_norm_squared_internal() == o_m.frob_sq_cached()
    assert g_m.get_frob_squared() == o_m.frob_sq()
    # a neighbouring matrix allocated right behind it must be untouched by the refresh (the old fold wrote past its scratch)
    other = gpu_from_coo(b, n, n, r[:30], c[:30], v[:30], dtype)
    before = other.export_leaves()[3].copy()
    for _ in range(3):
        g_m.update_internal_info()
    assert np.array_equal(other.export_leaves()[3], before)


@pytest.mark.parametrize("lam", [0.05, 0.01])
def test_cfg2_full_size_against_the_reference(lam):
    """BASELINE config 2 at FULL size (N=16384, leaf 64, tau=1e-6), both decay presets, against the unmodified reference run
    on the same matrices: identical assembled tiles and leaf norms, identical executed-product set, C within 1e-12.
    Where oracle/_ref is not built, the pinned port checks sampled C tiles on their own sub-problems (what bench.py --check
    runs; the port would take minutes on the whole product) and the flat rule the whole executed set."""
    cls = _ref_cls()
    n, b, tau = 16384, 64, 1e-6
    W = min(G.decay_width(lam), n - 1)
    if cls is not po.RefMatrix:
        A = HBSM(np.float64, b); A.generate_decay(n, lam, W, 1); A.update_internal_info()
        B = HBSM(np.float64, b); B.generate_decay(n, lam, W, 2); B.update_internal_info()
        Cg = HBSM(np.float64)
        nm, nr = HBSM.spamm(A, 0, B, 0, Cg, tau, True)
        res = sc.sampled_check(Cg, A, B, n, b, lam, W, (1, 2), True, tau, np.float64, n_samples=16)
        assert res["sampled_c_tiles"] == 16 and res["absent_tiles_confirmed"] == 2
        assert res["task_set_equal"] and res["leaf_norms_bit_equal"] and res["rel_err_max"] <= 1e-12
        abi, abj, an, _ = A.export_leaves(tiles=False)
        bbi, bbj, bn, _ = B.export_leaves(tiles=False)
        cs, cnt = sc.flat_rule_checksum(abi, abj, an, bbi, bbj, bn, True, tau)
        assert cnt == nm and cs == Cg.task_checksum() and nr == Cg.get_n_blocks()
        return
    mats = []
    for seed in (1, 2):
        r, c, v = G.decay_coo(n, lam, W, seed)
        ref = po.from_coo(cls, b, n, n, r, c, v)
        del r, c, v
        g = HBSM(np.float64, b); g.generate_decay(n, lam, W, seed); g.update_internal_info()
        gi, gj, gn, gt = g.export_leaves()
        ri, rj, rn, rtiles = ref.leaves()
        assert np.array_equal(gi, ri) and np.array_equal(gj, rj)
        assert np.array_equal(gn, rn), "leaf norms differ from the reference's update_internal_info()"
        assert np.array_equal(gt, rtiles), "device generator and reference assembly disagree"
        del gt, rtiles
        mats.append((g, ref))
    Cg = HBSM(np.float64)
    nm, nr = HBSM.spamm(mats[0][0], 0, mats[1][0], 0, Cg, tau, True)
    Cr, rnm, rnb, rt = cls.product(mats[0][1], 0, mats[1][1], 0, spamm=True, tau=tau, want_tasks=True)
    assert (nm, nr) == (rnm, rnb)
    assert Cg.task_checksum() == G.task_checksum(rt[:, 0], rt[:, 1], rt[:, 2])
    assert np.array_equal(sort_tasks(Cg.export_tasks()), sort_tasks(rt))
    gi, gj, _, gt = Cg.export_leaves(norms=False)
    ri, rj, _, rtiles = Cr.leaves()
    assert np.array_equal(gi, ri) and np.array_equal(gj, rj)
    assert rel_frob(gt, rtiles) <= 1e-12
    per_tile = np.linalg.norm(gt - rtiles, axis=1) / np.maximum(np.linalg.norm(rtiles, axis=1), 1e-300)
    assert per_tile.max() <= 1e-11


def test_sampled_check_hooks_at_headline_size():
    """What bench.py --check runs: the N=65536 headline SpAMM, 12 sampled C tiles + 2 absent coordinates recomputed by the
    reference on the tile's own sub-problem (oracle/sampled_check.py), k-lists and leaf norms bit-exact, values <= 1e-12;
    and the flat-rule checksum over the exported leaf norms equals the device checksum of the executed set."""
    n, b, lam, tau = 65536, 64, 0.01, 1e-6
    W = G.decay_width(lam)
    A = HBSM(np.float64, b); A.generate_decay(n, lam, W, 1); A.update_internal_info()
    B = HBSM(np.float64, b); B.generate_decay(n, lam, W, 2); B.update_internal_info()
    C = HBSM(np.float64)
    nm, nr = HBSM.spamm(A, 0, B, 0, C, tau, True)
    res = sc.sampled_check(C, A, B, n, b, lam, W, (1, 2), True, tau, np.float64, n_samples=12)
    assert res["sampled_c_tiles"] == 12 and res["task_set_equal"] and res["leaf_norms_bit_equal"]
    assert res["leaf_norms_compared"] > 500 and res["absent_tiles_confirmed"] == 2
    assert res["rel_err_max"] <= 1e-12
    abi, abj, an, _ = A.export_leaves(tiles=False)
    bbi, bbj, bn, _ = B.export_leaves(tiles=False)
    cs, cnt = sc.flat_rule_checksum(abi, abj, an, bbi, bbj, bn, True, tau)
    assert cnt == nm and cs == C.task_checksum()


def test_spamm_updated_false_leaves_the_operands_untouched():
    """spamm(..., updated=false) prunes against FRESH leaf norms but does not write the operands' caches (the reference
    refreshes copies, H:3990-4005)."""
    n, b, lam, tau = 1024, 32, 0.05, 1e-4
    W = G.decay_width(lam)
    A = HBSM(np.float64, b); A.generate_decay(n, lam, W, 1)          # norms never refreshed: cache is all zero
    B = HBSM(np.float64, b); B.generate_decay(n, lam, W, 2)
    C0 = HBSM(np.float64)
    assert HBSM.spamm(A, 0, B, 0, C0, tau, True)[0] == 0                # stale (zero) norms prune everything
    C1 = HBSM(np.float64)
    nm1, _ = HBSM.spamm(A, 0, B, 0, C1, tau, False)
    assert nm1 > 0
    assert A.get_frob_norm_squared_internal() == 0.0 and not A.export_leaves(tiles=False)[2].any()
    assert not B.export_leaves(tiles=False)[2].any()
    A.update_internal_info(); B.update_internal_info()
    C2 = HBSM(np.float64)
    nm2, _ = HBSM.spamm(A, 0, B, 0, C2, tau, True)
    assert nm1 == nm2 and np.array_equal(C1.export_leaves()[3], C2.export_leaves()[3])


def test_products_from_two_host_threads():
    """The reference's multiply/spamm are re-entrant statics (H:255-305) called from a worker pool: two host threads run
    SpAMM products concurrently (each on its own engine stream), sharing one operand, and get the single-thread results."""
    n, b, lam, tau = 4096, 64, 0.03, 1e-6
    W = G.decay_width(lam)
    A = HBSM(np.float64, b); A.generate_decay(n, lam, W, 1); A.update_internal_info()
    Bs = []
    for s in (2, 3):
        Bm = HBSM(np.float64, b); Bm.generate_decay(n, lam, W, s); Bm.update_internal_info(); Bs.append(Bm)
    want = []
    for Bm in Bs:
        Cm = HBSM(np.float64); nm, nr = HBSM.spamm(A, 0, Bm, 1, Cm, tau, True)
        want.append((nm, nr, Cm.export_leaves()[3]))
    got = [None, None]
    errs = []

    def work(i):
        try:
            for _ in range(4):
                Cm = HBSM(np.float64)
                nm, nr = HBSM.spamm(A, 0, Bs[i], 1, Cm, tau, True)
                got[i] = (nm, nr, Cm.export_leaves()[3])
                del Cm
        except Exception as ex:   # noqa: BLE001
            errs.append(ex)

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs
    for i in range(2):
        assert got[i][0] == want[i][0] and got[i][1] == want[i][1] and np.array_equal(got[i][2], want[i][2])


def test_wire_format_rejects_a_malformed_tree():
    """assign_from_buffer (H:1348) on a buffer whose nodes do not have the shape the header implies: rejected, not misread."""
    A = HBSM(np.float64, 4); A.resize(14, 14)
    A.assign_from_vectors([0, 9], [0, 9], [1.0, 2.0]); A.update_internal_info()
    data = bytearray(A.write_to_buffer())
    B = HBSM(np.float64); B.assign_from_buffer(bytes(data))
    assert np.array_equal(B.to_dense(), A.to_dense())
    bad = bytearray(data)
    bad[0:4] = np.int32(8).tobytes()            # root nRows: 16 -> 8 (a level too shallow for these dims)
    with pytest.raises(hb.HbsmError):
        HBSM(np.float64).assign_from_buffer(bytes(bad))
    bad = bytearray(data)
    hdr = 5 * 4 + 8 + 8                          # child-size table of the root
    bad[hdr:hdr + 8] = np.uint64(2 ** 62).tobytes()
    with pytest.raises(hb.HbsmError):
        HBSM(np.float64).assign_from_buffer(bytes(bad))


@pytest.mark.parametrize("b", [32, 64])
@pytest.mark.parametrize("tA,tB", [(0, 0), (1, 1)])
def test_grouped_fp32_kernels_on_irregular_structure(b, tA, tB):
    """The 2x2-group tcgen05 kernels (k_gemm_f32_g32 / g64) on a random block structure, where a group's executed
    combinations at one k are often NOT a rectangle (three of four, diagonal pairs, single members, missing members): the
    super-product split must leave every C tile with exactly its own k-list.  Exact multiply (structural rule, H:1873) and
    SpAMM (per-leaf-pair prune, H:6649-6651) against the oracle, and against the single-C-tile tensor kernels (variant 3)."""
    dtype = np.float32
    n = 12 * b
    ra, ca, va = G.random_block_sparse_coo(n, b, 0.45, 11, dtype)
    rb, cb, vb = G.random_block_sparse_coo(n, b, 0.45, 12, dtype)
    scale = np.exp(-0.002 * np.abs(ra - ca)).astype(dtype); va = va * scale     # norms that differ from tile to tile: SpAMM prunes unevenly
    scale = np.exp(-0.002 * np.abs(rb - cb)).astype(dtype); vb = vb * scale
    g_a, o_a = both_from_coo(b, n, n, ra, ca, va, dtype)
    g_b, o_b = both_from_coo(b, n, n, rb, cb, vb, dtype)
    _, _, an, _ = o_a.leaves(tiles=False); _, _, bn, _ = o_b.leaves(tiles=False)
    tau = float(np.sqrt(np.median(an) * np.median(bn)))                          # about half of the structural products survive
    for spamm in (False, True):
        res = {}
        for variant in (0, 3):
            hb.set_gemm_variant(variant)
            try:
                Cg = HBSM(dtype)
                nm, nr = (HBSM.spamm(g_a, tA, g_b, tB, Cg, tau, True) if spamm else HBSM.multiply(g_a, tA, g_b, tB, Cg))
                assert hb.stage_times()["gemm_kernel"] == 3
                res[variant] = (nm, nr, Cg.export_tasks(), Cg.to_dense())
            finally:
                hb.set_gemm_variant(0)
        Cr, rnm, rnb, rt = po.OrcMatrix.product(o_a, tA, o_b, tB, spamm=spamm, tau=tau, want_tasks=True)
        if spamm:
            assert 0 < rnm < n_struct, "the prune must drop some but not all structural products"
        else:
            n_struct = rnm
        for variant in (0, 3):
            nm, nr, tasks, dense = res[variant]
            assert (nm, nr) == (rnm, rnb)
            assert np.array_equal(sort_tasks(tasks), sort_tasks(rt))
            assert rel_frob(dense, Cr.to_dense()) <= 1e-5
        assert rel_frob(res[0][3], res[3][3]) <= 3e-6
