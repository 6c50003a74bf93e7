"""CPU tests (-m "not gpu") that PIN the oracle: the plain-C restatement (oracle/hbsm_oracle_impl.h) is checked
(1) against the reference's own known-answer tests (tests/known_answers.py, TO:/TC: citations),
(2) against the unmodified reference compiled in place (oracle/_ref) on seeded inputs, where that library exists,
(3) against the committed fixtures tests/golden/*.npz, which were generated from oracle/_ref by
    tests/golden/make_golden.py and travel to machines without /root/reference."""
import glob
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from hierarchical_block_sparse_lib_b200 import generators as G
import known_answers
import golden_cases
from helpers import OracleBackend, sort_tasks, rel_frob

HAVE_REF = os.path.exists(po.REF_SO)
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref not built (no /root/reference on this machine)")


@pytest.fixture(scope="module", autouse=True)
def _built(oracle_built):
    return oracle_built


def test_known_answers_oracle_port():
    assert known_answers.run_all(OracleBackend(po.OrcMatrix)) >= 30


@needs_ref
def test_known_answers_unmodified_reference():
    """The restated goldens are the reference's: its own code must reproduce them through our harness."""
    assert known_answers.run_all(OracleBackend(po.RefMatrix)) >= 30


@pytest.mark.parametrize("case", golden_cases.CASES, ids=[c["id"] for c in golden_cases.CASES])
def test_oracle_port_matches_golden_fixture(case):
    path = os.path.join(golden_cases.GOLDEN_DIR, case["id"] + ".npz")
    assert os.path.exists(path), "missing fixture %s: run tests/golden/make_golden.py where /root/reference exists" % path
    want = dict(np.load(path))
    if case.get("needs_serialize"):
        pytest.skip("the wire format is checked engine-vs-reference (fixture bytes come from the reference's own writer)")
    got = golden_cases.run_case(OracleBackend(po.OrcMatrix, case["dtype"]), case)
    golden_cases.compare(got, want, case)


@needs_ref
@pytest.mark.parametrize("case", golden_cases.CASES, ids=[c["id"] for c in golden_cases.CASES])
def test_golden_fixture_is_current(case):
    """Fixtures are outputs of the reference itself: regenerate in memory and compare bit for bit."""
    want = dict(np.load(os.path.join(golden_cases.GOLDEN_DIR, case["id"] + ".npz")))
    got = golden_cases.run_case(OracleBackend(po.RefMatrix, case["dtype"]), case)
    for k in want:
        assert np.array_equal(got[k], want[k]), k


@needs_ref
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("tA,tB", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_port_vs_reference_random_block_sparse(dtype, tA, tB):
    """cfg-1 law at reduced size: exact multiply and SpAMM task sets are bit-identical, values within tolerance."""
    n, b = 256, 16
    ra, ca, va = G.random_block_sparse_coo(n, b, 0.3, 1, dtype)
    rb, cb, vb = G.random_block_sparse_coo(n, b, 0.3, 2, dtype)
    tol = 1e-12 if dtype == np.float64 else 1e-5
    o = [po.from_coo(po.OrcMatrix, b, n, n, r, c, v, dtype) for r, c, v in ((ra, ca, va), (rb, cb, vb))]
    f = [po.from_coo(po.RefMatrix, b, n, n, r, c, v, dtype) for r, c, v in ((ra, ca, va), (rb, cb, vb))]
    for i in range(2):   # leaf norms bit-exact (H:646-652) and root norm
        assert np.array_equal(o[i].leaves(False)[2], f[i].leaves(False)[2])
        assert o[i].frob_sq_cached() == f[i].frob_sq_cached()
    for spamm, tau in ((False, 0.0), (True, 80.0), (True, 88.0)):
        Co, onm, onb, ot = po.OrcMatrix.product(o[0], tA, o[1], tB, spamm=spamm, tau=tau, want_tasks=True)
        Cf, fnm, fnb, ft = po.RefMatrix.product(f[0], tA, f[1], tB, spamm=spamm, tau=tau, want_tasks=True)
        assert (onm, onb) == (fnm, fnb)
        assert np.array_equal(sort_tasks(ot), sort_tasks(ft))
        assert rel_frob(Co.to_dense(), Cf.to_dense()) <= tol
        assert po.OrcMatrix.worth(o[0], tA, o[1], tB, spamm, tau) == po.RefMatrix.worth(f[0], tA, f[1], tB, spamm, tau)
    assert 0 < onm < po.OrcMatrix.product(o[0], tA, o[1], tB)[1]   # tau = 88 really prunes


@needs_ref
@pytest.mark.parametrize("n,b", [(1000, 32), (300, 7), (512, 64)])
def test_port_vs_reference_decay_spamm(n, b):
    W = min(G.decay_width(0.05), n - 1)
    ins = [G.decay_coo(n, 0.05, W, s) for s in (1, 2)]
    o = [po.from_coo(po.OrcMatrix, b, n, n, *x) for x in ins]
    f = [po.from_coo(po.RefMatrix, b, n, n, *x) for x in ins]
    for tau in (1e-8, 1e-4, 1e-2):
        for tA, tB in ((0, 0), (1, 0)):
            Co, onm, onb, ot = po.OrcMatrix.product(o[0], tA, o[1], tB, spamm=True, tau=tau, want_tasks=True)
            Cf, fnm, fnb, ft = po.RefMatrix.product(f[0], tA, f[1], tB, spamm=True, tau=tau, want_tasks=True)
            assert (onm, onb) == (fnm, fnb)
            assert np.array_equal(sort_tasks(ot), sort_tasks(ft))
            assert rel_frob(Co.to_dense(), Cf.to_dense()) <= 1e-12


@needs_ref
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_port_vs_reference_structure_and_symmetric(dtype):
    n, b = 200, 16
    W = G.decay_width(0.1)
    r, c, v = G.decay_coo(n, 0.1, W, 3, symmetric=True, dtype=dtype)
    up = r <= c
    rb, cb, vb = G.decay_coo(n, 0.1, W, 4, dtype=dtype)
    tol = 1e-12 if dtype == np.float64 else 2e-5
    for cls_pair in [(po.OrcMatrix, po.RefMatrix)]:
        O, F = cls_pair
        ou, fu = (po.from_coo(k, b, n, n, r[up], c[up], v[up], dtype) for k in (O, F))
        ob, fb = (po.from_coo(k, b, n, n, rb, cb, vb, dtype) for k in (O, F))
        assert np.array_equal(O.add(ou, ob).to_dense(), F.add(fu, fb).to_dense())
        assert np.array_equal(O.transpose(ob).to_dense(), F.transpose(fb).to_dense())
        assert np.array_equal(O.upper(ob).to_dense(), F.upper(fb).to_dense())
        assert np.array_equal(O.rescale(ob, 0.3).to_dense(), F.rescale(fb, 0.3).to_dense())
        assert rel_frob(O.symm_square(ou).to_dense(), F.symm_square(fu).to_dense()) <= tol
        assert rel_frob(O.symm_multiply(ou, 1, ob, 0).to_dense(), F.symm_multiply(fu, 1, fb, 0).to_dense()) <= tol
        assert rel_frob(O.symm_multiply(ob, 0, ou, 1).to_dense(), F.symm_multiply(fb, 0, fu, 1).to_dense()) <= tol
        for tr in (0, 1):
            assert rel_frob(O.symm_rk(ob, tr).to_dense(), F.symm_rk(fb, tr).to_dense()) <= tol
        ga = O.add(ou, ob); fa = F.add(fu, fb)
        assert np.array_equal(ga.leaves(False)[0], fa.leaves(False)[0]) and np.array_equal(ga.leaves(False)[1], fa.leaves(False)[1])


def test_flat_rule_equals_hierarchical_rule_on_port():
    """SURVEY 0.3: the hierarchical norm test collapses to the flat leaf-pair rule fl(nsqA*nsqB) > fl(tau*tau)."""
    n, b = 512, 16
    W = G.decay_width(0.08)
    A = po.from_coo(po.OrcMatrix, b, n, n, *G.decay_coo(n, 0.08, W, 1))
    B = po.from_coo(po.OrcMatrix, b, n, n, *G.decay_coo(n, 0.08, W, 2))
    abi, abj, an, _ = A.leaves(False); bbi, bbj, bn, _ = B.leaves(False)
    for tau in (1e-9, 1e-5, 1e-3, 0.1):
        _, nm, _, t = po.OrcMatrix.product(A, 0, B, 0, spamm=True, tau=tau, want_tasks=True)
        flat = [(i, j, k) for i, k, na in zip(abi, abj, an) for kk, j, nb in zip(bbi, bbj, bn)
                if kk == k and na * nb > np.float64(tau) * np.float64(tau)]
        assert np.array_equal(sort_tasks(t), sort_tasks(np.array(flat).reshape(-1, 3)))


@pytest.mark.parametrize("dtype,spamm,tau", [(np.float64, True, 1e-4), (np.float64, False, 0.0), (np.float32, True, 1e-3)])
def test_single_tile_subproblem_is_the_full_products_tile(dtype, spamm, tau):
    """oracle/sampled_check.reference_tile (block row of A times block column of B, run through the checker bench.py
    --check uses: the unmodified reference where oracle/_ref is built, else the pinned port) gives, for every sampled
    C tile, exactly the k-list and the values of that tile in the checker's FULL product -- the property bench.py
    --check and the full-size GPU tests rely on."""
    from oracle import sampled_check as sc
    K = sc.checker_class()
    n, b, lam = 1024, 32, 0.08
    W = min(G.decay_width(lam), n - 1)
    (ra, ca, va) = G.decay_coo(n, lam, W, 1, dtype=dtype)
    (rb, cb, vb) = G.decay_coo(n, lam, W, 2, dtype=dtype)
    A = po.from_coo(K, b, n, n, ra, ca, va, dtype)
    B = po.from_coo(K, b, n, n, rb, cb, vb, dtype)
    Cf, nm, nb, tasks = K.product(A, 0, B, 0, spamm=spamm, tau=tau, want_tasks=True)
    D = Cf.to_dense()
    cbi, cbj, _, _ = Cf.leaves(tiles=False)
    abi, abj, an, _ = A.leaves(tiles=False)
    have = set(zip(cbi.tolist(), cbj.tolist()))
    rng = np.random.default_rng(3)
    for t in [0, len(cbi) - 1] + list(rng.integers(0, len(cbi), 6)):
        ci, cj = int(cbi[t]), int(cbj[t])
        ks, tile, a_n, b_n = sc.reference_tile(K, n, b, lam, W, (1, 2), ci, cj, spamm, tau, dtype)
        want = np.sort(tasks[(tasks[:, 0] == ci) & (tasks[:, 1] == cj), 2])
        assert np.array_equal(ks, want)
        want_tile = D[ci * b:(ci + 1) * b, cj * b:(cj + 1) * b].astype(np.float64)
        assert tile is not None
        assert np.linalg.norm(tile - want_tile) <= (1e-6 if dtype == np.float32 else 1e-14) * np.linalg.norm(want_tile)
        for k, v in a_n.items():       # same leaves => bit-identical leaf norms
            assert v == an[(abi == ci) & (abj == k)][0]
    if spamm:                          # a coordinate outside C's structure: nothing executed in the sub-problem either
        ci = int(cbi[len(cbi) // 2])
        cj = max(j for (i, j) in have if i == ci) + 1
        if cj < n // b:
            ks, tile, _, _ = sc.reference_tile(K, n, b, lam, W, (1, 2), ci, cj, spamm, tau, dtype)
            assert len(ks) == 0
    # the flat-rule checksum over the reference's leaf norms equals the checksum of the reference's executed set
    bbi, bbj, bn, _ = B.leaves(tiles=False)
    cs, cnt = sc.flat_rule_checksum(abi, abj, an, bbi, bbj, bn, spamm, tau, dtype)
    assert cnt == nm and cs == G.task_checksum(tasks[:, 0], tasks[:, 1], tasks[:, 2])
