import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import hierarchical_block_sparse_lib_b200 as hb
from hierarchical_block_sparse_lib_b200 import generators as G
H = hb.HierarchicalBlockSparseMatrix
hb.init(0)
for b, n, lam in ((64, 16384, 0.01), (128, 16384, 0.01), (32, 8192, 0.02)):
    W = G.decay_width(lam)
    A = H(np.float32, b); A.generate_decay(n, lam, W, 1); A.update_internal_info()
    B = H(np.float32, b); B.generate_decay(n, lam, W, 2); B.update_internal_info()
    for it in range(3):
        C = H(np.float32); nm, nr = H.spamm(A, 0, B, 0, C, 1e-6, True); st = hb.stage_times(); del C
    print("b", b, "gemm_ms %.3f" % st["gemm_ms"], "TF %.1f" % (2.0 * b ** 3 * nm / st["gemm_ms"] / 1e9), flush=True)
