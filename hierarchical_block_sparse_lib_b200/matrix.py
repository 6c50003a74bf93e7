"""Python mirror of the reference's ``hbsm::HierarchicalBlockSparseMatrix<Treal>`` public interface
(reference source/HierarchicalBlockSparseMatrix.h:166-428) over the C ABI.  Same method names, argument meaning
and error behaviour (the reference's exception text arrives as ``HbsmError``), so the parity tests read like the
reference's own tests.  The C++ drop-in for the same interface is include/hbsm/HierarchicalBlockSparseMatrix.h.
"""
import ctypes as C
import numpy as np

from . import _capi
from ._capi import check, lib, HbsmError, StageTimes  # noqa: F401

_DT = {np.dtype(np.float64): _capi.HBSM_F64, np.dtype(np.float32): _capi.HBSM_F32}


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Params:
    def __init__(self, blocksize=-1):
        self.blocksize = blocksize


class HierarchicalBlockSparseMatrix:
    def __init__(self, dtype=np.float64, blocksize=None):
        self.dtype = np.dtype(dtype)
        self._h = C.c_void_p()
        check(lib().hbsm_create(_DT[self.dtype], C.byref(self._h)))
        if blocksize is not None:
            p = Params(blocksize)
            self.set_params(p)

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                lib().hbsm_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    # ---- sizing (H:181-196) ----
    def _int(self, fn):
        v = C.c_int(0)
        check(getattr(lib(), fn)(self._h, C.byref(v)))
        return v.value

    def _size(self, fn):
        v = C.c_size_t(0)
        check(getattr(lib(), fn)(self._h, C.byref(v)))
        return v.value

    def get_n_rows(self):
        r = C.c_int(0); c = C.c_int(0)
        check(lib().hbsm_dims(self._h, C.byref(r), C.byref(c)))
        return r.value

    def get_n_cols(self):
        r = C.c_int(0); c = C.c_int(0)
        check(lib().hbsm_dims(self._h, C.byref(r), C.byref(c)))
        return c.value

    def set_params(self, params):
        check(lib().hbsm_set_blocksize(self._h, int(params.blocksize)))

    def get_params(self):
        return Params(self._int("hbsm_get_blocksize"))

    def children_exist(self): return bool(self._int("hbsm_children_exist"))
    def empty(self): return bool(self._int("hbsm_is_empty"))
    def resize(self, n_rows, n_cols): check(lib().hbsm_resize(self._h, int(n_rows), int(n_cols)))
    def clear(self): check(lib().hbsm_clear(self._h))
    def get_depth(self): return self._int("hbsm_depth")
    def expected_depth(self): return self._int("hbsm_expected_depth")
    def check_if_matrix_is_consistent(self): return bool(self._int("hbsm_is_consistent"))
    def get_n_blocks(self): return self._size("hbsm_n_blocks")
    def get_n_block_multiplications(self): return self._size("hbsm_get_n_block_multiplications")
    def set_n_block_multiplicaitons(self, n): check(lib().hbsm_set_n_block_multiplications(self._h, int(n)))  # sic, H:220

    # ---- assembly / readback (H:198-239) ----
    def assign_from_vectors_general(self, rows, cols, values, useMax, boundaries_checked):
        if len(rows) != len(values) or len(cols) != len(values):
            raise HbsmError(_capi.HBSM_E_RUNTIME,
                            "Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: bad sizes.")  # H:677
        r = np.ascontiguousarray(rows, np.int32); c = np.ascontiguousarray(cols, np.int32)
        v = np.ascontiguousarray(values, self.dtype)
        check(lib().hbsm_assign_coo(self._h, len(v), _ptr(r), _ptr(c), _ptr(v), int(bool(useMax)),
                                    int(bool(boundaries_checked))))

    def assign_from_vectors(self, rows, cols, values):
        self.assign_from_vectors_general(rows, cols, values, False, False)

    def assign_from_vectors_max(self, rows, cols, values):
        self.assign_from_vectors_general(rows, cols, values, True, False)

    def assign_tiles(self, bi, bj, tiles):
        """Bulk path: whole column-major tiles at block coordinates (bi[t], bj[t])."""
        bi = np.ascontiguousarray(bi, np.int32); bj = np.ascontiguousarray(bj, np.int32)
        t = np.ascontiguousarray(tiles, self.dtype)
        check(lib().hbsm_assign_tiles(self._h, len(bi), _ptr(bi), _ptr(bj), _ptr(t)))

    def get_values(self, rows, cols):
        if len(rows) != len(cols):
            raise HbsmError(_capi.HBSM_E_RUNTIME, "Error in HierarchicalBlockSparseMatrix<Treal>::get_values: bad sizes.")
        r = np.ascontiguousarray(rows, np.int32); c = np.ascontiguousarray(cols, np.int32)
        out = np.zeros(len(r), self.dtype)
        check(lib().hbsm_get_values(self._h, len(r), _ptr(r), _ptr(c), _ptr(out)))
        return out

    def get_all_values(self):
        n = C.c_size_t(0)
        check(lib().hbsm_get_all_values(self._h, 0, None, None, None, C.byref(n)))
        r = np.zeros(n.value, np.int32); c = np.zeros(n.value, np.int32); v = np.zeros(n.value, self.dtype)
        if n.value:
            check(lib().hbsm_get_all_values(self._h, n.value, _ptr(r), _ptr(c), _ptr(v), C.byref(n)))
        return r, c, v

    def get_nnz(self): return self._size("hbsm_nnz")

    # ---- norms (H:214-223) ----
    def _real(self, fn):
        out = np.zeros(1, self.dtype)
        check(getattr(lib(), fn)(self._h, _ptr(out)))
        return out[0]

    def get_frob_squared(self): return self._real("hbsm_frob_squared")
    def get_frob_norm_squared_internal(self): return self._real("hbsm_frob_squared_cached")
    def update_internal_info(self): check(lib().hbsm_update_norms(self._h))

    # ---- operations ----
    def copy(self, other): check(lib().hbsm_copy(self._h, other._h))
    def rescale(self, other, alpha): check(lib().hbsm_rescale(self._h, other._h, float(alpha)))
    def get_upper_triangle(self, A): check(lib().hbsm_upper_triangle(self._h, A._h))

    @staticmethod
    def add(A, B, Cm):
        check(lib().hbsm_add(A._h, B._h, Cm._h))

    @staticmethod
    def multiply(A, tA, B, tB, Cm):
        """Returns (no_of_block_multiplies, no_of_resizes) -- the reference's two optional out-parameters (H:260)."""
        nm = C.c_size_t(0); nr = C.c_size_t(0)
        check(lib().hbsm_multiply(A._h, int(bool(tA)), B._h, int(bool(tB)), Cm._h, C.byref(nm), C.byref(nr)))
        return nm.value, nr.value

    @staticmethod
    def spamm(A, tA, B, tB, Cm, tau, updated=True):
        nm = C.c_size_t(0); nr = C.c_size_t(0)
        check(lib().hbsm_spamm(A._h, int(bool(tA)), B._h, int(bool(tB)), Cm._h, float(tau), int(bool(updated)),
                               C.byref(nm), C.byref(nr)))
        return nm.value, nr.value

    @staticmethod
    def multiply_accumulate(A, tA, B, tB, Cm, alpha, beta):
        """Cm <- alpha*op(A)*op(B) + beta*Cm in one call (hbsm_multiply_accumulate); Cm may be A and/or B, or unsized.
        Returns (n_mults, n_resizes): the leaf products executed and Cm's tile count."""
        nm = C.c_size_t(0); nr = C.c_size_t(0)
        check(lib().hbsm_multiply_accumulate(A._h, int(bool(tA)), B._h, int(bool(tB)), Cm._h, float(alpha), float(beta), 0, 0.0, 1,
                                             C.byref(nm), C.byref(nr)))
        return nm.value, nr.value

    @staticmethod
    def spamm_accumulate(A, tA, B, tB, Cm, alpha, beta, tau, updated=True):
        """Cm <- alpha*spamm(op(A), op(B), tau) + beta*Cm in one call, otherwise as multiply_accumulate."""
        nm = C.c_size_t(0); nr = C.c_size_t(0)
        check(lib().hbsm_multiply_accumulate(A._h, int(bool(tA)), B._h, int(bool(tB)), Cm._h, float(alpha), float(beta), 1, float(tau),
                                             int(bool(updated)), C.byref(nm), C.byref(nr)))
        return nm.value, nr.value

    @staticmethod
    def product_from_host(A, a_bi, a_bj, a_tiles, tA, B, b_bi, b_bj, b_tiles, tB, Cm, spamm=False, tau=0.0, out_tiles=None,
                          n_slabs=0):
        """Host-to-host multiply / SpAMM as one pipeline (hbsm_product_from_host): A and B are sized, tile-less matrices
        that end up assembled with fresh norms, Cm receives the product; `out_tiles` (numpy, [cap, b*b], ideally a view of
        pinned memory) receives C's tiles.  Returns (n_mults, n_blocks, c_bi, c_bj) with the coordinates of out_tiles' rows."""
        a_bi = np.ascontiguousarray(a_bi, np.int32); a_bj = np.ascontiguousarray(a_bj, np.int32)
        b_bi = np.ascontiguousarray(b_bi, np.int32); b_bj = np.ascontiguousarray(b_bj, np.int32)
        at = np.ascontiguousarray(a_tiles, A.dtype); bt = np.ascontiguousarray(b_tiles, B.dtype)
        cap = 0 if out_tiles is None else out_tiles.shape[0]
        cbi = np.zeros(max(cap, 1), np.int32); cbj = np.zeros(max(cap, 1), np.int32)
        nm = C.c_size_t(0); nr = C.c_size_t(0)
        check(lib().hbsm_product_from_host(A._h, len(a_bi), _ptr(a_bi), _ptr(a_bj), _ptr(at), int(bool(tA)),
                                           B._h, len(b_bi), _ptr(b_bi), _ptr(b_bj), _ptr(bt), int(bool(tB)),
                                           Cm._h, int(bool(spamm)), float(tau), int(n_slabs),
                                           None if out_tiles is None else _ptr(out_tiles), cap,
                                           _ptr(cbi) if cap else None, _ptr(cbj) if cap else None, C.byref(nm), C.byref(nr)))
        return nm.value, nr.value, cbi[:nr.value], cbj[:nr.value]

    @staticmethod
    def worth_to_multiply(A, tA, B, tB):
        v = C.c_int(0)
        check(lib().hbsm_worth_to_multiply(A._h, int(bool(tA)), B._h, int(bool(tB)), C.byref(v)))
        return bool(v.value)

    @staticmethod
    def worth_to_spamm(A, tA, B, tB, tau):
        v = C.c_int(0)
        check(lib().hbsm_worth_to_spamm(A._h, int(bool(tA)), B._h, int(bool(tB)), float(tau), C.byref(v)))
        return bool(v.value)

    @staticmethod
    def symm_multiply(A, sA, B, sB, Cm):
        check(lib().hbsm_symm_multiply(A._h, int(bool(sA)), B._h, int(bool(sB)), Cm._h))

    @staticmethod
    def symm_square(A, Cm):
        check(lib().hbsm_symm_square(A._h, Cm._h))

    @staticmethod
    def symm_rk(A, transposed, Cm):
        check(lib().hbsm_symm_rk(A._h, int(bool(transposed)), Cm._h))

    @staticmethod
    def symm_square_spamm(A, Cm, tau):
        nm = C.c_size_t(0); nr = C.c_size_t(0)
        check(lib().hbsm_symm_square_spamm(A._h, Cm._h, float(tau), C.byref(nm), C.byref(nr)))
        return nm.value, nr.value

    @staticmethod
    def transpose(A, Cm):
        check(lib().hbsm_transpose(A._h, Cm._h))

    @staticmethod
    def count_skips(A, tA, B, tB, taus, apply_truncation, apply_spamm):
        t = np.ascontiguousarray(taus, np.float64); out = np.zeros(len(t), np.uint64)
        check(lib().hbsm_count_skips(A._h, int(bool(tA)), B._h, int(bool(tB)), len(t), _ptr(t), int(bool(apply_truncation)),
                                     int(bool(apply_spamm)), _ptr(out)))
        return out

    @staticmethod
    def get_spamm_errors(A, tA, B, tB, taus):
        t = np.ascontiguousarray(taus, np.float64); out = np.zeros(len(t), np.float64); n = C.c_size_t(0)
        check(lib().hbsm_spamm_errors(A._h, int(bool(tA)), B._h, int(bool(tB)), len(t), _ptr(t), _ptr(out), C.byref(n)))
        return out[:n.value].astype(A.dtype)

    # ---- engine extras: SpAMM with error control (hbsm_spamm_error_bounds / hbsm_spamm_tau_for_error) ----
    @staticmethod
    def spamm_error_bounds(A, tA, B, tB, taus, updated=True, symm_square=False):
        """For each tau, a rigorous bound on ||P_exact - P_tau||_F (hence ||.||_2) of spamm(A, tA, B, tB, tau, updated) --
        or, with symm_square, of symm_square_spamm(A, tau) on sym(triu(.)) -- and the leaf pairs it skips.  The leaf GEMMs'
        own rounding is not included.  Returns (bounds float64, n_skipped uint64) numpy arrays."""
        t = np.ascontiguousarray(np.atleast_1d(np.asarray(taus, np.float64)))
        out = np.zeros(len(t), np.float64)
        ns = np.zeros(len(t), np.uint64)
        check(lib().hbsm_spamm_error_bounds(A._h, int(bool(tA)), B._h, int(bool(tB)), int(bool(symm_square)), int(bool(updated)),
                                            len(t), _ptr(t), _ptr(out), _ptr(ns)))
        return out, ns

    @staticmethod
    def spamm_tau_for_error(A, tA, B, tB, eps, updated=True, symm_square=False):
        """The largest-skipping tau whose bound (spamm_error_bounds) is <= eps.  Returns the hbsm_spamm_tol_info as a dict:
        tau, bound, level (the largest skipped norm^2 product, -1 when nothing is skipped), n_candidates, n_skipped,
        n_levels."""
        info = _capi.SpammTolInfo()
        check(lib().hbsm_spamm_tau_for_error(A._h, int(bool(tA)), B._h, int(bool(tB)), int(bool(symm_square)), int(bool(updated)),
                                             float(eps), C.byref(info)))
        return info.as_dict()

    def get_size(self):
        return self._size("hbsm_serialized_size")

    def write_to_buffer(self):
        """H:1159: the reference's wire format as bytes."""
        n = self.get_size()
        buf = np.zeros(n, np.uint8)
        check(lib().hbsm_serialize(self._h, _ptr(buf), n))
        return buf.tobytes()

    def assign_from_buffer(self, data):
        buf = np.frombuffer(bytes(data), np.uint8)
        check(lib().hbsm_deserialize(self._h, _ptr(buf), len(buf)))

    def frob_block_trunc(self, matrix_truncated, trunc_value):
        """H:4935: matrix_truncated = copy of self without the blocks of Frobenius norm < trunc_value; True if any was removed."""
        r = C.c_int(0)
        check(lib().hbsm_frob_block_trunc(self._h, matrix_truncated._h, float(trunc_value), C.byref(r)))
        return bool(r.value)

    # ---- parity / bench hooks ----
    def export_tasks(self):
        """Executed products of the call that produced this matrix, as an (n,3) int64 array of (ci, cj, k),
        sorted by (Morton key of the C tile, k)."""
        n = C.c_size_t(0)
        check(lib().hbsm_export_tasks(self._h, 0, None, None, None, C.byref(n)))
        ci = np.zeros(n.value, np.int64); cj = np.zeros(n.value, np.int64); k = np.zeros(n.value, np.int64)
        if n.value:
            check(lib().hbsm_export_tasks(self._h, n.value, _ptr(ci), _ptr(cj), _ptr(k), C.byref(n)))
        return np.stack([ci, cj, k], 1)

    def task_checksum(self):
        """Order-independent checksum of the executed-product set: sum of splitmix64(ci<<42 | cj<<21 | k) mod 2^64."""
        v = C.c_uint64(0)
        check(lib().hbsm_task_checksum(self._h, C.byref(v)))
        return int(v.value)

    def tile_tasks(self, bi, bj):
        """The k's (ascending) of the products accumulated into tile (bi, bj) of this product result; None if absent."""
        n = C.c_size_t(0); found = C.c_int(0)
        check(lib().hbsm_export_tile_tasks(self._h, int(bi), int(bj), 0, None, C.byref(n), C.byref(found)))
        if not found.value:
            return None
        k = np.zeros(n.value, np.int64)
        if n.value:
            check(lib().hbsm_export_tile_tasks(self._h, int(bi), int(bj), n.value, _ptr(k), C.byref(n), C.byref(found)))
        return k

    def export_leaves(self, tiles=True, norms=True):
        n = self.get_n_blocks()
        b = self.get_params().blocksize
        bi = np.zeros(n, np.int64); bj = np.zeros(n, np.int64)
        nrm = np.zeros(n, self.dtype) if norms else None
        t = np.zeros((n, b * b), self.dtype) if tiles else None
        m = C.c_size_t(0)
        if n:
            check(lib().hbsm_export_leaves(self._h, n, _ptr(bi), _ptr(bj), _ptr(nrm), _ptr(t), C.byref(m)))
        return bi, bj, nrm, t

    def get_tile(self, bi, bj):
        """Dense b x b block at block coordinates (bi, bj) as a (row, col) array; None if the tile does not exist."""
        b = self.get_params().blocksize
        buf = np.zeros(b * b, self.dtype)
        found = C.c_int(0)
        check(lib().hbsm_export_tile(self._h, int(bi), int(bj), _ptr(buf), C.byref(found)))
        return buf.reshape(b, b).T.copy() if found.value else None

    def to_dense(self):
        m, n = self.get_n_rows(), self.get_n_cols()
        b = self.get_params().blocksize
        bi, bj, _, t = self.export_leaves(norms=False)
        g = max(1, -(-max(m, n) // b))
        out = np.zeros((g * b + b, g * b + b), self.dtype)
        for i in range(len(bi)):
            out[bi[i] * b:(bi[i] + 1) * b, bj[i] * b:(bj[i] + 1) * b] = t[i].reshape(b, b).T
        return out[:m, :n]

    def generate_decay(self, n, lam, W, seed, symmetric=False, row_tile_lo=0, row_tile_hi=-1):
        table = decay_table(lam, W)
        check(lib().hbsm_generate_decay(self._h, int(n), _ptr(table), int(W), int(seed), int(bool(symmetric)),
                                        int(row_tile_lo), int(row_tile_hi)))

    # ---- engine extras: block-sparse times dense multivector, spectral estimates ----
    def multiply_dense(self, X, op="N", alpha=1.0, beta=0.0, Y=None):
        """Y = alpha * op(A) * X + beta * Y with op "N" (A), "T" (A^T) or "SYM_UPPER" (triu(A) + striu(A)^T); returns Y.

        X and Y are 1-D or 2-D, column-major with unit stride along dim 0 (any column stride >= the row count: it becomes
        the leading dimension).  numpy X of another layout or dtype is copied into a Fortran-ordered array; numpy Y must
        already have that layout and A's dtype, as it is written in place.  torch CUDA tensors of A's dtype and that layout
        run on the device, ordered on torch.cuda.current_stream(), without copies; other CUDA layouts are refused."""
        ops = {"N": _capi.HBSM_OP_N, "T": _capi.HBSM_OP_T, "SYM_UPPER": _capi.HBSM_OP_SYM_UPPER}
        if op not in ops:
            raise ValueError("multiply_dense: op must be one of %s" % sorted(ops))
        o = ops[op]
        M = self.get_n_cols() if o == _capi.HBSM_OP_T else self.get_n_rows()
        K = self.get_n_rows() if o == _capi.HBSM_OP_T else self.get_n_cols()
        if type(X).__module__.startswith("torch") and X.is_cuda:
            return self._multiply_dense_torch(o, M, K, X, float(alpha), float(beta), Y)
        vec = np.ndim(X) == 1
        X = np.asarray(X)
        if not _column_major(X, self.dtype):
            X = np.asfortranarray(X, dtype=self.dtype)
        m = 1 if vec else X.shape[1]
        if X.shape[0] != K:
            raise ValueError("multiply_dense: X has %d rows, op(A) has %d columns" % (X.shape[0], K))
        if Y is None:
            Y = np.zeros(M if vec else (M, m), self.dtype, order="F")
        elif not isinstance(Y, np.ndarray) or not _column_major(Y, self.dtype):
            raise ValueError("multiply_dense: Y must be a %s array with unit stride along dim 0" % self.dtype)
        if Y.shape[0] != M or (Y.shape[1] if Y.ndim == 2 else 1) != m:
            raise ValueError("multiply_dense: Y has shape %s, expected (%d, %d)" % (Y.shape, M, m))
        check(lib().hbsm_multiply_dense(self._h, o, m, _ptr(X), _ld(X, K), _ptr(Y), _ld(Y, M), float(alpha), float(beta)))
        return Y

    def _multiply_dense_torch(self, o, M, K, X, alpha, beta, Y):
        import torch
        tdt = {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32}[self.dtype]

        def ok(t):
            return t.is_cuda and t.dtype == tdt and t.dim() in (1, 2) and (t.shape[0] <= 1 or t.stride(0) == 1)
        if not ok(X):
            raise ValueError("multiply_dense: a CUDA X must be a 1-D or 2-D %s tensor with unit stride along dim 0 (got %s, "
                             "strides %s); it is never copied" % (tdt, X.dtype, tuple(X.stride())))
        m = 1 if X.dim() == 1 else X.shape[1]
        if X.shape[0] != K:
            raise ValueError("multiply_dense: X has %d rows, op(A) has %d columns" % (X.shape[0], K))
        if Y is None:
            Y = torch.zeros(M, device=X.device, dtype=tdt) if X.dim() == 1 else \
                torch.zeros((m, M), device=X.device, dtype=tdt).t()
        elif not (type(Y).__module__.startswith("torch") and ok(Y)):
            raise ValueError("multiply_dense: with a CUDA X, Y must be a CUDA %s tensor with unit stride along dim 0" % tdt)
        if Y.shape[0] != M or (Y.shape[1] if Y.dim() == 2 else 1) != m:
            raise ValueError("multiply_dense: Y has shape %s, expected (%d, %d)" % (tuple(Y.shape), M, m))
        ldx = max(1, K) if X.dim() == 1 or m <= 1 else X.stride(1)
        ldy = max(1, M) if Y.dim() == 1 or m <= 1 else Y.stride(1)
        stream = torch.cuda.current_stream(X.device).cuda_stream
        check(lib().hbsm_multiply_dense_device(self._h, o, m, C.c_void_p(X.data_ptr()), int(ldx), C.c_void_p(Y.data_ptr()),
                                               int(ldy), alpha, beta, C.c_void_p(stream)))
        return Y

    def spectral_norm_estimate(self, symmetric_upper=False, max_iter=200, rel_tol=1e-8):
        """||A||_2 by Lanczos, on A^T A or (symmetric_upper) on triu(A) + striu(A)^T.  Returns (norm, lambda_min,
        lambda_max, n_iter): the extreme Ritz values of the operator Lanczos ran on -- the eigenvalue bounds of
        triu(A) + striu(A)^T with symmetric_upper, those of A^T A (squared singular values) without, as in the C ABI."""
        nrm = C.c_double(0); lo = C.c_double(0); hi = C.c_double(0); it = C.c_int(0)
        check(lib().hbsm_spectral_norm(self._h, int(bool(symmetric_upper)), int(max_iter), float(rel_tol), C.byref(nrm),
                                       C.byref(lo), C.byref(hi), C.byref(it)))
        return nrm.value, lo.value, hi.value, it.value

    # ---- engine extras: truncation with spectral-norm error control ----
    def spectral_block_trunc(self, matrix_truncated, eps, symmetric_upper=False, max_iter=100):
        """matrix_truncated = self without the leaves of the largest nsq level v (leaf ||.||_F^2) whose error E_v -- the
        dropped leaves, or triu(E_v) + striu(E_v)^T with symmetric_upper -- the search accepts with ||E_v||_2 <= eps.  The
        result equals frob_block_trunc at any tau with v < tau^2 <= the next level.  Returns the hbsm_trunc_info as a dict:
        n_dropped, drop_nsq (-1 when nothing is dropped), n_frob, err_bound, certified_by_lanczos, n_decisions,
        lanczos_steps.  Acceptance beyond the Frobenius bound is a Lanczos estimate (see include/hbsm_b200.h)."""
        info = _capi.TruncInfo()
        check(lib().hbsm_spectral_block_trunc(self._h, int(bool(symmetric_upper)), float(eps), int(max_iter), matrix_truncated._h,
                                              C.byref(info)))
        d = info.as_dict()
        d["certified_by_lanczos"] = bool(d["certified_by_lanczos"])
        return d

    def truncation_spectral_errors(self, taus, symmetric_upper=False, max_iter=200, rel_tol=1e-8):
        """For each tau, the Lanczos estimate of ||E_tau||_2, E_tau = the leaves frob_block_trunc(tau) would drop (triu +
        striu^T with symmetric_upper), exactly as spectral_norm_estimate reports it for a matrix of E_tau's tiles.  Returns
        (norms float64, n_iter int32) numpy arrays."""
        t = np.ascontiguousarray(np.atleast_1d(np.asarray(taus, np.float64)))
        out = np.zeros(len(t), np.float64)
        its = np.zeros(len(t), np.int32)
        check(lib().hbsm_truncation_spectral_errors(self._h, int(bool(symmetric_upper)), len(t), _ptr(t), int(max_iter),
                                                    float(rel_tol), _ptr(out), _ptr(its)))
        return out, its


def _column_major(a, dtype):
    """numpy array usable in place: the dtype, 1-D or 2-D, unit stride along dim 0, column stride a multiple of the item size."""
    if a.dtype != dtype or a.ndim not in (1, 2):
        return False
    s = a.itemsize
    if a.shape[0] > 1 and a.strides[0] != s:
        return False
    return a.ndim == 1 or a.shape[1] <= 1 or (a.strides[1] % s == 0 and a.strides[1] >= s * max(1, a.shape[0]))


def _ld(a, rows):
    if a.ndim == 1 or a.shape[1] <= 1:
        return max(1, rows)
    return a.strides[1] // a.itemsize


def decay_table(lam, W):
    return np.ascontiguousarray(np.exp(-float(lam) * np.arange(W + 1, dtype=np.float64)))


def stage_times():
    st = StageTimes()
    check(lib().hbsm_stage_times_last(C.byref(st)))
    return st.as_dict()


def set_gemm_variant(v):
    check(lib().hbsm_set_gemm_variant(int(v)))


def init(device=0):
    check(lib().hbsm_init(int(device)))


def kernel_launch_count():
    return int(lib().hbsm_kernel_launch_count())


def device_info():
    name = C.create_string_buffer(256)
    sm = C.c_int(0); ma = C.c_int(0); mi = C.c_int(0)
    check(lib().hbsm_device_info(name, 256, C.byref(sm), C.byref(ma), C.byref(mi)))
    return {"name": name.value.decode(), "sm_count": sm.value, "cc": (ma.value, mi.value)}
