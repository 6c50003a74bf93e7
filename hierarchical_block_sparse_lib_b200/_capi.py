"""ctypes binding of the C ABI in include/hbsm_b200.h (libhbsm_b200.so, built in-tree by csrc/Makefile).

There is no CPU fallback: loading fails loudly when the library has not been built, and every compute call
fails with HBSM_E_CUDA when no sm_100 device is usable.
"""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libhbsm_b200.so")
CSRC = os.path.join(HERE, "csrc")

HBSM_F64, HBSM_F32 = 0, 1
HBSM_OK, HBSM_E_CUDA, HBSM_E_ARG, HBSM_E_RUNTIME = 0, 1, 2, 3
HBSM_OP_N, HBSM_OP_T, HBSM_OP_SYM_UPPER = 0, 1, 2


class StageTimes(C.Structure):
    _fields_ = [("norms_ms", C.c_double), ("index_ms", C.c_double), ("tasklist_ms", C.c_double),
                ("gemm_ms", C.c_double), ("total_ms", C.c_double), ("n_candidates", C.c_uint64),
                ("n_products", C.c_uint64), ("n_ctiles", C.c_uint64), ("gpu_launches", C.c_uint64),
                ("gemm_kernel", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class TruncInfo(C.Structure):
    """hbsm_trunc_info"""
    _fields_ = [("n_dropped", C.c_size_t), ("drop_nsq", C.c_double), ("n_frob", C.c_size_t), ("err_bound", C.c_double),
                ("certified_by_lanczos", C.c_int), ("n_decisions", C.c_int), ("lanczos_steps", C.c_longlong)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_H = C.c_void_p
_sz = C.c_size_t
_P = C.c_void_p
_I = C.c_int

# name -> (restype, argtypes); every symbol include/hbsm_b200.h declares
SIGNATURES = {
    "hbsm_init": (_I, [_I]),
    "hbsm_finalize": (_I, []),
    "hbsm_last_error": (C.c_char_p, []),
    "hbsm_device_info": (_I, [C.c_char_p, _sz, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "hbsm_kernel_launch_count": (C.c_uint64, []),
    "hbsm_create": (_I, [_I, C.POINTER(_H)]),
    "hbsm_destroy": (_I, [_H]),
    "hbsm_set_blocksize": (_I, [_H, _I]),
    "hbsm_get_blocksize": (_I, [_H, C.POINTER(_I)]),
    "hbsm_resize": (_I, [_H, _I, _I]),
    "hbsm_clear": (_I, [_H]),
    "hbsm_is_empty": (_I, [_H, C.POINTER(_I)]),
    "hbsm_children_exist": (_I, [_H, C.POINTER(_I)]),
    "hbsm_dims": (_I, [_H, C.POINTER(_I), C.POINTER(_I)]),
    "hbsm_depth": (_I, [_H, C.POINTER(_I)]),
    "hbsm_expected_depth": (_I, [_H, C.POINTER(_I)]),
    "hbsm_is_consistent": (_I, [_H, C.POINTER(_I)]),
    "hbsm_dtype": (_I, [_H, C.POINTER(_I)]),
    "hbsm_assign_coo": (_I, [_H, _sz, _P, _P, _P, _I, _I]),
    "hbsm_assign_tiles": (_I, [_H, _sz, _P, _P, _P]),
    "hbsm_get_values": (_I, [_H, _sz, _P, _P, _P]),
    "hbsm_get_all_values": (_I, [_H, _sz, _P, _P, _P, C.POINTER(_sz)]),
    "hbsm_export_tile": (_I, [_H, _I, _I, _P, C.POINTER(_I)]),
    "hbsm_nnz": (_I, [_H, C.POINTER(_sz)]),
    "hbsm_n_blocks": (_I, [_H, C.POINTER(_sz)]),
    "hbsm_get_n_block_multiplications": (_I, [_H, C.POINTER(_sz)]),
    "hbsm_set_n_block_multiplications": (_I, [_H, _sz]),
    "hbsm_update_norms": (_I, [_H]),
    "hbsm_frob_squared": (_I, [_H, _P]),
    "hbsm_frob_squared_cached": (_I, [_H, _P]),
    "hbsm_multiply": (_I, [_H, _I, _H, _I, _H, C.POINTER(_sz), C.POINTER(_sz)]),
    "hbsm_spamm": (_I, [_H, _I, _H, _I, _H, C.c_double, _I, C.POINTER(_sz), C.POINTER(_sz)]),
    "hbsm_product_begin": (_I, [_H, _I, _H, _I, _H, _I, C.c_double, _I, _I]),
    "hbsm_product_finish": (_I, [_H, _P, C.POINTER(_sz), C.POINTER(_sz)]),
    "hbsm_product_abort": (_I, []),
    "hbsm_product_begin_ex": (_I, [_H, _I, _H, _I, _H, _I, C.c_double, _I, _I, _I]),
    "hbsm_product_to_host": (_I, [_H, _I, _H, _I, _H, _I, C.c_double, _I, _P, _sz, C.POINTER(_sz), C.POINTER(_sz)]),
    "hbsm_product_from_host": (_I, [_H, _sz, _P, _P, _P, _I, _H, _sz, _P, _P, _P, _I, _H, _I, C.c_double, _I, _P, _sz, _P, _P,
                                    C.POINTER(_sz), C.POINTER(_sz)]),
    "hbsm_worth_to_multiply": (_I, [_H, _I, _H, _I, C.POINTER(_I)]),
    "hbsm_worth_to_spamm": (_I, [_H, _I, _H, _I, C.c_double, C.POINTER(_I)]),
    "hbsm_add": (_I, [_H, _H, _H]),
    "hbsm_transpose": (_I, [_H, _H]),
    "hbsm_upper_triangle": (_I, [_H, _H]),
    "hbsm_rescale": (_I, [_H, _H, C.c_double]),
    "hbsm_copy": (_I, [_H, _H]),
    "hbsm_frob_block_trunc": (_I, [_H, _H, C.c_double, C.POINTER(_I)]),
    "hbsm_leaf_norms": (_I, [_H, _sz, _P, C.POINTER(_sz)]),
    "hbsm_extract_quadrant": (_I, [_H, _I, _H, C.POINTER(_I)]),
    "hbsm_assemble_quadrants": (_I, [_H, _I, _I, _H, _H, _H, _H]),
    "hbsm_count_skips": (_I, [_H, _I, _H, _I, _sz, _P, _I, _I, _P]),
    "hbsm_spamm_errors": (_I, [_H, _I, _H, _I, _sz, _P, _P, C.POINTER(_sz)]),
    "hbsm_serialized_size": (_I, [_H, C.POINTER(_sz)]),
    "hbsm_serialize": (_I, [_H, _P, _sz]),
    "hbsm_deserialize": (_I, [_H, _P, _sz]),
    "hbsm_symm_multiply": (_I, [_H, _I, _H, _I, _H]),
    "hbsm_symm_square": (_I, [_H, _H]),
    "hbsm_symm_rk": (_I, [_H, _I, _H]),
    "hbsm_symm_square_spamm": (_I, [_H, _H, C.c_double, C.POINTER(_sz), C.POINTER(_sz)]),
    "hbsm_multiply_dense": (_I, [_H, _I, _I, _P, _I, _P, _I, C.c_double, C.c_double]),
    "hbsm_multiply_dense_device": (_I, [_H, _I, _I, _P, _I, _P, _I, C.c_double, C.c_double, _P]),
    "hbsm_spectral_norm": (_I, [_H, _I, _I, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                               C.POINTER(_I)]),
    "hbsm_spectral_block_trunc": (_I, [_H, _I, C.c_double, _I, _H, C.POINTER(TruncInfo)]),
    "hbsm_truncation_spectral_errors": (_I, [_H, _I, _sz, _P, _I, C.c_double, _P, _P]),
    "hbsm_export_tasks": (_I, [_H, _sz, _P, _P, _P, C.POINTER(_sz)]),
    "hbsm_export_leaves": (_I, [_H, _sz, _P, _P, _P, _P, C.POINTER(_sz)]),
    "hbsm_task_checksum": (_I, [_H, C.POINTER(C.c_uint64)]),
    "hbsm_export_tile_tasks": (_I, [_H, _I, _I, _sz, _P, C.POINTER(_sz), C.POINTER(_I)]),
    "hbsm_stage_times_last": (_I, [C.POINTER(StageTimes)]),
    "hbsm_set_gemm_variant": (_I, [_I]),
    "hbsm_device_table": (_I, [_H, C.POINTER(_sz), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P)]),
    "hbsm_assign_device_tiles": (_I, [_H, _sz, _P, _P, _P]),
    "hbsm_halo_reserve": (_I, [_H, _sz, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P)]),
    "hbsm_halo_commit": (_I, [_H, _sz]),
    "hbsm_leaf_inv_chol": (_I, [_H, _H, _I, _I]),
    "hbsm_comm_set_library": (_I, [C.c_char_p]),
    "hbsm_comm_unique_id": (_I, [_P]),
    "hbsm_comm_init": (_I, [_P, _I, _I]),
    "hbsm_comm_finalize": (_I, []),
    "hbsm_comm_info": (_I, [C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "hbsm_comm_barrier": (_I, []),
    "hbsm_comm_allreduce_f64": (_I, [C.POINTER(C.c_double), _I, _I]),
    "hbsm_comm_allgather_u64": (_I, [C.POINTER(C.c_uint64), _sz, C.POINTER(C.c_uint64)]),
    "hbsm_shard_rows": (_I, [_I, _I, _I, C.POINTER(_I), C.POINTER(_I)]),
    "hbsm_shard_rows_balanced": (_I, [C.POINTER(C.c_uint64), _I, _I, C.POINTER(_I)]),
    "hbsm_publish": (_I, [_H]),
    "hbsm_sharded_product": (_I, [_H, _I, _H, _I, _H, _I, C.c_double, _I, C.POINTER(_sz), C.POINTER(_sz)]),
    "hbsm_sharded_row_weights": (_I, [_H, _I, _H, _I, _I, C.c_double, _I, _I, _P]),
    "hbsm_shard_stats_last": (_I, [_P]),
    "hbsm_generate_decay": (_I, [_H, _I, _P, _I, C.c_uint64, _I, _I, _I]),
    "hbsm_morton_encode": (C.c_uint64, [C.c_uint32, C.c_uint32]),
    "hbsm_morton_decode": (None, [C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "hbsm_stream": (C.c_void_p, []),
}

_lib = None


def build(verbose=False):
    """Compile csrc/*.cu for sm_100a into lib/libhbsm_b200.so (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-s", "-j", str(min(8, os.cpu_count() or 1)), "-C", CSRC], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libhbsm_b200.so failed:\n%s\n%s" % (r.stdout, r.stderr))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)   # AttributeError here = the library does not export a declared symbol
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


class HbsmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


def check(rc):
    if rc != HBSM_OK:
        raise HbsmError(rc, lib().hbsm_last_error().decode(errors="replace"))
