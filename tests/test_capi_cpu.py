"""CPU tests of the drop-in boundary: the C-ABI library loads without a GPU, exports every symbol that
include/hbsm_b200.h declares (and nothing declared is missing from the ctypes table), handle bookkeeping that does
not touch the device works, and compute entry points FAIL LOUDLY (HBSM_E_CUDA) when no sm_100 device is present --
there is no CPU fallback."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from hierarchical_block_sparse_lib_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "hbsm_b200.h")


def declared_symbols():
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(hbsm_[a-z0-9_]+)\s*\(", txt)))


def have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_library_builds_and_loads():
    _capi.build()
    assert os.path.exists(_capi.LIB_PATH)
    assert _capi.lib() is not None


def test_every_declared_symbol_is_exported_and_bound():
    names = declared_symbols()
    assert len(names) >= 50
    lib = C.CDLL(_capi.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "libhbsm_b200.so does not export %s" % n
        assert n in _capi.SIGNATURES, "%s is declared in the header but missing from the ctypes table" % n
    extra = set(_capi.SIGNATURES) - set(names)
    assert not extra, "ctypes table binds undeclared symbols: %s" % sorted(extra)


def test_exports_are_c_abi_only():
    """Only extern "C" hbsm_* symbols are visible (-fvisibility=hidden): no C++/torch types cross the boundary."""
    out = subprocess.run(["nm", "-D", "--defined-only", _capi.LIB_PATH], capture_output=True, text=True).stdout
    syms = [l.split()[-1] for l in out.splitlines() if " T " in l]
    ours = [s for s in syms if s.startswith("hbsm_")]
    assert set(ours) == set(declared_symbols())
    assert not [s for s in syms if s.startswith("_Z") and "hbsm" in s]


def test_kernels_are_sm100a_only():
    out = subprocess.run(["cuobjdump", "--list-elf", _capi.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_handle_bookkeeping_without_device():
    L = _capi.lib()
    h = C.c_void_p()
    assert L.hbsm_create(_capi.HBSM_F64, C.byref(h)) == 0
    v = C.c_int(-1)
    assert L.hbsm_is_empty(h, C.byref(v)) == 0 and v.value == 1
    assert L.hbsm_set_blocksize(h, 64) == 0
    assert L.hbsm_get_blocksize(h, C.byref(v)) == 0 and v.value == 64
    assert L.hbsm_expected_depth(h, C.byref(v)) == 0
    assert L.hbsm_create(7, C.byref(C.c_void_p())) == _capi.HBSM_E_ARG
    assert b"dtype" in L.hbsm_last_error()
    assert L.hbsm_destroy(h) == 0
    assert L.hbsm_morton_encode(0b101, 0b011) == 0b011011   # digit = 2*colbit + rowbit (H:52-56), MSB first
    r = C.c_uint32(); c = C.c_uint32()
    L.hbsm_morton_decode(0b011011, C.byref(r), C.byref(c))
    assert (r.value, c.value) == (0b101, 0b011)


def test_gemm_variant_accepts_only_the_existing_kernels():
    """0 (tensor-core kernels), 1 (generic FMA) and 3 (fp32 single-C-tile) select leaf kernels; anything else is refused."""
    L = _capi.lib()
    try:
        for v in (0, 1, 3):
            assert L.hbsm_set_gemm_variant(v) == 0, v
        for v in (2, 4, -1):
            assert L.hbsm_set_gemm_variant(v) == _capi.HBSM_E_ARG, v
            assert b"variant" in L.hbsm_last_error()
    finally:
        assert L.hbsm_set_gemm_variant(0) == 0


@pytest.mark.skipif(have_gpu(), reason="a GPU is present: the loud-failure path cannot be exercised")
def test_compute_fails_loudly_without_gpu():
    L = _capi.lib()
    assert L.hbsm_init(0) == _capi.HBSM_E_CUDA
    assert b"no CPU fallback" in L.hbsm_last_error() or b"CUDA" in L.hbsm_last_error()
    h = C.c_void_p()
    L.hbsm_create(_capi.HBSM_F64, C.byref(h))
    L.hbsm_set_blocksize(h, 4)
    assert L.hbsm_resize(h, 16, 16) == _capi.HBSM_E_CUDA
    import hierarchical_block_sparse_lib_b200 as hb
    with pytest.raises(hb.HbsmError):
        A = hb.HierarchicalBlockSparseMatrix(np.float64, 4)
        A.resize(16, 16)
        A.assign_from_vectors([0], [0], [1.0])
    L.hbsm_destroy(h)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "hierarchical_block_sparse_lib_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")) or f == "Makefile":
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), os.path.join(dp, f)
                assert "oracle/" not in txt.replace("never imports oracle/", ""), os.path.join(dp, f)
