"""The C-ABI library: builds for sm_100a, loads without a GPU, exports every declared symbol, fails loudly."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from kirag_b200 import _build, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "kirag_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(kirag_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_table_agree():
    decl = declared_symbols()
    assert len(decl) >= 20
    assert sorted(_lib.SIGNATURES) == decl


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    assert lib.kirag_abi_version() == _lib.ABI_VERSION
    for name in declared_symbols():
        assert hasattr(lib, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", _build.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (kirag_[a-z0-9_]+)", out))
    assert exported == set(declared_symbols())


def test_built_for_sm100a_with_tcgen05_and_tma():
    cuobjdump = os.path.join(os.path.dirname(_build.find_nvcc()), "cuobjdump")  # the toolkit that built the library
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    elf = subprocess.run([cuobjdump, "-lelf", _build.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in elf
    sass = subprocess.run([cuobjdump, "-sass", _build.LIB_PATH], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass      # tcgen05.mma
    assert "LDTM" in sass         # tcgen05.ld
    assert "UBLKCP" in sass       # cp.async.bulk (TMA engine)


def test_no_gpu_means_loud_failure_not_fallback():
    lib = _lib.load()
    if lib.kirag_device_count() > 0:
        pytest.skip("a GPU is visible")
    h = ctypes.c_void_p()
    rc = lib.kirag_index_create(64, 0, 0, ctypes.byref(h))
    assert rc != 0 and h.value is None
    assert "no CUDA device" in _lib.last_error() and "no CPU path" in _lib.last_error()
    from kirag_b200 import IndexFlatIP

    with pytest.raises(RuntimeError):
        IndexFlatIP(64)


def test_argument_validation_without_gpu():
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.kirag_index_create(0, 0, 0, ctypes.byref(h)) != 0 and "dimension" in _lib.last_error()
    assert lib.kirag_index_create(64, 1, 0, ctypes.byref(h)) != 0 and "inner-product" in _lib.last_error()
    D = np.zeros(4, dtype=np.float32)
    I = np.zeros(4, dtype=np.int64)
    assert lib.kirag_index_search(None, None, 1, 4, D.ctypes.data, I.ctypes.data, 0, 0, None) != 0
    assert "null index" in _lib.last_error()
    assert lib.kirag_index_ntotal(None) == -1
    assert lib.kirag_merge_topk(None, None, 0, 1, 1, None, None, 0, 0, None) != 0


def test_product_package_never_imports_the_oracle():
    """The product path must not route through oracle/ (or any CPU fallback)."""
    pkg = os.path.join(ROOT, "kirag_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "liboracle" not in src, f
