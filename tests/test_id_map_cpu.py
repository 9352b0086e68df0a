"""IndexIDMap without a GPU: flag and argument checks that come before any device is looked at, Python id
normalisation, the load errors of crafted IxMp files, and the test-side IxMp writer / reader."""
import ctypes

import numpy as np
import pytest

from kirag_b200 import _lib, as_faiss, faiss_api
from tests import ixmp_oracle


def test_id_map_flag_is_known_and_checked_before_the_device():
    lib = _lib.load()
    h = ctypes.c_void_p()
    for flags in (_lib.INDEX_ID_MAP, _lib.INDEX_ID_MAP | _lib.INDEX_HOST_MASTER):
        assert lib.kirag_index_create_ex(64, 0, 0, flags, ctypes.byref(h)) != 0 and h.value is None
        assert "unknown flag bits" not in _lib.last_error()
    assert lib.kirag_index_create_ex(64, 0, 0, _lib.INDEX_ID_MAP | 32, ctypes.byref(h)) != 0
    assert "unknown flag bits 0x20" in _lib.last_error()
    assert lib.kirag_index_create_ex(100, 0, 0, _lib.INDEX_ID_MAP | _lib.INDEX_HOST_MASTER, ctypes.byref(h)) != 0
    assert "host master needs the bf16 shadow" in _lib.last_error()
    devs = (ctypes.c_int * 2)(0, 0)
    assert lib.kirag_index_create_multi(64, 0, devs, 2, _lib.INDEX_ID_MAP | 64, ctypes.byref(h)) != 0
    assert "unknown flag bits 0x40" in _lib.last_error()


def test_entry_points_reject_null_handles():
    lib = _lib.load()
    n = ctypes.c_int64(5)
    x = np.zeros((1, 64), np.float32)
    ids = np.zeros(1, np.int64)
    assert lib.kirag_index_add_with_ids(None, x.ctypes.data, ids.ctypes.data, 1, 0, None) != 0
    assert "null index" in _lib.last_error()
    assert lib.kirag_index_remove_ids_ex(None, ids.ctypes.data, 1, 0, ctypes.byref(n), None) != 0
    assert "null index" in _lib.last_error() and n.value == 5
    assert lib.kirag_index_id_map(None, 0, 1, ids.ctypes.data, 0, None) != 0 and "null argument" in _lib.last_error()
    assert lib.kirag_index_flags(None) == -1 and "null index" in _lib.last_error()


def test_add_with_ids_arguments_are_normalised_like_faiss():
    x, ids = faiss_api._id_pairs([[1, 2], [3, 4]], np.array([7, -9], dtype=np.int32), 2)
    assert x.dtype == np.float32 and ids.dtype == np.int64 and ids.tolist() == [7, -9] and ids.flags.c_contiguous
    x, ids = faiss_api._id_pairs(np.zeros((3, 2), np.float64), np.arange(6, dtype=np.uint64)[::2], 2)
    assert ids.tolist() == [0, 2, 4] and x.dtype == np.float32
    with pytest.raises(AssertionError, match="not same nb of vectors as ids"):
        faiss_api._id_pairs(np.zeros((3, 2)), [1, 2], 2)
    with pytest.raises(AssertionError, match="not same nb of vectors as ids"):
        faiss_api._id_pairs(np.zeros((2, 2)), [[1], [2]], 2)
    with pytest.raises(AssertionError, match="dimension"):
        faiss_api._id_pairs(np.zeros((2, 3)), [1, 2], 2)
    with pytest.raises(AssertionError):
        faiss_api._id_pairs(np.zeros(4), [1, 2, 3, 4], 2)


def test_as_faiss_exports_the_id_map_surface():
    mod = as_faiss.make_module()
    assert mod.IndexIDMap is faiss_api.IndexIDMap and mod.vector_to_array is faiss_api.vector_to_array
    v = np.arange(4, dtype=np.int64)
    out = mod.vector_to_array(v)
    assert out.tolist() == [0, 1, 2, 3] and out is not v


def test_ixmp_oracle_round_trips():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((37, 12)).astype(np.float32)
    ids = rng.integers(-(1 << 62), 1 << 62, 37)
    ids[5] = ids[9]
    data = ixmp_oracle.ixmp_bytes(x, ids)
    x2, ids2 = ixmp_oracle.read_ixmp(data)
    assert np.array_equal(x2.view(np.uint32), x.view(np.uint32)) and np.array_equal(ids2, ids)
    # the embedded block is the IxFI file of the rows
    p = 4 + 4 + 8 + 16 + 1 + 4
    assert data[p:p + len(ixmp_oracle.ixfi_bytes(x))] == ixmp_oracle.ixfi_bytes(x)
    assert len(data) == p + len(ixmp_oracle.ixfi_bytes(x)) + 8 + 8 * 37


def load_error(path, flags=0, multi=False):
    lib = _lib.load()
    h = ctypes.c_void_p()
    if multi:
        devs = (ctypes.c_int * 2)(0, 0)
        rc = lib.kirag_index_load_multi(str(path).encode(), devs, 2, flags, ctypes.byref(h))
    else:
        rc = lib.kirag_index_load_ex(str(path).encode(), 0, flags, ctypes.byref(h))
    assert rc != 0 and h.value is None
    return _lib.last_error()


@pytest.mark.parametrize("multi", [False, True])
def test_load_reports_every_header_error_before_the_device(tmp_path, multi):
    x = np.ones((3, 8), np.float32)
    ids = np.array([5, -1, 5], np.int64)
    good = ixmp_oracle.ixmp_bytes(x, ids)
    cases = {
        "ixm2": (b"IxM2" + good[4:], "IndexIDMap2 file (IxM2), which is not supported"),
        "sub": (ixmp_oracle.ixmp_bytes(x, ids, sub=b"IxHf" + ixmp_oracle.ixfi_bytes(x)[4:]),
                "is not an IxFI (IndexFlatIP) block (fourcc 0x66487849)"),
        "sub_disagrees": (b"IxMp" + ixmp_oracle.header_fields(8, 4) + good[37:],
                          "the IxMp header (d=8 ntotal=4) and its IxFI block (d=8 ntotal=3) disagree"),
        "short_count": (good[:-32] + np.uint64(2).tobytes() + ids[:2].tobytes(), "holds 2 ids for 3 rows"),
        "short_ids": (good[:-8], "has 202 bytes; an IxMp file of 3 rows x 8 has 210"),
        "long": (good + b"\0", "has 211 bytes; an IxMp file of 3 rows x 8 has 210"),
        "no_ids": (good[:-32], "truncated: no id vector after the 3 rows"),
        "metric": (b"IxMp" + ixmp_oracle.header_fields(8, 3, metric=1) + good[37:], "inconsistent IxMp header"),
    }
    assert len(good) == 37 + 141 + 8 + 24
    for name, (data, msg) in cases.items():
        p = tmp_path / f"{name}.faiss"
        p.write_bytes(data)
        err = load_error(p, multi=multi)
        assert msg in err, (name, err)
        assert "device" not in err.lower(), (name, err)
    # the id-map flag is never a load flag, even on a good file
    p = tmp_path / "good.faiss"
    p.write_bytes(good)
    assert "KIRAG_INDEX_ID_MAP is not a load flag" in load_error(p, _lib.INDEX_ID_MAP, multi=multi)
    # a good file reaches the device lookup (here: there is none, or it answers)
    if _lib.load().kirag_device_count() == 0:
        assert "no CUDA device" in load_error(p, multi=multi)


def test_python_id_map_requires_a_flat_index():
    with pytest.raises(AssertionError):
        faiss_api.IndexIDMap(object())
