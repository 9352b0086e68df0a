"""Host-resident fp32 master: argument checks that need no GPU (they come before the device lookup)."""
import ctypes

import pytest

from kirag_b200 import _lib


def test_create_ex_rejects_unknown_flags_and_host_master_without_shadow():
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.kirag_index_create_ex(64, 0, 0, 2, ctypes.byref(h)) != 0 and h.value is None
    assert "unknown flag bits" in _lib.last_error()
    assert lib.kirag_index_create_ex(64, 0, 0, _lib.INDEX_HOST_MASTER | 8, ctypes.byref(h)) != 0
    assert "unknown flag bits" in _lib.last_error()
    assert lib.kirag_index_create_ex(100, 0, 0, _lib.INDEX_HOST_MASTER, ctypes.byref(h)) != 0 and h.value is None
    assert "host master needs the bf16 shadow" in _lib.last_error()
    # the older checks still come first
    assert lib.kirag_index_create_ex(0, 0, 0, _lib.INDEX_HOST_MASTER, ctypes.byref(h)) != 0
    assert "dimension" in _lib.last_error()


def test_load_ex_rejects_flags_before_reading_a_device(tmp_path):
    import numpy as np

    lib = _lib.load()
    path = tmp_path / "idx.faiss"
    # a valid IxFI header for d = 100, ntotal = 0
    hdr = (b"IxFI" + np.int32(100).tobytes() + np.int64(0).tobytes() + np.int64(1 << 20).tobytes() * 2 + b"\x01"
           + np.int32(0).tobytes() + np.uint64(0).tobytes())
    path.write_bytes(hdr)
    h = ctypes.c_void_p()
    assert lib.kirag_index_load_ex(str(path).encode(), 0, _lib.INDEX_HOST_MASTER, ctypes.byref(h)) != 0
    assert "host master needs the bf16 shadow" in _lib.last_error()
    assert lib.kirag_index_load_ex(str(path).encode(), 0, 4, ctypes.byref(h)) != 0
    assert "unknown flag bits" in _lib.last_error()


def test_python_master_argument_is_checked(monkeypatch):
    from kirag_b200 import faiss_api

    monkeypatch.delenv("KIRAG_MASTER", raising=False)
    with pytest.raises(AssertionError):
        faiss_api.IndexFlatIP(64, master="disk")
    with pytest.raises(AssertionError):
        faiss_api.read_index("/nonexistent.faiss", master="hbm")
    monkeypatch.setenv("KIRAG_MASTER", "bogus")
    with pytest.raises(AssertionError):
        faiss_api.IndexFlatIP(64)
    with pytest.raises(AssertionError):
        faiss_api.read_index("/nonexistent.faiss")
    assert faiss_api._master_flags("host") == _lib.INDEX_HOST_MASTER
    assert faiss_api._master_flags("device") == 0
    monkeypatch.setenv("KIRAG_MASTER", "host")
    assert faiss_api._master_flags(None) == _lib.INDEX_HOST_MASTER
    monkeypatch.delenv("KIRAG_MASTER")
    assert faiss_api._master_flags(None) == 0


def test_storage_bytes_needs_an_index():
    lib = _lib.load()
    dev, host = ctypes.c_int64(-1), ctypes.c_int64(-1)
    assert lib.kirag_index_storage_bytes(None, ctypes.byref(dev), ctypes.byref(host)) != 0
    assert "null index" in _lib.last_error()
