"""Multi-device index (IndexFlatIP(devices=[...])): argument checks that need no GPU, and the stripe arithmetic."""
import ctypes

import numpy as np
import pytest

from kirag_b200 import _lib


def test_create_multi_rejects_bad_arguments_before_any_device():
    lib = _lib.load()
    h = ctypes.c_void_p()
    devs = (ctypes.c_int * 2)(0, 0)
    assert lib.kirag_index_create_multi(64, 0, devs, 0, 0, ctypes.byref(h)) != 0 and h.value is None
    assert "empty device list" in _lib.last_error()
    assert lib.kirag_index_create_multi(64, 0, None, 2, 0, ctypes.byref(h)) != 0
    assert "empty device list" in _lib.last_error()
    assert lib.kirag_index_create_multi(64, 0, devs, 2, 2, ctypes.byref(h)) != 0 and h.value is None
    assert "unknown flag bits" in _lib.last_error()
    assert lib.kirag_index_create_multi(100, 0, devs, 2, _lib.INDEX_HOST_MASTER, ctypes.byref(h)) != 0
    assert "host master needs the bf16 shadow" in _lib.last_error()
    assert lib.kirag_index_create_multi(0, 0, devs, 2, 0, ctypes.byref(h)) != 0 and "dimension" in _lib.last_error()
    many = (ctypes.c_int * 17)(*([0] * 17))
    assert lib.kirag_index_create_multi(64, 0, many, 17, 0, ctypes.byref(h)) != 0 and "maximum" in _lib.last_error()
    assert lib.kirag_index_shards(None, None, None, 0) == -1 and "null index" in _lib.last_error()


def test_load_multi_checks_the_file_and_flags(tmp_path):
    lib = _lib.load()
    devs = (ctypes.c_int * 1)(0)
    h = ctypes.c_void_p()
    bad = tmp_path / "bad.faiss"
    bad.write_bytes(b"nope" + bytes(64))
    assert lib.kirag_index_load_multi(str(bad).encode(), devs, 1, 0, ctypes.byref(h)) != 0
    assert "not an IxFI" in _lib.last_error()
    path = tmp_path / "idx.faiss"
    path.write_bytes(b"IxFI" + np.int32(100).tobytes() + np.int64(0).tobytes() + np.int64(1 << 20).tobytes() * 2
                     + b"\x01" + np.int32(0).tobytes() + np.uint64(0).tobytes())
    assert lib.kirag_index_load_multi(str(path).encode(), devs, 1, _lib.INDEX_HOST_MASTER, ctypes.byref(h)) != 0
    assert "host master needs the bf16 shadow" in _lib.last_error()
    assert lib.kirag_index_load_multi(str(path).encode(), devs, 0, 0, ctypes.byref(h)) != 0
    assert "empty device list" in _lib.last_error()


def test_python_devices_argument_is_checked(monkeypatch):
    from kirag_b200 import faiss_api

    monkeypatch.delenv("KIRAG_DEVICES", raising=False)
    with pytest.raises(AssertionError):
        faiss_api.IndexFlatIP(64, devices=[])
    with pytest.raises(AssertionError):
        faiss_api.IndexFlatIP(64, device=0, devices=[0, 1])
    with pytest.raises(AssertionError):
        faiss_api.read_index("/nonexistent.faiss", device=0, devices=[0])
    assert faiss_api._resolve_devices(None, None) is None
    assert faiss_api._resolve_devices(3, None) is None
    assert faiss_api._resolve_devices(None, (0, 0, 1)) == [0, 0, 1]
    for bad in ("0,,1", "a", "0;1", "", "1,-2"):
        monkeypatch.setenv("KIRAG_DEVICES", bad)
        with pytest.raises(AssertionError):
            faiss_api.IndexFlatIP(64)
        with pytest.raises(AssertionError):
            faiss_api.read_index("/nonexistent.faiss")
    monkeypatch.setenv("KIRAG_DEVICES", "0,1,2,3,4,5,6,7")
    assert faiss_api._resolve_devices(None, None) == list(range(8))
    assert faiss_api._resolve_devices(2, None) is None  # an explicit device wins over the environment
    monkeypatch.setenv("KIRAG_DEVICES", " 1, 0 ")
    assert faiss_api._resolve_devices(None, None) == [1, 0]


def stripe_map(G, ids):
    ids = np.ascontiguousarray(ids, dtype=np.int64)
    shard = np.empty(len(ids), dtype=np.int32)
    local = np.empty(len(ids), dtype=np.int64)
    back = np.empty(len(ids), dtype=np.int64)
    assert _lib.load().kirag_debug_stripe_map(G, ids.ctypes.data, len(ids), shard.ctypes.data, local.ctypes.data,
                                              back.ctypes.data) == 0
    return shard, local, back


def stripe_rows(n, G):
    out = (ctypes.c_int64 * G)()
    assert _lib.load().kirag_debug_stripe_rows(n, G, out) == 0
    return list(out)


@pytest.mark.parametrize("G", [1, 2, 3, 8, 16])
def test_stripe_round_trip_and_layout(G):
    n = 128 * G * 5 + 77
    ids = np.arange(n, dtype=np.int64)
    shard, local, back = stripe_map(G, ids)
    assert np.array_equal(back, ids)
    assert np.array_equal(shard, (ids // 128) % G)
    assert np.array_equal(local, (ids // (128 * G)) * 128 + ids % 128)
    rows = stripe_rows(n, G)
    for s in range(G):
        mine = local[shard == s]
        # the rows of a shard are local rows 0..rows-1, in the order of their global ids
        assert np.array_equal(mine, np.arange(rows[s]))
    big = np.array([2**40 + 5, 2**33 * 3 + 127], dtype=np.int64)
    assert np.array_equal(stripe_map(G, big)[2], big)


@pytest.mark.parametrize("G", [2, 3, 8])
def test_stripe_balance_after_random_add_sequences(G):
    rng = np.random.default_rng(G)
    for _ in range(20):
        total = 0
        got = [0] * G
        for n in rng.choice([1, 7, 128, 1000, 100000, int(rng.integers(1, 5000))], size=12):
            before, after = stripe_rows(total, G), stripe_rows(total + int(n), G)
            assert all(a >= b for a, b in zip(after, before))
            got = [g + a - b for g, a, b in zip(got, after, before)]
            total += int(n)
            assert sum(got) == total
            assert max(got) - min(got) <= 128
            assert got[0] == max(got)  # the partial stripe at the end fills shard 0 first
        assert got == stripe_rows(total, G)
    assert stripe_rows(100, 8) == [100] + [0] * 7  # fewer rows than one stripe per shard: trailing shards empty


def test_stripe_hooks_reject_bad_arguments():
    lib = _lib.load()
    assert lib.kirag_debug_stripe_rows(10, 0, (ctypes.c_int64 * 1)()) != 0
    ids = np.array([-1], dtype=np.int64)
    assert lib.kirag_debug_stripe_map(2, ids.ctypes.data, 1, None, None, None) != 0
    assert "negative row" in _lib.last_error()
