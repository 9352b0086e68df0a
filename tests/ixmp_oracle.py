"""FAISS's IxMp (IndexIDMap) container restated in numpy, for the tests: write_index_header, the complete IxFI block of
the sub-index, then WRITEVECTOR(id_map) (u64 count, int64 ids).  Test infrastructure; the product never imports it."""
import numpy as np


def ixfi_bytes(x: np.ndarray) -> bytes:
    n, d = x.shape
    return (b"IxFI" + header_fields(d, n) + np.uint64(n * d).tobytes()
            + np.ascontiguousarray(x, dtype="<f4").tobytes())


def header_fields(d: int, ntotal: int, metric: int = 0) -> bytes:
    """faiss write_index_header after the fourcc: d, ntotal, two dummies of 1 << 20, is_trained, metric."""
    return (np.int32(d).tobytes() + np.int64(ntotal).tobytes() + np.int64(1 << 20).tobytes() * 2 + b"\x01"
            + np.int32(metric).tobytes())


def ixmp_bytes(x: np.ndarray, ids, sub: bytes = None) -> bytes:
    """The IxMp file of an IndexIDMap over an IndexFlatIP holding the rows x with the ids `ids`."""
    n, d = x.shape
    ids = np.ascontiguousarray(ids, dtype="<i8")
    return (b"IxMp" + header_fields(d, n) + (ixfi_bytes(x) if sub is None else sub) + np.uint64(ids.size).tobytes()
            + ids.tobytes())


def read_ixmp(data: bytes):
    """(rows float32 [n, d], ids int64 [n]) of an IxMp file over IxFI."""
    assert data[:4] == b"IxMp"
    d = int(np.frombuffer(data, np.int32, 1, 4)[0])
    n = int(np.frombuffer(data, np.int64, 1, 8)[0])
    p = 4 + 4 + 8 + 16 + 1 + 4
    assert data[p:p + 4] == b"IxFI"
    assert int(np.frombuffer(data, np.int32, 1, p + 4)[0]) == d and int(np.frombuffer(data, np.int64, 1, p + 8)[0]) == n
    q = p + 4 + 4 + 8 + 16 + 1 + 4
    assert int(np.frombuffer(data, np.uint64, 1, q)[0]) == n * d
    q += 8
    x = np.frombuffer(data, "<f4", n * d, q).reshape(n, d)
    q += 4 * n * d
    assert int(np.frombuffer(data, np.uint64, 1, q)[0]) == n
    ids = np.frombuffer(data, "<i8", n, q + 8)
    assert q + 8 + 8 * n == len(data)
    return x.copy(), ids.copy()
