"""IndexFlatIP.remove_ids without a GPU: argument normalisation in Python, and the piece plan of the in-place compaction
(kirag_debug_remove_plan) against a numpy restatement."""
import ctypes

import numpy as np
import pytest

from kirag_b200 import _lib, as_faiss, faiss_api


def test_selectors_and_id_arrays_are_normalised_like_faiss():
    assert faiss_api._id_array([[3, 1], [2, 7]]).tolist() == [3, 1, 2, 7]
    a = faiss_api._id_array(np.array([5, -1, 2], dtype=np.int32))
    assert a.dtype == np.int64 and a.flags.c_contiguous and a.tolist() == [5, -1, 2]
    assert faiss_api._id_array(np.arange(10, dtype=np.uint64)[::3]).tolist() == [0, 3, 6, 9]
    assert faiss_api._id_array(7).tolist() == [7]
    assert faiss_api._id_array([]).size == 0
    for bad in (None, "12", 1.5, [0.5, 1.0], object(), {"a": 1}, np.array([True, False])):
        with pytest.raises(AssertionError):
            faiss_api._id_array(bad)
    b = faiss_api.IDSelectorBatch([4, 4, 9])
    assert b.ids.dtype == np.int64 and b.ids.tolist() == [4, 4, 9]
    r = faiss_api.IDSelectorRange(np.int64(3), 10)
    assert (r.imin, r.imax) == (3, 10) and type(r.imin) is int
    mod = as_faiss.make_module()
    assert mod.IDSelectorBatch is faiss_api.IDSelectorBatch and mod.IDSelectorRange is faiss_api.IDSelectorRange


def test_remove_entry_points_check_their_arguments_without_a_gpu():
    lib = _lib.load()
    n = ctypes.c_int64(5)
    assert lib.kirag_index_remove_ids(None, None, 0, ctypes.byref(n), None) != 0 and "null index" in _lib.last_error()
    assert n.value == 5  # nothing written on a rejected call
    assert lib.kirag_index_remove_range(None, 0, 1, ctypes.byref(n), None) != 0 and "null index" in _lib.last_error()


def plan(kept, ntotal, first, G, d=64, budget=0):
    lib = _lib.load()
    kept = np.ascontiguousarray(kept, dtype=np.int32)
    summary = np.zeros(5, dtype=np.int64)
    rc = lib.kirag_debug_remove_plan(kept.ctypes.data, ntotal, first, G, d, budget, summary.ctypes.data, None, 0)
    assert rc == 0, _lib.last_error()
    pieces = np.zeros((max(int(summary[3]), 1), 4), dtype=np.int64)
    rc = lib.kirag_debug_remove_plan(kept.ctypes.data, ntotal, first, G, d, budget, summary.ctypes.data,
                                     pieces.ctypes.data, pieces.shape[0])
    assert rc == 0, _lib.last_error()
    return [int(v) for v in summary], pieces[: int(summary[3])]


def check_plan(removed_mask, G, d=64, budget=0):
    """The plan of one removal against the rows it has to move: ranks of the kept rows, pieces in order and within
    budget, rounds as piece boundaries, every source range covering its kept rows, and sources never below the rows
    already written (the in-place invariant)."""
    n = removed_mask.size
    ng = (n + 127) // 128
    padded = np.ones(ng * 128, dtype=bool)
    padded[:n] = removed_mask
    kept_counts = 128 - padded.reshape(ng, 128).sum(axis=1)
    first = int(np.argmax(removed_mask)) if removed_mask.any() else n
    (n_removed, j_start, n_new, n_pieces, bud), pieces = plan(kept_counts, n, first, G, d, budget)
    kept_rows = np.flatnonzero(~removed_mask)  # kept_rows[j] = old row of new row j
    assert n_removed == int(removed_mask.sum()) and n_new == kept_rows.size
    R = 128 * G
    assert bud % R == 0 and bud >= R
    if budget > 0:
        assert bud == budget
    if n_removed == 0:
        assert n_pieces == 0 and j_start == n
        return pieces
    assert j_start == first
    # rows below the first removed one are untouched: new row j is old row j there
    assert np.array_equal(kept_rows[:j_start], np.arange(j_start))
    assert np.all(kept_rows >= np.arange(n_new))  # rank(i) <= i
    if n_new == j_start:
        assert n_pieces == 0
        return pieces
    assert pieces[0, 0] == j_start and pieces[-1, 1] == n_new
    assert np.array_equal(pieces[1:, 0], pieces[:-1, 1])
    for j0, j1, i0, i1 in pieces:
        assert 0 < j1 - j0 <= bud
        assert j1 % R == 0 or j1 == n_new
        assert i0 % 128 == 0 and (i1 % 128 == 0 or i1 == n) and i0 < i1 <= n
        src = kept_rows[j0:j1]
        assert src[0] >= i0 and src[-1] < i1  # the source range holds every row the piece needs
        assert j1 <= i1                      # sources lie at or after the rows the piece writes
        assert src[0] >= j0                  # ... and after every row an earlier piece wrote
    # the next piece never reads what this one wrote
    for (j0, j1, _, _), (k0, k1, _, _) in zip(pieces[:-1], pieces[1:]):
        assert kept_rows[k0] >= j1
    return pieces


@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_plan_matches_numpy_restatement(G):
    rng = np.random.default_rng(G)
    for n in (1, 127, 128, 129, 5000, 70001):
        sels = {
            "row0": np.arange(n) == 0,
            "last": np.arange(n) == n - 1,
            "middle": np.arange(n) == n // 2,
            "tile": (np.arange(n) >= 256) & (np.arange(n) < 384),
            "cross": (np.arange(n) >= 100) & (np.arange(n) < 1000),
            "p1": rng.random(n) < 0.01,
            "p50": rng.random(n) < 0.5,
            "odd": np.arange(n) % 2 == 1,
            "all": np.ones(n, dtype=bool),
            "none": np.zeros(n, dtype=bool),
        }
        for name, mask in sels.items():
            for budget in (0, 128 * G, 384 * G):
                check_plan(mask, G, budget=budget)


def test_plan_pieces_follow_the_staging_budget():
    n = 1_000_000
    mask = np.zeros(n, dtype=bool)
    mask[0] = True
    pieces = check_plan(mask, 1, d=1024)
    # 64 MiB of fp32 rows of 1024 columns: 16384 rows per piece
    assert (pieces[:, 1] - pieces[:, 0]).max() == 16384 and len(pieces) == -(-(n - 1) // 16384)
    pieces = check_plan(mask, 8, d=1024)
    assert (pieces[:, 1] - pieces[:, 0]).max() == 16384
    mask[:] = False
    mask[-1] = True  # removing the last row moves nothing
    assert len(check_plan(mask, 1, d=1024)) == 0


def test_plan_rejects_bad_arguments():
    lib = _lib.load()
    summary = np.zeros(5, dtype=np.int64)
    kept = np.array([128, 200], dtype=np.int32)
    assert lib.kirag_debug_remove_plan(kept.ctypes.data, 256, 0, 1, 64, 0, summary.ctypes.data, None, 0) != 0
    assert "out of range" in _lib.last_error()
    kept = np.array([128, 127], dtype=np.int32)
    assert lib.kirag_debug_remove_plan(kept.ctypes.data, 256, 5, 1, 64, 0, summary.ctypes.data, None, 0) != 0
    assert "first removed row" in _lib.last_error()
    assert lib.kirag_debug_remove_plan(kept.ctypes.data, 256, 128, 2, 64, 128, summary.ctypes.data, None, 0) != 0
    assert "multiple" in _lib.last_error()
    assert lib.kirag_debug_remove_plan(kept.ctypes.data, 256, 128, 0, 64, 0, summary.ctypes.data, None, 0) != 0
