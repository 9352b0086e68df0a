"""IndexFlatIP.remove_ids on the B200.  Every case removes rows from an index A and builds a fresh index B from the kept
rows in order; A must match B exactly: ntotal, reconstruct_n, search D/I on AUTO and EXACT, range_search lims/D/I and
the bytes of the saved file (the escalation counts may differ: A keeps the certificate constants of the larger row set).
"""
import ctypes

import numpy as np
import pytest

from tests.conftest import unit_rows
from tests.helpers import exact_topk_f64, int_corpus
from tests.test_search_gpu import e5_like_rows

pytestmark = pytest.mark.gpu

AUTO, EXACT = 0, 1


@pytest.fixture(scope="module")
def fa():
    from kirag_b200 import faiss_api

    assert faiss_api.get_num_gpus() >= 1, "no CUDA device: the product has no CPU path"
    return faiss_api


def build(fa, x, **kw):
    ix = fa.IndexFlatIP(x.shape[1], **kw) if kw else fa.IndexFlatIP(x.shape[1], device=0)
    ix.add(x)
    return ix


def same_as_fresh(fa, A, B, xq, tmp_path, shapes=((32, 100),), radius=None):
    assert A.ntotal == B.ntotal
    assert np.array_equal(A.reconstruct_n().view(np.uint32), B.reconstruct_n().view(np.uint32))
    for nq, k in shapes:
        for path in (AUTO, EXACT):
            Da, Ia, _ = A.search_ex(xq[:nq], k, path=path)
            Db, Ib, _ = B.search_ex(xq[:nq], k, path=path)
            assert np.array_equal(Ia, Ib), f"nq={nq} k={k} path={path}: ids differ from the fresh index"
            assert np.array_equal(Da.view(np.uint32), Db.view(np.uint32)), f"nq={nq} k={k} path={path}: scores"
    if radius is not None:
        la, Da, Ia = A.range_search(xq[:8], radius)
        lb, Db, Ib = B.range_search(xq[:8], radius)
        assert np.array_equal(la, lb) and np.array_equal(Ia, Ib) and np.array_equal(Da.view(np.uint32), Db.view(np.uint32))
    fa.write_index(A, tmp_path / "a.faiss")
    fa.write_index(B, tmp_path / "b.faiss")
    assert (tmp_path / "a.faiss").read_bytes() == (tmp_path / "b.faiss").read_bytes()


def selections(n, rng):
    """name -> (what remove_ids gets, boolean mask of the removed rows)"""
    ar = np.arange(n)
    out = {
        "row0": ([0], ar == 0),
        "last": ([n - 1], ar == n - 1),
        "middle": ([n // 2 + 5], ar == n // 2 + 5),
        "tile": (np.arange(1280, 1408), (ar >= 1280) & (ar < 1408)),
        "cross": (np.arange(1000, 5001), (ar >= 1000) & (ar < 5001)),
        "p1": None, "p50": None,
        "every_other": (ar[1::2], ar % 2 == 1),
        "dup_and_outside": (np.array([7, 7, -3, n, n + 100, 3, 7, -1]), (ar == 7) | (ar == 3)),
        "empty": (np.array([], dtype=np.int64), np.zeros(n, dtype=bool)),
    }
    for name, p in (("p1", 0.01), ("p50", 0.5)):
        m = rng.random(n) < p
        out[name] = (rng.permutation(np.flatnonzero(m)), m)  # unsorted ids
    return out


@pytest.fixture(scope="module")
def unit_data():
    rng = np.random.default_rng(2026)
    return unit_rows(rng, 200_000, 1024), unit_rows(rng, 4096, 1024), rng


@pytest.fixture(scope="module")
def sels(unit_data):
    return selections(len(unit_data[0]), unit_data[2])


@pytest.mark.parametrize("name", ["row0", "last", "middle", "tile", "cross", "p1", "p50", "every_other",
                                  "dup_and_outside", "empty"])
def test_unit_corpus_selections(fa, unit_data, sels, name, tmp_path):
    xb, xq, _ = unit_data
    ids, mask = sels[name]
    A = build(fa, xb)
    assert A.remove_ids(ids) == int(mask.sum())
    B = build(fa, xb[~mask])
    shapes = ((1, 1), (32, 100), (300, 2048), (4096, 100)) if name != "row0" else \
        tuple((nq, k) for nq in (1, 32, 300, 4096) for k in (1, 100, 2048))
    same_as_fresh(fa, A, B, xq, tmp_path, shapes=shapes, radius=0.1)


def test_selectors(fa, unit_data, tmp_path):
    xb, xq, _ = unit_data
    xb = xb[:50_000]
    A = build(fa, xb)
    assert A.remove_ids(fa.IDSelectorRange(-5, 300)) == 300
    assert A.remove_ids(fa.IDSelectorRange(40_000, 10 ** 12)) == 9700
    keep = np.ones(len(xb), dtype=bool)
    keep[:300] = False
    keep[40_300:] = False  # the second range is in new ids: old rows 40300.. are new rows 40000..
    assert A.ntotal == int(keep.sum())
    assert A.remove_ids(fa.IDSelectorBatch(np.array([[1, 2], [2, 9]]))) == 3
    kept_ids = np.flatnonzero(keep)
    keep[kept_ids[[1, 2, 9]]] = False
    assert A.remove_ids(fa.IDSelectorRange(10, 10)) == 0 and A.remove_ids([]) == 0
    with pytest.raises(AssertionError):
        A.remove_ids("3")
    with pytest.raises(AssertionError):
        A.remove_ids(object())
    same_as_fresh(fa, A, build(fa, xb[keep]), xq, tmp_path, radius=0.1)


def test_shadow_rows_are_unchanged(fa, unit_data, sels):
    """The bf16 shadow of the kept rows is bit-identical after the compaction: same values, same order in K."""
    xb, xq, _ = unit_data
    A = build(fa, xb)
    before = A.debug_scores(xq[:8])
    _, mask = sels["p50"]
    A.remove_ids(np.flatnonzero(mask))
    after = A.debug_scores(xq[:8])
    assert np.array_equal(after.view(np.uint32), before[~mask].view(np.uint32))


def test_integer_data_is_exact(fa, tmp_path):
    rng = np.random.default_rng(5)
    xb, xq = int_corpus(rng, 30_000, 256), int_corpus(rng, 16, 256)
    A = build(fa, xb)
    mask = rng.random(len(xb)) < 0.3
    A.remove_ids(np.flatnonzero(mask))
    for path in (AUTO, EXACT):
        D, I, _ = A.search_ex(xq, 50, path=path)
        S, Iref = exact_topk_f64(xb[~mask], xq, 50)
        assert np.array_equal(I, Iref) and np.array_equal(D.astype(np.float64), S)
    same_as_fresh(fa, A, build(fa, xb[~mask]), xq, tmp_path, radius=40.0)


def test_e5_like_clustered_and_no_shadow_corpora(fa, tmp_path):
    rng = np.random.default_rng(11)
    e5 = e5_like_rows(rng, 40_000, 1024)[0], e5_like_rows(rng, 50, 1024)[0], 0.8
    centers = unit_rows(rng, 8, 128)
    cl = centers[rng.integers(0, 8, 60_000)] + 0.004 * rng.standard_normal((60_000, 128)).astype(np.float32)
    cl = (cl / np.linalg.norm(cl, axis=1, keepdims=True)).astype(np.float32)
    clq = (centers[:4] + 0.01 * unit_rows(rng, 4, 128)).astype(np.float32)
    no_shadow = unit_rows(rng, 20_000, 100), unit_rows(rng, 32, 100), 0.2
    for xb, xq, radius in (e5, (cl, clq, 0.99), no_shadow):
        for mask in (np.arange(len(xb)) < 3000, rng.random(len(xb)) < 0.2):
            A = build(fa, xb)
            A.remove_ids(np.flatnonzero(mask))
            same_as_fresh(fa, A, build(fa, xb[~mask]), xq, tmp_path, radius=radius)
    A = build(fa, cl)
    A.remove_ids(np.arange(0, 60_000, 3))
    _, _, st = A.search_ex(clq, 10, path=AUTO)
    assert st["n_rescan"] + st["n_retry"] + st["n_exact"] >= 1, st  # still escalates, and still right
    same_as_fresh(fa, A, build(fa, np.delete(cl, np.arange(0, 60_000, 3), axis=0)), clq, tmp_path)


def test_remove_all_then_add_is_a_fresh_index(fa, tmp_path):
    """After every row is removed the index decides its centre again from the rows added next.  The centre is a mean
    summed with float atomics, so two builds agree on it to rounding only: A's shadow scores are compared with a fresh
    index's within that rounding, and against an index that kept the first rows' decision (not centred)."""
    rng = np.random.default_rng(3)
    xa = unit_rows(rng, 10_000, 1024)              # no common component: not centred
    xe, _ = e5_like_rows(rng, 10_000, 1024)        # centred
    xq = e5_like_rows(rng, 16, 1024)[0]
    for master in ("device", "host"):
        A = build(fa, xa, device=0, master=master)
        assert A.remove_ids(fa.IDSelectorRange(0, A.ntotal)) == 10_000 and A.ntotal == 0
        D, I = A.search(xq, 3)
        assert np.all(I == -1)
        A.add(xe)
        B = build(fa, xe, device=0, master=master)
        C = build(fa, xa, device=0, master=master)
        C.add(xe)
        sb = B.debug_scores(xq).astype(np.float64)
        err_a = np.sqrt(np.mean((A.debug_scores(xq) - sb) ** 2))
        err_c = np.sqrt(np.mean((C.debug_scores(xq)[10_000:] - sb) ** 2))
        assert err_a * 4 < err_c, (err_a, err_c)
        same_as_fresh(fa, A, B, xq, tmp_path, radius=0.8)


def test_add_remove_sequences(fa, tmp_path):
    rng = np.random.default_rng(9)
    xq = unit_rows(rng, 32, 256)
    A = fa.IndexFlatIP(256, device=0)
    rows = np.zeros((0, 256), dtype=np.float32)
    for step in range(6):
        x = unit_rows(rng, int(rng.integers(1, 9000)), 256)
        A.add(x)
        rows = np.concatenate([rows, x])
        m = rng.random(len(rows)) < rng.choice([0.0, 0.01, 0.3, 0.9])
        assert A.remove_ids(np.flatnonzero(m)) == int(m.sum())
        rows = rows[~m]
        same_as_fresh(fa, A, build(fa, rows), xq, tmp_path, radius=0.15)


def test_host_master_equals_device_master(fa, unit_data, sels, tmp_path):
    xb, xq, _ = unit_data
    for name in ("row0", "last", "cross", "p50", "dup_and_outside"):
        ids, mask = sels[name]
        dev, host = build(fa, xb), build(fa, xb, device=0, master="host")
        assert dev.remove_ids(ids) == host.remove_ids(ids) == int(mask.sum())
        same_as_fresh(fa, host, dev, xq, tmp_path, shapes=((32, 100), (300, 2048)), radius=0.1)
        assert host.storage_bytes()["host"] > 0


def multi_configs(fa):
    out = [[0] * g for g in (1, 2, 3, 8)]
    n = fa.get_num_gpus()
    if n >= 2:
        out.append(list(range(min(8, n))))
    return out


@pytest.mark.parametrize("master", ["device", "host"])
def test_multi_device_equals_a_fresh_single_device_index(fa, unit_data, sels, master, tmp_path):
    xb, xq, _ = unit_data
    xb = xb[:100_000]
    rng = np.random.default_rng(17)
    for devices in multi_configs(fa):
        G = len(devices)
        for sel in ("row0", "tile", "p50", "all_but_one"):
            A = build(fa, xb, devices=devices, master=master)
            if sel == "all_but_one":
                mask = np.ones(len(xb), dtype=bool)
                mask[int(rng.integers(len(xb)))] = False
            else:
                mask = selections(len(xb), rng)[sel][1]
            assert A.remove_ids(np.flatnonzero(mask)) == int(mask.sum())
            B = build(fa, xb[~mask])
            same_as_fresh(fa, A, B, xq, tmp_path, shapes=((32, 100), (300, 2048)), radius=0.1)
            rows, want = np.zeros(G, dtype=np.int64), np.zeros(G, dtype=np.int64)
            i64p = ctypes.POINTER(ctypes.c_int64)
            assert A._lib.kirag_index_shards(A._h, None, rows.ctypes.data_as(i64p), G) == G
            assert A._lib.kirag_debug_stripe_rows(A.ntotal, G, want.ctypes.data_as(i64p)) == 0
            assert np.array_equal(rows, want)


def test_handle_state(fa, unit_data, tmp_path):
    import torch

    xb, xq, _ = unit_data
    xb = xb[:20_000]
    A = build(fa, xb)
    q = torch.from_numpy(xq[:4]).cuda(0)
    # a pending asynchronous search is completed first
    D, I = A.search_device_async(q, 10)
    A.remove_ids([0, 1])
    Dr, Ir = build(fa, xb).search(xq[:4], 10)
    assert np.array_equal(I.cpu().numpy(), Ir)
    # a cached graph is recaptured: the state token changed with ntotal
    Dg, Ig = A.search_device_graph(q, 10)
    tok = A.state_token()
    A.remove_ids([5])
    assert A.state_token() != tok
    Dg, Ig = A.search_device_graph(q, 10)
    keep = np.ones(len(xb), dtype=bool)
    keep[[0, 1, 7]] = False  # row 5 of the index was old row 7
    Db, Ib = build(fa, xb[keep]).search(xq[:4], 10)
    assert np.array_equal(Ig.cpu().numpy(), Ib) and np.array_equal(Dg.cpu().numpy(), Db)
    # a range result that was never fetched is dropped
    lims = np.zeros(5, dtype=np.int64)
    assert A._lib.kirag_index_range_search(A._h, q.data_ptr(), 4, 0.1, 1, 0, AUTO, lims.ctypes.data, None, None) == 0
    A.remove_ids([3])
    assert lims[4] > 0
    Dr, Ir = np.zeros(lims[4], dtype=np.float32), np.zeros(lims[4], dtype=np.int64)
    assert A._lib.kirag_index_range_fetch(A._h, Dr.ctypes.data, Ir.ctypes.data, 0, None) != 0
    # storage stays mapped
    st = A.storage_bytes()
    A.remove_ids(fa.IDSelectorRange(0, A.ntotal))
    assert A.storage_bytes() == st and A.ntotal == 0


def test_as_faiss_passes_remove_ids_through(fa, unit_data, tmp_path):
    import kirag_b200.as_faiss  # noqa: F401
    import sys

    faiss = sys.modules["faiss"]
    xb, xq, _ = unit_data
    xb = xb[:5000]
    ix = faiss.IndexFlatIP(1024)
    ix.add(xb)
    assert ix.remove_ids(np.array([0, 10, 4999])) == 3
    assert ix.remove_ids(faiss.IDSelectorBatch([1])) == 1 and ix.remove_ids(faiss.IDSelectorRange(0, 1)) == 1
    keep = np.ones(5000, dtype=bool)
    keep[[0, 10, 4999, 2, 1]] = False
    same_as_fresh(fa, ix, build(fa, xb[keep]), xq, tmp_path)
