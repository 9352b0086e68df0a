"""IndexIDMap on the B200.  Every case compares an id map against a plain IndexFlatIP holding the same rows: D and lims
bit-equal, I equal to the ids of the plain index's rows (-1 kept).  Removals are compared with a fresh id map built from
the kept rows and the kept ids.  External ids are random int64 values with negatives, values near 2**62 and duplicates.
"""
import ctypes

import numpy as np
import pytest

from tests import ixmp_oracle
from tests.conftest import unit_rows
from tests.test_search_gpu import e5_like_rows

pytestmark = pytest.mark.gpu

AUTO, EXACT, FAST = 0, 1, 2


@pytest.fixture(scope="module")
def fa():
    from kirag_b200 import faiss_api

    assert faiss_api.get_num_gpus() >= 1, "no CUDA device: the product has no CPU path"
    return faiss_api


def ext_ids(rng, n):
    ids = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)
    m = min(50, n // 4)
    ids[n // 2:n // 2 + m] = ids[:m]  # duplicates
    ids[m:m + 10] = (1 << 62) - np.arange(10) if n > m + 10 else ids[m:m + 10]
    ids[n - 1] = -1  # an id that looks like padding
    return ids


def mapped(I, ids):
    return np.where(I >= 0, ids[np.clip(I, 0, None)], -1)


def make_pair(fa, x, ids, **kw):
    kw = kw or {"device": 0}
    P = fa.IndexFlatIP(x.shape[1], **kw)
    P.add(x)
    M = fa.IndexIDMap(fa.IndexFlatIP(x.shape[1], **kw))
    M.add_with_ids(x, ids)
    return P, M


def same_search(P, M, ids, xq, k, path):
    Dp, Ip, sp = P.search_ex(xq, k, path=path)
    Dm, Im, sm = M.search_ex(xq, k, path=path)
    assert np.array_equal(Dm.view(np.uint32), Dp.view(np.uint32)), f"scores differ (nq={len(xq)} k={k} path={path})"
    assert np.array_equal(Im, mapped(Ip, ids)), f"ids differ (nq={len(xq)} k={k} path={path})"
    for key in ("n_fast", "n_exact", "n_rescan", "n_retry", "path"):
        assert sp[key] == sm[key], key
    return sm


def same_range(P, M, ids, xq, radius, path=AUTO):
    import os

    old = os.environ.get("KIRAG_PATH")
    os.environ["KIRAG_PATH"] = str(path)
    try:
        lp, Dp, Ip = P.range_search(xq, radius)
        lm, Dm, Im = M.range_search(xq, radius)
    finally:
        if old is None:
            del os.environ["KIRAG_PATH"]
        else:
            os.environ["KIRAG_PATH"] = old
    assert np.array_equal(lm, lp) and np.array_equal(Dm.view(np.uint32), Dp.view(np.uint32))
    assert np.array_equal(Im, ids[Ip])
    return int(lm[-1])


@pytest.fixture(scope="module")
def unit_pair(fa):
    rng = np.random.default_rng(11)
    x = unit_rows(rng, 200_000, 1024)
    xq = unit_rows(rng, 4096, 1024)
    ids = ext_ids(rng, len(x))
    P, M = make_pair(fa, x, ids)
    return P, M, x, xq, ids


@pytest.mark.parametrize("path", [AUTO, EXACT, FAST])
@pytest.mark.parametrize("nq", [1, 32, 128, 300, 4096])
@pytest.mark.parametrize("k", [1, 100, 2048])
def test_search_returns_the_ids_of_the_plain_rows(unit_pair, path, nq, k):
    P, M, _, xq, ids = unit_pair
    same_search(P, M, ids, xq[:nq], k, path)


def test_id_map_members(fa, unit_pair):
    P, M, x, _, ids = unit_pair
    assert M.ntotal == P.ntotal == len(x) and M.d == 1024 and M.is_trained and M.metric_type == fa.METRIC_INNER_PRODUCT
    assert np.array_equal(M.id_map, ids) and np.array_equal(fa.vector_to_array(M.id_map), ids)
    assert np.array_equal(M.index.reconstruct_n(5, 3).view(np.uint32), x[5:8].view(np.uint32))
    assert M.storage_bytes()["device"] >= P.storage_bytes()["device"] + 8 * len(x)


def test_escalation_writers_map_their_rows(fa):
    """Clustered rows (certificate failures: second pass, overflow retries) and all-equal rows (exact scan): every
    writer that rewrites rows maps them."""
    rng = np.random.default_rng(5)
    xc, _ = e5_like_rows(rng, 60_000, 1024, common=0.97)
    xe = np.tile(unit_rows(rng, 1, 1024), (20_000, 1))
    for x in (xc, xe):
        ids = ext_ids(rng, len(x))
        P, M = make_pair(fa, x, ids)
        xq = x[rng.choice(len(x), 64, replace=False)] + 0.01 * unit_rows(rng, 64, 1024)
        for k in (10, 100):
            same_search(P, M, ids, xq, k, AUTO)


def test_async_finish_and_graph_replay_map_rewritten_rows(fa):
    import torch

    rng = np.random.default_rng(6)
    x, _ = e5_like_rows(rng, 60_000, 1024, common=0.97)
    ids = ext_ids(rng, len(x))
    P, M = make_pair(fa, x, ids)
    q = torch.from_numpy(x[:32] + 0.01 * unit_rows(rng, 32, 1024)).cuda(0)
    Dp, Ip = P.search_device(q, 50)
    Da, Ia = M.search_device_async(q, 50)
    M.finish()
    torch.cuda.synchronize()
    idm = M.id_map
    assert torch.equal(Da, Dp) and np.array_equal(Ia.cpu().numpy(), mapped(Ip.cpu().numpy(), idm))
    for round_ in range(2):
        Dg, Ig = M.search_device_graph(q, 50)
        Dp, Ip = P.search_device(q, 50)
        torch.cuda.synchronize()
        assert torch.equal(Dg, Dp) and np.array_equal(Ig.cpu().numpy(), mapped(Ip.cpu().numpy(), M.id_map)), round_
        tok = M.state_token()
        extra = x[:1000] * 1.01
        more = ext_ids(rng, 1000)
        M.add_with_ids_device(torch.from_numpy(extra).cuda(0), torch.from_numpy(more).cuda(0))
        P.add(extra)
        assert M.state_token() != tok
    with pytest.raises(RuntimeError, match="id_offset must be 0"):
        M.index.search_device(q, 5, id_offset=7)


def test_range_search_maps_every_pass(unit_pair):
    P, M, _, xq, ids = unit_pair
    for path in (AUTO, EXACT):
        assert same_range(P, M, ids, xq[:16], 0.08, path) > 0
    # most rows pass: the candidate buffer overflows and the second pass answers
    assert same_range(P, M, ids, xq[:2], -0.05) > 100_000
    assert same_range(P, M, ids, xq[:2], -np.inf) == 2 * M.ntotal


def test_exact_path_for_d100(fa):
    rng = np.random.default_rng(7)
    x = unit_rows(rng, 5000, 100)
    ids = ext_ids(rng, len(x))
    P, M = make_pair(fa, x, ids)
    xq = unit_rows(rng, 40, 100)
    st = same_search(P, M, ids, xq, 20, AUTO)
    assert st["path"] == EXACT
    same_range(P, M, ids, xq, 0.2)


@pytest.fixture(scope="module")
def mid_data():
    rng = np.random.default_rng(8)
    x = unit_rows(rng, 30_000, 256)
    return x, unit_rows(rng, 64, 256), ext_ids(rng, len(x))


def kinds(fa):
    out = [("G1", {"devices": [0]}), ("G2", {"devices": [0, 0]}), ("G3", {"devices": [0, 0, 0]}),
           ("G8", {"devices": [0] * 8}), ("host", {"device": 0, "master": "host"})]
    n = fa.get_num_gpus()
    if n > 1:
        out.append((f"all{n}", {"devices": list(range(n))}))
    return out


def test_multi_device_and_host_master_equal_the_single_device_map(fa, mid_data, tmp_path):
    x, xq, ids = mid_data
    _, S = make_pair(fa, x, ids)
    Ds, Is = S.search(xq, 64)
    ls, Drs, Irs = S.range_search(xq[:8], 0.1)
    fa.write_index(S, tmp_path / "s.faiss")
    ref = (tmp_path / "s.faiss").read_bytes()
    for name, kw in kinds(fa):
        M = fa.IndexIDMap(fa.IndexFlatIP(256, **kw))
        M.add_with_ids(x[:10_000], ids[:10_000])
        M.add_with_ids(x[10_000:], ids[10_000:])
        D, I = M.search(xq, 64)
        assert np.array_equal(D.view(np.uint32), Ds.view(np.uint32)) and np.array_equal(I, Is), name
        lm, Dm, Im = M.range_search(xq[:8], 0.1)
        assert np.array_equal(lm, ls) and np.array_equal(Im, Irs) and np.array_equal(Dm, Drs), name
        assert np.array_equal(M.id_map, ids), name
        fa.write_index(M, tmp_path / f"{name}.faiss")
        assert (tmp_path / f"{name}.faiss").read_bytes() == ref, name
        with pytest.raises(RuntimeError, match="id_offset must be 0"):
            M.index.search_ex(xq[:1], 5, id_offset=3)


def fresh(fa, x, ids, **kw):
    M = fa.IndexIDMap(fa.IndexFlatIP(x.shape[1], **(kw or {"device": 0})))
    if len(x):
        M.add_with_ids(x, ids)
    return M


def same_as_fresh(fa, A, B, xq, tmp_path):
    assert A.ntotal == B.ntotal
    assert np.array_equal(A.id_map, B.id_map)
    assert np.array_equal(A.index.reconstruct_n().view(np.uint32), B.index.reconstruct_n().view(np.uint32))
    if B.ntotal:
        for path in (AUTO, EXACT):
            Da, Ia, _ = A.search_ex(xq, 50, path=path)
            Db, Ib, _ = B.search_ex(xq, 50, path=path)
            assert np.array_equal(Ia, Ib) and np.array_equal(Da.view(np.uint32), Db.view(np.uint32)), path
        la, Da, Ia = A.range_search(xq[:4], 0.1)
        lb, Db, Ib = B.range_search(xq[:4], 0.1)
        assert np.array_equal(la, lb) and np.array_equal(Ia, Ib) and np.array_equal(Da.view(np.uint32), Db.view(np.uint32))
    fa.write_index(A, tmp_path / "a.faiss")
    fa.write_index(B, tmp_path / "b.faiss")
    assert (tmp_path / "a.faiss").read_bytes() == (tmp_path / "b.faiss").read_bytes()


def removals(ids, rng):
    """name -> (selection, boolean mask of the rows it removes)"""
    absent = np.array([12345, -(1 << 61) + 3], dtype=np.int64)
    absent = absent[~np.isin(absent, ids)]
    dup = ids[:3]  # ids[:50] also sit at n // 2 .. : every row of a duplicated id goes
    some = rng.choice(ids, len(ids) // 100, replace=False)
    lo, hi = np.sort(ids)[len(ids) // 3], np.sort(ids)[len(ids) // 2]
    return {
        "batch_absent_repeated": (np.concatenate([some, some[:7], absent]), np.isin(ids, some)),
        "duplicated_ids": (dup, np.isin(ids, dup)),
        "minus_one": (np.array([-1]), ids == -1),
        "range": (("range", lo, hi), (ids >= lo) & (ids < hi)),
        "range_empty": (("range", 5, 5), np.zeros(len(ids), bool)),
        "device": (("device", some), np.isin(ids, some)),
        "all": (ids, np.ones(len(ids), bool)),
    }


@pytest.mark.parametrize("kind", ["single", "host", "G3"])
def test_remove_ids_selects_by_external_id(fa, mid_data, tmp_path, kind):
    import torch

    x, xq, ids = mid_data
    kw = {"single": {}, "host": {"device": 0, "master": "host"}, "G3": {"devices": [0, 0, 0]}}[kind]
    rng = np.random.default_rng(9)
    for name, (sel, mask) in removals(ids, rng).items():
        if kind != "single" and name not in ("batch_absent_repeated", "range", "all"):
            continue
        A = fresh(fa, x, ids, **kw)
        if isinstance(sel, tuple) and sel[0] == "range":
            n = A.remove_ids(fa.IDSelectorRange(sel[1], sel[2]))
        elif isinstance(sel, tuple):
            n = A.remove_ids_device(torch.from_numpy(sel[1]).cuda(0))
        else:
            n = A.remove_ids(fa.IDSelectorBatch(sel) if name == "duplicated_ids" else sel)
        assert n == int(mask.sum()), name
        B = fresh(fa, x[~mask], ids[~mask], **kw)
        same_as_fresh(fa, A, B, xq, tmp_path)
        if name == "all":
            A.add_with_ids(x[:500], ids[:500])
            same_as_fresh(fa, A, fresh(fa, x[:500], ids[:500], **kw), xq, tmp_path)


def test_positional_remove_ids_device_on_a_plain_index(fa, mid_data):
    import torch

    x, xq, _ = mid_data
    A = fa.IndexFlatIP(256, device=0)
    A.add(x)
    rows = np.array([5, 5, 70, -2, 10**9, 29_999], dtype=np.int64)
    assert A.remove_ids_device(torch.from_numpy(rows).cuda(0)) == 3
    keep = np.setdiff1d(np.arange(len(x)), rows)
    B = fa.IndexFlatIP(256, device=0)
    B.add(x[keep])
    Da, Ia = A.search(xq, 20)
    Db, Ib = B.search(xq, 20)
    assert np.array_equal(Ia, Ib) and np.array_equal(Da, Db)


def test_ixmp_file_matches_faiss_layout_and_loads_everywhere(fa, mid_data, tmp_path):
    x, xq, ids = mid_data
    P, M = make_pair(fa, x, ids)
    fa.write_index(M, tmp_path / "m.faiss")
    fa.write_index(P, tmp_path / "p.faiss")
    data = (tmp_path / "m.faiss").read_bytes()
    assert data == ixmp_oracle.ixmp_bytes(x, ids)
    assert data[37:37 + len((tmp_path / "p.faiss").read_bytes())] == (tmp_path / "p.faiss").read_bytes()
    D0, I0 = M.search(xq, 30)
    for kw in ({"device": 0}, {"devices": [0, 0, 0]}, {"device": 0, "master": "host"}):
        L = fa.read_index(tmp_path / "m.faiss", **kw)
        assert isinstance(L, fa.IndexIDMap) and np.array_equal(L.id_map, ids), kw
        D, I = L.search(xq, 30)
        assert np.array_equal(I, I0) and np.array_equal(D, D0), kw
        L.add_with_ids(x[:3], [1, 2, 3])
        assert L.ntotal == len(x) + 3
    assert isinstance(fa.read_index(tmp_path / "p.faiss", device=0), fa.IndexFlatIP)
    E = fresh(fa, x[:0], ids[:0])
    fa.write_index(E, tmp_path / "e.faiss")
    assert (tmp_path / "e.faiss").read_bytes() == ixmp_oracle.ixmp_bytes(x[:0], ids[:0])
    assert fa.read_index(tmp_path / "e.faiss", device=0).ntotal == 0


def test_faiss_style_code_runs_through_as_faiss_and_errors_raise(tmp_path, mid_data):
    from kirag_b200 import as_faiss
    from kirag_b200.sharded import ShardedFlatIP

    faiss = as_faiss.make_module()
    x, xq, ids = mid_data
    index = faiss.IndexIDMap(faiss.IndexFlatIP(256))
    index.add_with_ids(x, ids)
    D, I = index.search(xq, 10)
    assert np.isin(I, ids).all()
    assert index.remove_ids(np.array(I[:, 0])) >= 1
    assert index.remove_ids(faiss.IDSelectorRange(0, 1 << 62)) > 0
    faiss.write_index(index, str(tmp_path / "f.index"))
    back = faiss.read_index(str(tmp_path / "f.index"))
    assert np.array_equal(faiss.vector_to_array(back.id_map), index.id_map)
    index.reset()
    assert index.ntotal == 0 and index.id_map.size == 0
    index.add_with_ids(x[:10], np.arange(10))
    with pytest.raises(RuntimeError, match="add does not work on IndexIDMap"):
        index.add(x[:1])
    with pytest.raises(RuntimeError, match="add_with_ids not implemented"):
        faiss.IndexFlatIP(256).add_with_ids(x[:1], [1])
    plain = faiss.IndexFlatIP(256)
    plain.add(x[:1])
    with pytest.raises(RuntimeError, match="index must be empty on input"):
        faiss.IndexIDMap(plain)
    with pytest.raises(RuntimeError, match="reconstruct not implemented"):
        index.reconstruct(0)
    with pytest.raises(AssertionError, match="not same nb of vectors as ids"):
        index.add_with_ids(x[:3], [1, 2])
    with pytest.raises(RuntimeError, match="add does not work on IndexIDMap"):
        index.index.add(x[:1])  # the shared handle carries the map
    with pytest.raises(RuntimeError, match="IndexIDMap"):
        ShardedFlatIP(256, 100, rank=0, world_size=1, local_index=index)
    with pytest.raises(RuntimeError, match="index_id_map"):
        from kirag_b200 import _lib

        lib = _lib.load()
        out = np.zeros(1, np.int64)
        _lib.check(lib.kirag_index_id_map(plain._h, 0, 1, ctypes.c_void_p(out.ctypes.data), 0, None), "index_id_map")
