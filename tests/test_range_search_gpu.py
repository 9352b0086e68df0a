"""Range search on the B200 (IndexFlatIP.range_search): exact against the fp64 restatement on integer data, the filter
path bit-equal to the fp32 scan, the second pass and the long-segment sort, edge cases and every Python entry point."""
import numpy as np
import pytest

from tests.conftest import unit_rows
from tests.helpers import int_corpus
from tests.range_oracle import flat_ip_range_search
from tests.test_search_gpu import e5_like_rows

pytestmark = pytest.mark.gpu

AUTO, EXACT, FAST = 0, 1, 2


@pytest.fixture(scope="module")
def fa():
    from kirag_b200 import faiss_api

    assert faiss_api.get_num_gpus() >= 1, "no CUDA device: the product has no CPU path"
    return faiss_api


def build(fa, xb):
    ix = fa.IndexFlatIP(xb.shape[1])
    if len(xb):
        ix.add(xb)
    return ix


def range_ex(ix, xq, radius, path=AUTO, id_offset=0):
    """range_search_device with an explicit path, results on the host, plus the stats."""
    import torch

    lims, D, I = ix.range_search_device(torch.from_numpy(np.ascontiguousarray(xq)).cuda(ix.device), radius,
                                        id_offset=id_offset, path=path)
    return lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy(), dict(ix.last_stats)


def assert_same(a, b, what=""):
    for x, y, name in zip(a[:3], b[:3], ("lims", "D", "I")):
        assert x.dtype == y.dtype and np.array_equal(x, y), f"{what}: {name} differs"


def assert_ordered(lims, D, I):
    for i in range(len(lims) - 1):
        d, ids = D[lims[i]:lims[i + 1]], I[lims[i]:lims[i + 1]]
        assert np.all((d[:-1] > d[1:]) | ((d[:-1] == d[1:]) & (ids[:-1] < ids[1:]))), f"query {i}: order"


# all five scan kernels: 64r / 128r / 256s at d = 1024, 64s / 128s at d = 2560
@pytest.mark.parametrize("n,d,nq", [(20000, 1024, 1), (20000, 1024, 100), (20000, 1024, 300),
                                    (10000, 2560, 1), (10000, 2560, 100)])
def test_integer_data_equals_the_oracle_exactly(fa, n, d, nq):
    rng = np.random.default_rng(n + d + nq)
    xb, xq = int_corpus(rng, n, d), int_corpus(rng, nq, d)
    xb[n // 2:n // 2 + 5] = xb[11]  # equal scores: ids ascending
    s0 = np.sort(xq[0].astype(np.float64) @ xb.T.astype(np.float64))[::-1]
    radius = float(s0[40])  # an integer that rows of query 0 score exactly: they must be absent
    ix = build(fa, xb)
    got = range_ex(ix, xq, radius)
    ref = flat_ip_range_search(xb, xq, radius)
    assert_same(got, ref, f"n={n} d={d} nq={nq}")
    assert got[3]["path"] == AUTO and got[3]["n_fast"] == nq and got[3]["levels"] == 1
    assert int(np.sum(s0 == radius)) > 0 and got[0][1] == int(np.sum(s0 > radius))


def test_unit_vectors_auto_equals_exact_and_the_topk_prefix(fa):
    rng = np.random.default_rng(1)
    xb, xq = unit_rows(rng, 200_000, 1024), unit_rows(rng, 16, 1024)
    ix = build(fa, xb)
    Dk, Ik, _ = ix.search_ex(xq, 2048, path=AUTO)
    radius = float(np.median(Dk[:, 99]))
    got = range_ex(ix, xq, radius)
    assert_same(got, range_ex(ix, xq, radius, path=EXACT), "AUTO vs EXACT")
    lims, D, I, st = got
    assert st["n_fast"] == 16 and st["n_overflow"] == 0
    for i in range(16):
        m = int(np.sum(Dk[i] > radius))
        assert m < 2048 and lims[i + 1] - lims[i] == m
        assert np.array_equal(D[lims[i]:lims[i + 1]], Dk[i, :m]) and np.array_equal(I[lims[i]:lims[i + 1]], Ik[i, :m])


def test_overflowed_buffers_take_the_second_pass(fa, monkeypatch):
    monkeypatch.setenv("KIRAG_CAND_CAP", "1024")
    rng = np.random.default_rng(2)
    xb = unit_rows(rng, 100_000, 128)
    u = unit_rows(rng, 1, 128)[0]
    near = rng.choice(100_000, 3000, replace=False)
    xb[near] = u + 0.3 * unit_rows(rng, 3000, 128)  # ~3000 hits for queries along u, a handful for the others
    xq = np.concatenate([u[None, :] + 0.05 * unit_rows(rng, 4, 128), unit_rows(rng, 60, 128)]).astype(np.float32)
    ix = build(fa, xb)
    got = range_ex(ix, xq, 0.3)
    lims, _, _, st = got
    assert st["n_overflow"] >= 4 and st["levels"] == 2 and st["n_fast"] + st["n_overflow"] == 64
    assert np.all(np.diff(lims)[:4] > 2000) and np.all(np.diff(lims)[4:] < 100)
    assert_same(got, range_ex(ix, xq, 0.3, path=EXACT), "AUTO vs EXACT")
    assert_ordered(*got[:3])


def test_minus_inf_returns_every_row_through_the_run_merges(fa):
    rng = np.random.default_rng(3)
    n = 50_000
    xb = unit_rows(rng, n, 64)
    xb[30_000:30_010] = xb[5]  # ties far apart in the lists
    xq = unit_rows(rng, 3, 64)
    ix = build(fa, xb)
    got = range_ex(ix, xq, float("-inf"))
    lims, D, I, st = got
    assert lims.tolist() == [0, n, 2 * n, 3 * n] and st["n_overflow"] == 3
    for i in range(3):
        assert np.array_equal(np.sort(I[lims[i]:lims[i + 1]]), np.arange(n)), f"query {i}: every row exactly once"
    assert_ordered(lims, D, I)
    assert_same(got, range_ex(ix, xq, float("-inf"), path=EXACT), "AUTO vs EXACT")


def test_edge_cases_and_id_offset(fa):
    rng = np.random.default_rng(4)
    xb, xq = int_corpus(rng, 3000, 64), int_corpus(rng, 5, 64)
    ix = build(fa, xb)
    for r in (float("inf"), float("nan")):
        lims, D, I = ix.range_search(xq, r)
        assert lims.tolist() == [0] * 6 and D.shape == (0,) and I.shape == (0,)
    lims, D, I = ix.range_search(xq[:0], 1.0)
    assert lims.tolist() == [0] and D.shape == (0,)
    lims, D, I = build(fa, np.zeros((0, 64), dtype=np.float32)).range_search(xq, -1e30)
    assert lims.tolist() == [0] * 6
    base = range_ex(ix, xq, 20.0)
    shifted = range_ex(ix, xq, 20.0, id_offset=1_000_000)
    assert np.array_equal(shifted[2], base[2] + 1_000_000) and np.array_equal(shifted[1], base[1])
    assert_same(base, flat_ip_range_search(xb, xq, 20.0), "int data")
    # the held result belongs to the last call: fetching twice, or after another call, is an error
    lib = ix._lib
    lims = np.zeros(6, dtype=np.int64)
    assert lib.kirag_index_range_search(ix._h, xq.ctypes.data, 5, 20.0, 0, 0, 0, lims.ctypes.data, None, None) == 0
    D = np.empty(int(lims[-1]), dtype=np.float32)
    I = np.empty(int(lims[-1]), dtype=np.int64)
    ix.search(xq, 3)
    assert lib.kirag_index_range_fetch(ix._h, D.ctypes.data, I.ctypes.data, 0, None) != 0
    from kirag_b200 import _lib

    assert "no range-search result is held" in _lib.last_error()
    assert lib.kirag_index_range_search(ix._h, xq.ctypes.data, 5, 20.0, 0, 0, 0, lims.ctypes.data, None, None) == 0
    assert lib.kirag_index_range_fetch(ix._h, D.ctypes.data, I.ctypes.data, 0, None) == 0
    assert np.array_equal(I, base[2]) and np.array_equal(D, base[1])
    assert lib.kirag_index_range_fetch(ix._h, D.ctypes.data, I.ctypes.data, 0, None) != 0


def test_dimension_without_shadow_runs_on_the_exact_path(fa):
    rng = np.random.default_rng(6)
    xb, xq = int_corpus(rng, 7000, 100), int_corpus(rng, 9, 100)
    ix = build(fa, xb)
    got = range_ex(ix, xq, 25.0)
    assert got[3]["path"] == EXACT and got[3]["n_exact"] == 9
    assert_same(got, flat_ip_range_search(xb, xq, 25.0), "d=100")


def test_e5_like_centred_corpus_auto_equals_exact(fa):
    rng = np.random.default_rng(7)
    xb, mu = e5_like_rows(rng, 100_000, 512, 0.93)
    xq, _ = e5_like_rows(np.random.default_rng(8), 32, 512, 0.93)
    xq = (0.5 * xq + 0.5 * mu[None, :]).astype(np.float32)
    xq /= np.linalg.norm(xq, axis=1, keepdims=True)
    ix = build(fa, xb)
    Dk, _, _ = ix.search_ex(xq, 100, path=EXACT)
    radius = float(np.median(Dk[:, 99]))
    got = range_ex(ix, xq, radius)
    assert got[0][-1] > 0 and got[3]["path"] == AUTO
    assert_same(got, range_ex(ix, xq, radius, path=EXACT), "e5-like")


def test_host_device_and_faiss_spelling_agree(fa):
    import sys

    import kirag_b200.as_faiss  # noqa: F401

    faiss = sys.modules["faiss"]
    rng = np.random.default_rng(9)
    xb, xq = unit_rows(rng, 30_000, 128), unit_rows(rng, 7, 128)
    ix = faiss.IndexFlatIP(128)
    ix.add(xb)
    lims, D, I = ix.range_search(xq, 0.25)
    assert lims.shape == (8,) and lims.dtype == np.int64 and D.dtype == np.float32 and I.dtype == np.int64
    assert D.shape == (lims[-1],) and I.shape == (lims[-1],) and lims[-1] > 0
    assert_same((lims, D, I), range_ex(ix, xq, 0.25), "host vs device")
    assert_ordered(lims, D, I)


def test_numpy_range_search_honours_kirag_path(fa, monkeypatch):
    rng = np.random.default_rng(11)
    xb, xq = unit_rows(rng, 30_000, 128), unit_rows(rng, 6, 128)
    ix = build(fa, xb)
    auto = ix.range_search(xq, 0.25)
    assert ix.last_stats["path"] == AUTO and ix.last_stats["n_fast"] == 6
    monkeypatch.setenv("KIRAG_PATH", str(EXACT))
    exact = ix.range_search(xq, 0.25)
    assert ix.last_stats["path"] == EXACT and ix.last_stats["n_exact"] == 6 and ix.last_stats["n_fast"] == 0
    assert_same(auto, exact, "KIRAG_PATH=1")


def test_sharded_world_size_1_equals_the_plain_index(fa):
    import torch

    from kirag_b200.sharded import ShardedFlatIP

    rng = np.random.default_rng(10)
    xb, xq = unit_rows(rng, 20_000, 256), unit_rows(rng, 5, 256)
    sh = ShardedFlatIP(256, 20_000, rank=0, world_size=1)
    sh.add_shard(xb)
    lims, D, I = sh.range_search(torch.from_numpy(xq).cuda(sh.index.device), 0.2)
    ref = build(fa, xb).range_search(xq, 0.2)
    assert_same((lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()), ref, "sharded world 1")
