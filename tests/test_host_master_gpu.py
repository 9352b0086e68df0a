"""Host-resident fp32 master (IndexFlatIP(master="host")): every case builds one seeded dataset in a device-master and a
host-master index and requires bit-equal results, through search, the escalation ladder, range search, the
device-pointer entry points, add / reconstruct / save / load and the KiRAG-facing wrappers.  Each test pins at most a
few hundred MB of host memory."""
import os
import sys

import numpy as np
import pytest

from tests.conftest import unit_rows
from tests.helpers import assert_topk_parity, int_corpus
from tests.test_search_gpu import e5_like_rows

pytestmark = pytest.mark.gpu

AUTO, EXACT, FAST = 0, 1, 2
STAT_KEYS = ("n_fast", "n_exact", "n_cert_fail", "n_overflow", "n_rescan", "n_retry")


@pytest.fixture(scope="module")
def fa():
    from kirag_b200 import faiss_api

    assert faiss_api.get_num_gpus() >= 1, "no CUDA device: the product has no CPU path"
    return faiss_api


def pair(fa, xb, pieces=None):
    """The same rows in a device-master and a host-master index (added in `pieces` if given)."""
    out = []
    for master in ("device", "host"):
        ix = fa.IndexFlatIP(xb.shape[1], master=master)
        assert ix.master == master
        for lo, hi in (pieces or [(0, len(xb))]):
            ix.add(xb[lo:hi])
        out.append(ix)
    return out


def same_search(dev, host, xq, k, path):
    Dd, Id, sd = dev.search_ex(xq, k, path=path)
    Dh, Ih, sh = host.search_ex(xq, k, path=path)
    assert np.array_equal(Id, Ih) and np.array_equal(Dd, Dh), f"k={k} path={path}: host master differs"
    assert {key: sd[key] for key in STAT_KEYS} == {key: sh[key] for key in STAT_KEYS}, (sd, sh)
    return Dh, Ih, sh


@pytest.fixture(scope="module")
def unit_pair(fa):
    rng = np.random.default_rng(101)
    xb = unit_rows(rng, 20000, 512)
    return pair(fa, xb)


@pytest.mark.parametrize("nq", [1, 32, 128, 300, 1000])
@pytest.mark.parametrize("k", [10, 100, 2048])
def test_search_equals_device_master(fa, unit_pair, nq, k):
    dev, host = unit_pair
    xq = unit_rows(np.random.default_rng(nq * 7 + k), nq, 512)
    for path in (AUTO, EXACT, FAST):
        same_search(dev, host, xq, k, path)


# all five scan kernels: 64r / 128r / 256s at d = 1024, 64s / 128s at d = 2560
@pytest.mark.parametrize("n,d,nq", [(20000, 1024, 1), (20000, 1024, 100), (20000, 1024, 300),
                                    (10000, 2560, 1), (10000, 2560, 100)])
def test_integer_data_is_exact(fa, n, d, nq):
    rng = np.random.default_rng(n + d + nq)
    xb, xq = int_corpus(rng, n, d), int_corpus(rng, nq, d)
    dev, host = pair(fa, xb)
    D, I, _ = same_search(dev, host, xq, 50, AUTO)
    assert_topk_parity(D, I, xb, xq, 50, exact=True, what=f"host master n={n} d={d} nq={nq}")


def test_clustered_corpus_takes_the_second_pass(fa):
    rng = np.random.default_rng(7)
    centers = unit_rows(rng, 8, 128)
    xb = centers[rng.integers(0, 8, 40000)] + 0.004 * rng.standard_normal((40000, 128)).astype(np.float32)
    xb = (xb / np.linalg.norm(xb, axis=1, keepdims=True)).astype(np.float32)
    xq = (centers[:4] + 0.01 * unit_rows(rng, 4, 128)).astype(np.float32)
    dev, host = pair(fa, xb)
    D, I, st = same_search(dev, host, xq, 10, AUTO)
    assert st["n_rescan"] >= 1, st
    assert_topk_parity(D, I, xb, xq, 10, what=f"clustered {st}")
    De, Ie, _ = same_search(dev, host, xq, 10, EXACT)
    assert np.array_equal(I, Ie) and np.array_equal(D, De)


def test_all_equal_corpus_goes_to_the_staged_exact_scan(fa):
    rng = np.random.default_rng(8)
    xb = np.repeat(unit_rows(rng, 1, 256), 30000, axis=0)
    xq = unit_rows(rng, 5, 256)
    dev, host = pair(fa, xb)
    D, I, st = same_search(dev, host, xq, 20, AUTO)
    assert st["n_exact"] >= 1, st
    assert np.array_equal(I, np.tile(np.arange(20), (5, 1)))


def test_forced_exact_path_spans_query_groups_and_staged_pieces(fa):
    # 600 queries > 512 per group: two groups; 50k rows x 4 KB = 200 MB: four 64-MB pieces per group
    rng = np.random.default_rng(9)
    xb, xq = unit_rows(rng, 50_000, 1024), unit_rows(rng, 600, 1024)
    dev, host = pair(fa, xb)
    D, I, st = same_search(dev, host, xq, 10, EXACT)
    assert st["n_exact"] == 600
    Da, Ia, _ = same_search(dev, host, xq, 10, AUTO)
    assert np.array_equal(I, Ia) and np.array_equal(D, Da)


def test_e5_like_corpus_and_a_late_centre(fa):
    rng = np.random.default_rng(31)
    xb, mu = e5_like_rows(rng, 20000, 128)
    xq = (0.85 * mu[None, :] + 0.5 * unit_rows(rng, 64, 128)).astype(np.float32)
    xq /= np.linalg.norm(xq, axis=1, keepdims=True)
    dev, host = pair(fa, xb)
    same_search(dev, host, xq, 10, AUTO)
    # small first adds: the centre is decided once 4096 rows exist and the rows before are converted again
    dev2, host2 = pair(fa, xb, pieces=[(0, 1000), (1000, 3000), (3000, 5000), (5000, 20000)])
    D2, I2, _ = same_search(dev2, host2, xq, 10, AUTO)
    D, I, _ = same_search(dev, host, xq, 10, AUTO)
    assert np.array_equal(I, I2) and np.array_equal(D, D2)


def range_both(dev, host, xq, radius, path):
    out = []
    for ix in (dev, host):
        out.append(ix.range_search_device(_cuda(xq, ix), radius, path=path))
    (ld, Dd, Id), (lh, Dh, Ih) = out
    assert ld.equal(lh) and Dd.equal(Dh) and Id.equal(Ih), f"range radius={radius} path={path}: host master differs"
    assert dev.last_stats["n_overflow"] == host.last_stats["n_overflow"]
    return lh.cpu().numpy(), Dh.cpu().numpy(), Ih.cpu().numpy(), dict(host.last_stats)


def _cuda(x, ix):
    import torch

    return torch.from_numpy(np.ascontiguousarray(x)).cuda(ix.device)


def test_range_search_second_pass(fa, monkeypatch):
    monkeypatch.setenv("KIRAG_CAND_CAP", "1024")
    rng = np.random.default_rng(2)
    xb = unit_rows(rng, 100_000, 128)
    u = unit_rows(rng, 1, 128)[0]
    near = rng.choice(100_000, 3000, replace=False)
    xb[near] = u + 0.3 * unit_rows(rng, 3000, 128)
    xq = np.concatenate([u[None, :] + 0.05 * unit_rows(rng, 4, 128), unit_rows(rng, 60, 128)]).astype(np.float32)
    dev, host = pair(fa, xb)
    lims, D, I, st = range_both(dev, host, xq, 0.3, AUTO)
    assert st["n_overflow"] >= 4 and st["levels"] == 2
    le, De, Ie, _ = range_both(dev, host, xq, 0.3, EXACT)
    assert np.array_equal(lims, le) and np.array_equal(D, De) and np.array_equal(I, Ie)


def test_range_search_minus_inf(fa):
    rng = np.random.default_rng(3)
    n = 50_000
    xb = unit_rows(rng, n, 64)
    xq = unit_rows(rng, 3, 64)
    dev, host = pair(fa, xb)
    lims, D, I, st = range_both(dev, host, xq, float("-inf"), AUTO)
    assert lims.tolist() == [0, n, 2 * n, 3 * n]
    le, De, Ie, _ = range_both(dev, host, xq, float("-inf"), EXACT)
    assert np.array_equal(D, De) and np.array_equal(I, Ie)


def test_device_pointer_entry_points(fa):
    import torch

    rng = np.random.default_rng(12)
    xb, xq = unit_rows(rng, 30000, 256), unit_rows(rng, 4, 256)
    dev, host = pair(fa, xb)
    q = _cuda(xq, host)
    Dd, Id = dev.search_device(q, 10, id_offset=1000)
    Dh, Ih = host.search_device(q, 10, id_offset=1000)
    assert torch.equal(Dd, Dh) and torch.equal(Id, Ih)
    Da, Ia = host.search_device_async(q, 10, id_offset=1000)
    host.finish()
    assert torch.equal(Da, Dd) and torch.equal(Ia, Id)
    for _ in range(2):  # capture, then replay
        Dg, Ig = host.search_device_graph(q, 10, id_offset=1000)
        assert torch.equal(Dg, Dd) and torch.equal(Ig, Id)
    assert int(Ih.min()) >= 1000


def test_adds_reconstruct_save_and_load(fa, tmp_path):
    rng = np.random.default_rng(13)
    xb, xq = unit_rows(rng, 12000, 256), unit_rows(rng, 20, 256)
    dev = fa.IndexFlatIP(256, master="device")
    host = fa.IndexFlatIP(256, master="host")
    for ix in (dev, host):
        ix.add(xb[:5000])                                  # host rows
        ix.add_device(_cuda(xb[5000:9000], ix))            # device rows
        for lo in range(9000, 12000, 250):                 # many small adds
            ix.add(xb[lo:lo + 250])
    assert host.ntotal == 12000
    assert np.array_equal(host.reconstruct_n(0, 12000), xb)
    assert np.array_equal(host.reconstruct(777), xb[777])
    same_search(dev, host, xq, 10, AUTO)
    pd, ph = tmp_path / "dev.faiss", tmp_path / "host.faiss"
    fa.write_index(dev, str(pd))
    fa.write_index(host, str(ph))
    assert pd.read_bytes() == ph.read_bytes()
    host2 = fa.read_index(str(pd), master="host")
    dev2 = fa.read_index(str(ph), master="device")
    assert host2.master == "host" and dev2.master == "device"
    same_search(dev2, host2, xq, 10, AUTO)
    same_search(dev, host2, xq, 10, AUTO)
    assert np.array_equal(host2.reconstruct_n(0, 12000), xb)
    host.reset()
    assert host.master == "host" and host.ntotal == 0 and host.storage_bytes()["host"] == 0
    host.add(xb)
    same_search(dev, host, xq, 10, AUTO)


def test_storage_bytes(fa):
    rng = np.random.default_rng(14)
    n, d = 40000, 512
    xb = unit_rows(rng, n, d)
    dev, host = pair(fa, xb)
    sd, sh = dev.storage_bytes(), host.storage_bytes()
    assert sd["host"] == 0 and sd["device"] >= n * d * 6
    assert sh["host"] >= n * d * 4
    # the shadow alone: rows rounded up to 128-row tiles, bytes up to the device's mapping granularity (a few MiB)
    tile_rows = -(-n // 128) * 128
    gran = 32 << 20
    assert n * d * 2 <= sh["device"] <= -(-(tile_rows * d * 2) // gran) * gran, sh
    assert sh["device"] < sd["device"]


def test_kirag_master_env_through_as_faiss_and_indexer(fa, monkeypatch, tmp_path):
    import kirag_b200.as_faiss  # noqa: F401  (installs the module as `faiss`)
    from kirag_b200.index import Indexer

    faiss = sys.modules["faiss"]
    rng = np.random.default_rng(15)
    xb, xq = unit_rows(rng, 5000, 128), unit_rows(rng, 3, 128)
    ref = fa.IndexFlatIP(128, master="device")
    ref.add(xb)
    Dr, Ir = ref.search(xq, 5)
    monkeypatch.setenv("KIRAG_MASTER", "host")
    ix = faiss.IndexFlatIP(128)
    assert ix.master == "host"
    ix.add(xb)
    D, I = ix.search(xq, 5)
    assert np.array_equal(D, Dr) and np.array_equal(I, Ir)
    indexer = Indexer(128)
    assert indexer.index.master == "host"
    indexer.index_data([str(100 + i) for i in range(5000)], xb)
    res = indexer.search_knn(xq, 5)
    assert [r[0] for r in res] == [[str(100 + j) for j in row] for row in Ir.tolist()]
    os.makedirs(tmp_path / "ix", exist_ok=True)
    indexer.serialize(str(tmp_path / "ix"))
    back = Indexer(128)
    back.deserialize_from(str(tmp_path / "ix"))
    assert back.index.master == "host" and back.index.ntotal == 5000
    res2 = back.search_knn(xq, 5)
    assert [r[0] for r in res2] == [r[0] for r in res]
    assert all(np.array_equal(a[1], b[1]) for a, b in zip(res, res2))


def test_sharded_world_one_equals_the_flat_index(fa):
    import torch

    from kirag_b200.sharded import ShardedFlatIP

    rng = np.random.default_rng(16)
    xb, xq = unit_rows(rng, 20000, 128), unit_rows(rng, 3, 128)
    sh = ShardedFlatIP(128, 20000, rank=0, world_size=1, device=0, master="host")
    assert sh.index.master == "host"
    sh.add_shard(torch.from_numpy(xb).cuda())
    D, I = sh.search(torch.from_numpy(xq).cuda(), 10)
    ref = fa.IndexFlatIP(128, master="device")
    ref.add(xb)
    Dr, Ir = ref.search(xq, 10)
    assert np.array_equal(D.cpu().numpy(), Dr) and np.array_equal(I.cpu().numpy(), Ir)
