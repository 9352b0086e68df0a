"""Multi-device index (IndexFlatIP(devices=[...])): every case builds the same rows in a single-device index and in
multi-device indexes and requires bit-equal results: D/I, range-search lims/D/I, reconstruct and saved files.

Every case runs with G shards on one GPU (devices=[0]*G, G in 1, 2, 3, 8: all of the striping, worker and merge logic
runs on a box with one GPU) and again on distinct GPUs, list(range(min(8, visible))), when at least two are visible."""
import ctypes
import os

import numpy as np
import pytest

from tests.conftest import unit_rows
from tests.helpers import int_corpus
from tests.test_search_gpu import e5_like_rows

pytestmark = pytest.mark.gpu

AUTO, EXACT, FAST = 0, 1, 2
CONFIGS = ["1x0", "2x0", "3x0", "8x0", "distinct"]


@pytest.fixture(scope="module")
def fa():
    from kirag_b200 import faiss_api

    assert faiss_api.get_num_gpus() >= 1, "no CUDA device: the product has no CPU path"
    return faiss_api


def config_devices(fa, name):
    if name == "distinct":
        n = fa.get_num_gpus()
        if n < 2:
            pytest.skip("distinct GPUs: fewer than two visible")
        return list(range(min(8, n)))
    g, dev = name.split("x")
    return [int(dev)] * int(g)


@pytest.fixture(params=CONFIGS)
def devs(request, fa):
    return config_devices(fa, request.param)


def build(fa, xb, devices=None, pieces=None, master=None):
    ix = fa.IndexFlatIP(xb.shape[1], device=None if devices else 0, devices=devices, master=master)
    for lo, hi in (pieces or [(0, len(xb))]):
        ix.add(xb[lo:hi])
    return ix


def same_search(ref, ix, xq, k, path=AUTO, id_offset=0):
    Dr, Ir, _ = ref.search_ex(xq, k, path=path, id_offset=id_offset)
    D, I, st = ix.search_ex(xq, k, path=path, id_offset=id_offset)
    assert np.array_equal(I, Ir), f"k={k} path={path}: ids differ from the single-device index"
    assert np.array_equal(D.view(np.uint32), Dr.view(np.uint32)), f"k={k} path={path}: scores differ"
    assert st["nq"] == len(xq)
    return D, I, st


def range_ex(ix, xq, radius, path=AUTO, id_offset=0):
    from kirag_b200 import _lib

    xq = np.ascontiguousarray(xq, dtype=np.float32)
    n = len(xq)
    lims = np.zeros(n + 1, dtype=np.int64)
    st = _lib.SearchStats()
    _lib.check(ix._lib.kirag_index_range_search(ix._h, xq.ctypes.data, n, float(radius), 0, int(id_offset), path,
                                                lims.ctypes.data, ctypes.byref(st), None), "range_search")
    D = np.empty(int(lims[n]), dtype=np.float32)
    I = np.empty(int(lims[n]), dtype=np.int64)
    _lib.check(ix._lib.kirag_index_range_fetch(ix._h, D.ctypes.data, I.ctypes.data, 0, None), "range_fetch")
    return lims, D, I, st.as_dict()


def same_range(ref, ix, xq, radius, path=AUTO, id_offset=0):
    want = range_ex(ref, xq, radius, path, id_offset)
    got = range_ex(ix, xq, radius, path, id_offset)
    for a, b, what in zip(got[:3], want[:3], ("lims", "D", "I")):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), f"radius={radius} path={path}: range {what} differs"
    return got


def check_shards(ix, devices):
    from kirag_b200 import _lib

    G = len(devices)
    d_out = (ctypes.c_int * G)()
    r_out = (ctypes.c_int64 * G)()
    assert ix._lib.kirag_index_shards(ix._h, d_out, r_out, G) == G
    rows = list(r_out)
    assert list(d_out) == devices and sum(rows) == ix.ntotal and max(rows) - min(rows) <= 128
    want = (ctypes.c_int64 * G)()
    assert _lib.load().kirag_debug_stripe_rows(ix.ntotal, G, want) == 0
    assert rows == list(want)


# ---------------------------------------------------------------------------------------------- unit vectors ----
N_UNIT, D_UNIT = 200_000, 1024


@pytest.fixture(scope="module")
def unit_data():
    rng = np.random.default_rng(901)
    return unit_rows(rng, N_UNIT, D_UNIT)


@pytest.fixture(scope="module")
def unit_ref(fa, unit_data):
    return build(fa, unit_data)


@pytest.fixture(scope="module")
def unit_multi(fa, unit_data):
    cache = {}

    def get(devices):
        key = tuple(devices)
        if key not in cache:
            cache[key] = build(fa, unit_data, devices)
        return cache[key]

    return get


@pytest.fixture(scope="module")
def unit_answers(unit_ref):
    cache = {}

    def get(nq, k, path):
        if (nq, k, path) not in cache:
            xq = unit_rows(np.random.default_rng(nq * 31 + k), nq, D_UNIT)
            cache[(nq, k, path)] = (xq,) + unit_ref.search_ex(xq, k, path=path)
        return cache[(nq, k, path)]

    return get


@pytest.mark.parametrize("config", CONFIGS)
@pytest.mark.parametrize("nq", [1, 32, 128, 300, 4096])
@pytest.mark.parametrize("k", [1, 10, 100, 2048])
def test_search_is_bit_equal(fa, unit_multi, unit_answers, config, nq, k):
    devices = config_devices(fa, config)
    ix = unit_multi(devices)
    assert ix.devices == devices and ix.ntotal == N_UNIT
    for path in (AUTO, EXACT, FAST):
        xq, Dr, Ir, sr = unit_answers(nq, k, path)
        D, I, st = ix.search_ex(xq, k, path=path)
        if path == FAST and len(devices) > 1 and sr["n_cert_fail"] + st["n_cert_fail"] > 0:
            # FAST returns uncertified answers as they are (k = 2048 has no over-fetch), and which queries fail differs
            # with the rows of an index: answers that are exact in both are compared
            _, _, Xi, _ = unit_answers(nq, k, EXACT)
            ok = np.all(Ir == Xi, axis=1) & np.all(I == Xi, axis=1)
            assert np.array_equal(D[ok].view(np.uint32), Dr[ok].view(np.uint32))
            continue
        assert np.array_equal(I, Ir), f"nq={nq} k={k} path={path}: ids differ"
        assert np.array_equal(D.view(np.uint32), Dr.view(np.uint32)), f"nq={nq} k={k} path={path}: scores differ"
        assert st["nq"] == nq and st["kernel_launches"] > 0
        if path == EXACT:
            assert st["n_exact"] == nq * len(devices)


def test_shards_device_entry_points_and_id_offset(fa, unit_multi, unit_ref, unit_data, devs):
    import torch

    ix = unit_multi(devs)
    check_shards(ix, devs)
    xq = unit_rows(np.random.default_rng(5), 64, D_UNIT)
    same_search(unit_ref, ix, xq, 50, id_offset=1_000_000_007)
    Dr, Ir = unit_ref.search(xq, 20)
    qt = torch.from_numpy(xq).cuda(devs[0])
    Dd, Id = ix.search_device(qt, 20)
    assert Dd.device == qt.device and np.array_equal(Id.cpu().numpy(), Ir) and np.array_equal(Dd.cpu().numpy(), Dr)
    # range search on the device entry point, with an id offset
    want = range_ex(unit_ref, xq[:8], 0.1, id_offset=5)
    lims, D, I = ix.range_search_device(qt[:8], 0.1, id_offset=5)
    assert np.array_equal(lims.cpu().numpy(), want[0]) and np.array_equal(D.cpu().numpy(), want[1])
    assert np.array_equal(I.cpu().numpy(), want[2])
    rows = np.array([0, 1, 127, 128, 129, 1000, 70_000, N_UNIT - 1])
    got = np.stack([ix.reconstruct(int(r)) for r in rows])
    assert np.array_equal(got, unit_data[rows])
    assert np.array_equal(ix.reconstruct_n(777, 5000), unit_data[777:5777])
    out = torch.empty((3000, D_UNIT), dtype=torch.float32, device=qt.device)
    from kirag_b200 import _lib

    _lib.check(ix._lib.kirag_index_reconstruct(ix._h, 100_123, 3000, ctypes.c_void_p(out.data_ptr()), 1, None), "rec")
    torch.cuda.synchronize(qt.device)
    assert np.array_equal(out.cpu().numpy(), unit_data[100_123:103_123])


# ------------------------------------------------------------------------------------------- special corpora ----
def fp64_topk(xb, xq, k):
    """The exact answer by (score desc, id asc), scores in fp64 (integer data: exact in fp32 too)."""
    s = xq.astype(np.float64) @ xb.astype(np.float64).T
    m = min(k, xb.shape[0])
    I = np.full((len(xq), k), -1, dtype=np.int64)
    D = np.full((len(xq), k), np.finfo(np.float32).min, dtype=np.float32)
    ids = np.arange(xb.shape[0])
    for i in range(len(xq)):
        order = np.lexsort((ids, -s[i]))[:m]
        I[i, :m] = order
        D[i, :m] = s[i, order]
    return D, I


def test_integer_data_is_exact(fa, devs):
    rng = np.random.default_rng(17)
    xb, xq = int_corpus(rng, 30_000, 1024), int_corpus(rng, 40, 1024)
    ix = build(fa, xb, devs)
    Do, Io = fp64_topk(xb, xq, 100)
    for path in (AUTO, EXACT):
        D, I, _ = ix.search_ex(xq, 100, path=path)
        assert np.array_equal(I, Io) and np.array_equal(D, Do), f"path={path}"


def test_ties_across_shards_come_back_by_ascending_id(fa, devs):
    rng = np.random.default_rng(23)
    xb = unit_rows(rng, 5000, 256)
    dup = [5, 130, 300, 777, 1025, 2100, 4999]  # in different stripes, so on different shards when G > 1
    xb[dup] = xb[5]
    xq = np.concatenate([xb[5:6], unit_rows(rng, 7, 256)])
    ref, ix = build(fa, xb), build(fa, xb, devs)
    for path in (AUTO, EXACT):
        D, I, _ = same_search(ref, ix, xq, 10, path)
        assert I[0, :7].tolist() == dup and np.all(D[0, :7] == D[0, 0])


@pytest.mark.parametrize("n", [1, 100, 300, 128 * 8 + 5])
def test_small_indexes_empty_shards_and_k_beyond_ntotal(fa, devs, n):
    rng = np.random.default_rng(n)
    xb = unit_rows(rng, n, 128)
    xq = unit_rows(rng, 9, 128)
    ref, ix = build(fa, xb), build(fa, xb, devs)
    check_shards(ix, devs)
    for k in (1, 64, 200, 2048):
        for path in (AUTO, EXACT):
            D, I, _ = same_search(ref, ix, xq, k, path)
            if k > n:
                assert np.all(I[:, n:] == -1) and np.all(D[:, n:] == np.finfo(np.float32).min)
    same_range(ref, ix, xq, 0.0)


def test_clustered_corpus_escalates(fa, devs):
    rng = np.random.default_rng(7)
    centers = unit_rows(rng, 8, 128)
    xb = centers[rng.integers(0, 8, 60_000)] + 0.004 * rng.standard_normal((60_000, 128)).astype(np.float32)
    xb = (xb / np.linalg.norm(xb, axis=1, keepdims=True)).astype(np.float32)
    xq = (centers[:4] + 0.01 * unit_rows(rng, 4, 128)).astype(np.float32)
    ref, ix = build(fa, xb), build(fa, xb, devs)
    _, _, st = same_search(ref, ix, xq, 10, AUTO)
    assert st["n_rescan"] + st["n_retry"] + st["n_exact"] >= 1, st  # some shard had to escalate
    same_search(ref, ix, xq, 10, EXACT)


def test_e5_like_corpus(fa, devs):
    rng = np.random.default_rng(11)
    xb, mu = e5_like_rows(rng, 40_000, 1024)
    xq = e5_like_rows(rng, 50, 1024)[0]
    ref, ix = build(fa, xb), build(fa, xb, devs)
    for path in (AUTO, EXACT):
        same_search(ref, ix, xq, 100, path)
    same_range(ref, ix, xq[:5], 0.8)


def test_dimension_without_shadow(fa, devs):
    rng = np.random.default_rng(13)
    xb, xq = unit_rows(rng, 20_000, 100), unit_rows(rng, 33, 100)
    ref, ix = build(fa, xb), build(fa, xb, devs)
    for path in (AUTO, EXACT):
        _, _, st = same_search(ref, ix, xq, 64, path)
        assert st["n_exact"] == 33 * len(devs)
    same_range(ref, ix, xq, 0.2)


def test_incremental_adds_from_host_and_device(fa, devs):
    import torch

    rng = np.random.default_rng(19)
    sizes = [1, 7, 1000, 100_000, 7, 1]
    xb = unit_rows(rng, sum(sizes), 512)
    ref = fa.IndexFlatIP(512, device=0)
    ix = fa.IndexFlatIP(512, devices=devs)
    xq = unit_rows(rng, 20, 512)
    lo = 0
    for i, n in enumerate(sizes):
        ref.add(xb[lo:lo + n])
        if i % 2:
            ix.add_device(torch.from_numpy(xb[lo:lo + n]).cuda(devs[0]))
        else:
            ix.add(xb[lo:lo + n])
        lo += n
        assert ix.ntotal == lo
        check_shards(ix, devs)
        same_search(ref, ix, xq, 10)
    assert np.array_equal(ix.reconstruct_n(0, lo), xb)
    same_search(ref, ix, xq, 2048, EXACT)


# -------------------------------------------------------------------------------------------------- range search ----
def test_range_search(fa, devs, monkeypatch):
    rng = np.random.default_rng(29)
    xb = unit_rows(rng, 100_000, 128)
    u = unit_rows(rng, 1, 128)[0]
    near = rng.choice(100_000, 12_000, replace=False)  # > 1024 hits per shard at G = 8 for the queries along u
    xb[near] = u + 0.3 * unit_rows(rng, 12_000, 128)
    xq = np.concatenate([u[None, :] + 0.05 * unit_rows(rng, 4, 128), unit_rows(rng, 60, 128)]).astype(np.float32)
    ref, ix = build(fa, xb), build(fa, xb, devs)
    for path in (AUTO, EXACT):
        same_range(ref, ix, xq, 0.3, path)
    same_range(ref, ix, xq, 0.3, id_offset=12345)
    monkeypatch.setenv("KIRAG_CAND_CAP", "1024")  # the near queries overflow and take the second pass
    lims, _, _, st = same_range(ref, ix, xq, 0.3)
    assert st["n_overflow"] >= 4 * len(devs) and np.all(np.diff(lims)[:4] > 8000)
    monkeypatch.delenv("KIRAG_CAND_CAP")
    lims, D, I, _ = same_range(ref, ix, xq, float("nan"))
    assert lims[-1] == 0
    # a fetched result is released; the next search drops an unfetched one
    from kirag_b200 import _lib

    assert ix._lib.kirag_index_range_fetch(ix._h, D.ctypes.data, I.ctypes.data, 0, None) != 0
    assert "no range-search result" in _lib.last_error()


def test_range_search_minus_inf_past_one_sort_run_per_shard(fa, devs):
    G = len(devs)
    n = 9000 * G  # every shard holds more than 8192 rows: each shard list goes through the run merges
    rng = np.random.default_rng(31)
    xb = unit_rows(rng, n, 64)
    xb[n - 10:] = xb[3]  # ties far apart, on different shards
    xq = unit_rows(rng, 3, 64)
    ref, ix = build(fa, xb), build(fa, xb, devs)
    lims, D, I, _ = same_range(ref, ix, xq, float("-inf"))
    assert lims.tolist() == [0, n, 2 * n, 3 * n]
    same_range(ref, ix, xq, float("-inf"), path=EXACT)


# ----------------------------------------------------------------------------------------- save / load / master ----
def test_save_and_load_across_kinds(fa, devs, tmp_path):
    rng = np.random.default_rng(37)
    xb = unit_rows(rng, 70_001, 256)
    xq = unit_rows(rng, 16, 256)
    ref, ix = build(fa, xb), build(fa, xb, devs, pieces=[(0, 5), (5, 70_000), (70_000, 70_001)])
    fa.write_index(ref, tmp_path / "single.faiss")
    fa.write_index(ix, tmp_path / "multi.faiss")
    assert (tmp_path / "single.faiss").read_bytes() == (tmp_path / "multi.faiss").read_bytes()
    from_single = fa.read_index(tmp_path / "single.faiss", devices=devs)
    from_multi = fa.read_index(tmp_path / "multi.faiss", device=0)
    assert from_single.devices == devs and from_multi.devices == [0]
    check_shards(from_single, devs)
    same_search(ref, from_single, xq, 100)
    same_search(ref, from_multi, xq, 100)
    fa.write_index(from_single, tmp_path / "again.faiss")
    assert (tmp_path / "again.faiss").read_bytes() == (tmp_path / "single.faiss").read_bytes()


def test_host_master_and_storage_bytes(fa, devs):
    rng = np.random.default_rng(41)
    n, d = 50_000, 512
    xb, xq = unit_rows(rng, n, d), unit_rows(rng, 40, d)
    ref = build(fa, xb)
    dev_ix = build(fa, xb, devs)
    host_ix = build(fa, xb, devs, master="host")
    assert host_ix.master == "host"
    for path in (AUTO, EXACT):
        same_search(ref, host_ix, xq, 100, path)
    same_range(ref, host_ix, xq, 0.1)
    assert np.array_equal(host_ix.reconstruct_n(123, 4567), xb[123:4690])
    sd, sh = dev_ix.storage_bytes(), host_ix.storage_bytes()
    assert sd["host"] == 0 and sd["device"] >= n * d * 6
    assert sh["host"] >= n * d * 4 and n * d * 2 <= sh["device"] < n * d * 4
    host_ix.reset()
    assert host_ix.ntotal == 0 and host_ix.devices == devs and host_ix.master == "host"


# ------------------------------------------------------------------------------------------- KiRAG-facing paths ----
def test_kirag_devices_through_as_faiss(fa, devs, monkeypatch, tmp_path):
    import kirag_b200.as_faiss as af

    faiss = af.make_module()
    monkeypatch.setenv("KIRAG_DEVICES", ",".join(str(v) for v in devs))
    rng = np.random.default_rng(43)
    xb, xq = unit_rows(rng, 20_000, 256), unit_rows(rng, 12, 256)
    ix = faiss.IndexFlatIP(256)
    assert ix.devices == devs
    ix.add(xb)
    ref = fa.IndexFlatIP(256, device=0)
    ref.add(xb)
    same_search(ref, ix, xq, 10)
    faiss.write_index(ix, str(tmp_path / "x.faiss"))
    back = faiss.read_index(str(tmp_path / "x.faiss"), faiss.IO_FLAG_MMAP)
    assert back.devices == devs
    same_search(ref, back, xq, 10)
    ix.reset()
    assert ix.devices == devs and ix.ntotal == 0


def test_reference_indexer_with_kirag_devices(fa, devs, monkeypatch):
    from tests import refenv

    root = refenv.snapshot_root()
    if root is None:
        pytest.skip("baseline/_ref snapshot missing or stale: run __graft_entry__.build() in the build container")
    import kirag_b200.as_faiss as af

    monkeypatch.setenv("KIRAG_DEVICES", ",".join(str(v) for v in devs))
    rng = np.random.default_rng(47)
    xb, xq = unit_rows(rng, 30_000, 1024), unit_rows(rng, 40, 1024)
    with refenv.reference_modules(root, af.make_module()) as ref:
        ix = ref.index.Indexer(1024, "inner_product")
        assert ix.index.devices == devs
        ix.index_data([str(3 * i + 1) for i in range(10_000)], xb[:10_000])
        ix.index_data([str(3 * i + 1) for i in range(10_000, 30_000)], xb[10_000:])
        res = ix.search_knn(xq, 10, verbose=False)
    single = fa.IndexFlatIP(1024, device=0)
    single.add(xb)
    Dr, Ir = single.search(xq, 10)
    assert [r[0] for r in res] == [[str(3 * i + 1) for i in row] for row in Ir]
    assert np.array_equal(np.stack([r[1] for r in res]), Dr)


def test_entry_points_that_raise(fa, devs):
    import torch
    from kirag_b200 import _lib

    rng = np.random.default_rng(53)
    xb = unit_rows(rng, 3000, 128)
    ix = build(fa, xb, devs)
    qt = torch.from_numpy(unit_rows(rng, 4, 128)).cuda(devs[0])
    for call in (lambda: ix.search_device_async(qt, 5), ix.finish, ix.state_token, ix.pending_flags_ptr,
                 lambda: ix.search_device_graph(qt, 5), lambda: ix.debug_scores(xb[:2])):
        with pytest.raises(RuntimeError, match="multi-device"):
            call()
    lib = ix._lib
    D = torch.empty((4, 5), device=qt.device)
    I = torch.empty((4, 5), dtype=torch.int64, device=qt.device)
    assert lib.kirag_index_search_async(ix._h, ctypes.c_void_p(qt.data_ptr()), 4, 5, ctypes.c_void_p(D.data_ptr()),
                                        ctypes.c_void_p(I.data_ptr()), 0, None) != 0
    assert "multi-device" in _lib.last_error()
    for rc in (lib.kirag_index_search_finish(ix._h, None, None), lib.kirag_index_search_rearm(ix._h, None),
               lib.kirag_index_state_token(ix._h, ctypes.byref(ctypes.c_uint64())),
               lib.kirag_index_search_flags(ix._h, ctypes.byref(ctypes.c_void_p())),
               lib.kirag_index_device_ptrs(ix._h, None, None)):
        assert rc != 0 and "multi-device" in _lib.last_error()


_FIRST_SEARCH = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from kirag_b200 import faiss_api
G, k = int(sys.argv[2]), int(sys.argv[3])
rng = np.random.default_rng(G * k)
xb = rng.standard_normal((5000, 64)).astype(np.float32)
xq = rng.standard_normal((9, 64)).astype(np.float32)
ix = faiss_api.IndexFlatIP(64, devices=[0] * G)
ix.add(xb)
D, I = ix.search(xq, k)  # the first merge launch of this process
ref = faiss_api.IndexFlatIP(64, device=0)
ref.add(xb)
Dr, Ir = ref.search(xq, k)
assert np.array_equal(I, Ir) and np.array_equal(D, Dr)
print("ok")
"""


@pytest.mark.parametrize("G,k", [(2, 256), (4, 128), (8, 64), (1, 512), (2, 255)])
def test_merge_just_under_the_shared_memory_opt_in_as_first_search(G, k):
    """G * k near 512: four merge groups need just under 48 KB of dynamic shared memory, which with the kernel's static
    shared memory exceeds the default per-block limit; the first search of a fresh process must work."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ)
    env.pop("KIRAG_DEVICES", None)
    out = subprocess.run([sys.executable, "-c", _FIRST_SEARCH, root, str(G), str(k)], capture_output=True, text=True,
                         env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]
