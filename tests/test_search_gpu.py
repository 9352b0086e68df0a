"""Parity of the CUDA search (through the C ABI) against the oracle / fp64 ground truth.  Needs a B200."""
import os

import numpy as np
import pytest

from oracle import oracle
from tests.conftest import unit_rows
from tests.helpers import assert_topk_parity, exact_topk_f64, int_corpus, load_search_golden

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
LOWEST = np.float32(-3.4028234663852886e38)
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


def bf16_round(a):
    """round-to-nearest-even to bf16, returned as float32 (numpy restatement of __float2bfloat16_rn)."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return r.astype(np.uint32).view(np.float32)


# ---------------------------------------------------------------- edge cases ---
def test_hand_checkable_ties_padding_k1(fa):
    xb = np.array([[3, 0], [1, 5], [3, 9], [0, 1], [3, -2]], dtype=np.float32)
    xq = np.array([[1, 0]], dtype=np.float32)
    ix = build(fa, xb)  # d=2: not a multiple of 64 -> exact path only
    D, I = ix.search(xq, 3)
    assert I.tolist() == [[0, 2, 4]] and D.tolist() == [[3, 3, 3]]
    assert ix.search(xq, 2)[1].tolist() == [[0, 2]]
    assert ix.search(xq, 1)[1].tolist() == [[0]]
    D, I = ix.search(xq, 8)
    assert I.tolist() == [[0, 2, 4, 1, 3, -1, -1, -1]] and np.all(D[0, 5:] == LOWEST)
    assert ix.last_stats["n_exact"] == 1


def test_empty_index_and_empty_queries(fa):
    ix = fa.IndexFlatIP(64)
    assert ix.ntotal == 0 and ix.is_trained
    D, I = ix.search(np.ones((2, 64), dtype=np.float32), 3)
    assert np.all(I == -1) and np.all(D == LOWEST)
    ix.add(np.ones((3, 64), dtype=np.float32))
    D, I = ix.search(np.zeros((0, 64), dtype=np.float32), 3)
    assert D.shape == (0, 3) and I.shape == (0, 3)


def test_argument_errors(fa):
    ix = build(fa, np.ones((4, 64), dtype=np.float32))
    with pytest.raises(AssertionError):
        ix.search(np.ones((1, 32), dtype=np.float32), 3)
    with pytest.raises(AssertionError):
        ix.search(np.ones((1, 64), dtype=np.float32), 0)
    with pytest.raises(AssertionError):
        ix.add(np.ones((1, 63), dtype=np.float32))
    with pytest.raises(RuntimeError):
        ix.search(np.ones((1, 64), dtype=np.float32), 5000)  # k beyond the supported maximum
    with pytest.raises(NotImplementedError):
        fa.IndexFlatL2(64)


# ------------------------------------------------------ tensor-core scores ---
@pytest.mark.parametrize("n,d,nq", [(300, 64, 5), (1000, 128, 32), (777, 1024, 3), (4096, 1024, 40), (513, 256, 100),
                                    (300, 192, 200),
                                    # large d, where the plan streams the 64- / 128-query tiles
                                    (1000, 2560, 5), (1000, 2560, 40), (600, 1536, 100), (300, 4096, 1), (300, 4096, 128)])
def test_tcgen05_scores_match_bf16_reference(fa, n, d, nq):
    """The MMA itself (descriptors, swizzled layout, TMEM read-out): dense approximate scores equal the
    fp32-accumulated product of the bf16-rounded operands."""
    rng = np.random.default_rng(n + d + nq)
    xb = rng.standard_normal((n, d)).astype(np.float32)
    xq = rng.standard_normal((nq, d)).astype(np.float32)
    ix = build(fa, xb)
    got = ix.debug_scores(xq)  # [n, nq]
    ref = bf16_round(xb).astype(np.float64) @ bf16_round(xq).astype(np.float64).T
    scale = np.linalg.norm(xb, axis=1)[:, None] * np.linalg.norm(xq, axis=1)[None, :]
    assert got.shape == (n, nq)
    assert np.max(np.abs(got - ref) / scale) < 2e-6  # fp32 accumulation of exact bf16 products


@pytest.mark.parametrize("code,n,d,nq", [("64r", 1300, 256, 1), ("64r", 1300, 256, 40), ("64s", 1300, 256, 5),
                                         ("64s", 1300, 256, 40), ("128r", 1300, 256, 100), ("128s", 1300, 256, 65),
                                         ("128s", 1300, 256, 100), ("256s", 1300, 256, 200), ("256s", 1300, 256, 300),
                                         # ragged tile groups at three d
                                         ("256s", 3000, 128, 260), ("256s", 1100, 1024, 600), ("256s", 129, 64, 257)])
def test_every_scan_kernel_variant_scores_match_bf16_reference(fa, monkeypatch, code, n, d, nq):
    """Every instantiation of the scan kernel, forced through KIRAG_DEBUG_BQ (the default plan only exercises the ones
    it picks at the dimension of the index): 64 / 128-query tiles resident (r) and streamed (s), 256-query tiles
    streamed."""
    monkeypatch.setenv("KIRAG_DEBUG_BQ", code)
    rng = np.random.default_rng(n + d + nq + len(code))
    xb = rng.standard_normal((n, d)).astype(np.float32)
    xq = rng.standard_normal((nq, d)).astype(np.float32)
    got = build(fa, xb).debug_scores(xq)
    ref = bf16_round(xb).astype(np.float64) @ bf16_round(xq).astype(np.float64).T
    scale = np.linalg.norm(xb, axis=1)[:, None] * np.linalg.norm(xq, axis=1)[None, :]
    assert np.max(np.abs(got - ref) / scale) < 2e-6
    xi, qi = int_corpus(rng, 700, 128), int_corpus(rng, nq, 128)
    goti = build(fa, xi).debug_scores(qi)
    assert np.array_equal(goti, (xi.astype(np.float64) @ qi.astype(np.float64).T).astype(np.float32))


def test_unknown_scan_kernel_variant_is_an_error(fa, monkeypatch):
    monkeypatch.setenv("KIRAG_DEBUG_BQ", "512")
    rng = np.random.default_rng(3)
    ix = build(fa, rng.standard_normal((300, 64)).astype(np.float32))
    with pytest.raises(RuntimeError):
        ix.debug_scores(rng.standard_normal((4, 64)).astype(np.float32))


def test_small_batches_on_the_resident_64_kernel(fa):
    """Batches of up to 64 queries (the resident 64-query tile) and just above: exact answers."""
    rng = np.random.default_rng(77)
    xb = unit_rows(rng, 60000, 128)
    ix = build(fa, xb)
    for nq in (1, 8, 32, 33, 64):
        xq = unit_rows(rng, nq, 128)
        D, I, st = ix.search_ex(xq, 10, path=AUTO)
        assert st["n_fast"] == nq, st
        assert_topk_parity(D, I, xb, xq, 10, what=f"nq={nq} {st}")


@pytest.mark.parametrize("d", [2560, 4096])
def test_large_d_batches_on_the_streamed_small_tiles(fa, d):
    """At d = 2560 / 4096 the default plan streams the 64- and 128-query tiles (the resident query half would leave
    too short a ring).  Each query has k planted neighbours far above the rest, so every first pass certifies and
    the streamed kernels answer every query."""
    rng = np.random.default_rng(d)
    n, k, batches = 40000, 10, (1, 40, 100)
    xb = unit_rows(rng, n, d)
    xq_all = unit_rows(rng, sum(batches), d)
    tgt = rng.choice(n, (len(xq_all), k), replace=False)
    for i in range(len(xq_all)):
        near = xq_all[i][None, :] + 0.3 * unit_rows(rng, k, d)
        xb[tgt[i]] = near / np.linalg.norm(near, axis=1, keepdims=True)
    ix = build(fa, xb)
    q0 = 0
    for nq in batches:
        xq = xq_all[q0:q0 + nq]
        D, I, st = ix.search_ex(xq, k, path=AUTO)
        assert st["n_fast"] == nq, (nq, st)
        assert all(set(I[r]) == set(tgt[q0 + r]) for r in range(nq)), nq
        De, Ie, _ = ix.search_ex(xq, k, path=EXACT)
        assert np.array_equal(I, Ie) and np.array_equal(D, De), (nq, st)
        q0 += nq


def test_tcgen05_scores_exact_on_integers(fa):
    rng = np.random.default_rng(0)
    xb, xq = int_corpus(rng, 1500, 128), int_corpus(rng, 17, 128)
    got = build(fa, xb).debug_scores(xq)
    assert np.array_equal(got, (xb.astype(np.float64) @ xq.astype(np.float64).T).astype(np.float32))


# ------------------------------------------------------------ exact path ---
@pytest.mark.parametrize("n,d,nq,k", [(1000, 64, 5, 10), (300, 100, 3, 100), (50, 30, 4, 64), (20000, 128, 9, 7),
                                      (9000, 1024, 6, 100), (8193, 7, 2, 2048)])
def test_exact_path_integer_data_bit_exact(fa, n, d, nq, k):
    rng = np.random.default_rng(n + d)
    xb, xq = int_corpus(rng, n, d), int_corpus(rng, nq, d)
    D, I, st = build(fa, xb).search_ex(xq, k, path=EXACT)
    assert st["n_exact"] == nq and st["n_fast"] == 0
    assert_topk_parity(D, I, xb, xq, k, exact=True, what="exact path")
    Do, Io = oracle.flat_ip_search(xb, xq, k)
    assert np.array_equal(I, Io) and np.array_equal(D, Do)


@pytest.mark.parametrize("n,d,nq,k", [(5000, 96, 9, 20), (30000, 1024, 5, 100), (100, 1024, 2, 10)])
def test_exact_path_unit_vectors(fa, n, d, nq, k):
    rng = np.random.default_rng(n)
    xb, xq = unit_rows(rng, n, d), unit_rows(rng, nq, d)
    D, I, _ = build(fa, xb).search_ex(xq, k, path=EXACT)
    assert_topk_parity(D, I, xb, xq, k, what="exact path")


# ---------------------------------------------------------- filter (fast) path ---
@pytest.mark.parametrize("n,d,nq,k", [(1000, 64, 5, 10), (5000, 128, 32, 10), (20000, 64, 33, 20), (70000, 128, 7, 100),
                                      (3000, 1024, 130, 10), (40000, 256, 300, 5), (129, 64, 1, 3), (127, 64, 2, 200)])
def test_auto_path_integer_data_bit_exact(fa, n, d, nq, k):
    rng = np.random.default_rng(n * 3 + d)
    xb, xq = int_corpus(rng, n, d), int_corpus(rng, nq, d)
    D, I, st = build(fa, xb).search_ex(xq, k, path=AUTO)
    assert st["n_fast"] + st["n_exact"] == nq
    assert_topk_parity(D, I, xb, xq, k, exact=True, what=f"auto path {st}")
    Do, Io = oracle.flat_ip_search(xb, xq, k)
    assert np.array_equal(I, Io) and np.array_equal(D, Do)


@pytest.mark.parametrize("n,d,nq,k", [(100000, 128, 16, 10), (50000, 1024, 8, 20), (200000, 64, 64, 100),
                                      (60000, 1024, 256, 20), (30000, 768, 1, 10),
                                      # every kernel variant of the filter scan: resident 64-query tile,
                                      # 2-CTA resident 128-query tile (65..128 queries), 2-CTA 256-query tiles
                                      (70000, 1024, 64, 10), (80000, 1024, 100, 10), (50000, 256, 128, 20),
                                      (40000, 1024, 65, 20), (40000, 1024, 700, 10)])
def test_auto_path_unit_vectors_uses_the_filter(fa, n, d, nq, k):
    rng = np.random.default_rng(n + k)
    xb, xq = unit_rows(rng, n, d), unit_rows(rng, nq, d)
    ix = build(fa, xb)
    D, I, st = ix.search_ex(xq, k, path=AUTO)
    assert st["n_fast"] >= nq * 0.9, st  # i.i.d. data: the certificate passes
    assert st["levels"] >= 2 and st["n_overflow"] == 0, st
    n_swaps = assert_topk_parity(D, I, xb, xq, k, what=f"auto path {st}")
    # the two paths return bit-identical scores (canonical summation order) and ids
    De, Ie, _ = ix.search_ex(xq, k, path=EXACT)
    assert np.array_equal(I, Ie) and np.array_equal(D, De), f"fast vs exact differ (near-tie swaps vs fp64: {n_swaps})"


@pytest.mark.parametrize("n,nq,k", [(20000, 8, 10), (70000, 64, 10), (70000, 129, 10), (300000, 4, 100), (300000, 300, 100)])
def test_levels_follow_the_host_schedule(fa, n, nq, k):
    """The number of filter launches of a search equals the host-side schedule hook (tests/test_host_logic.py
    checks that hook's invariants on CPU)."""
    import ctypes

    from kirag_b200 import _lib

    rng = np.random.default_rng(n + nq)
    xb, xq = unit_rows(rng, n, 128), unit_rows(rng, nq, 128)
    D, I, st = build(fa, xb).search_ex(xq, k, path=AUTO)
    out = (ctypes.c_int64 * 64)()
    n_levels = _lib.load().kirag_debug_level_schedule(n, nq, k, 128, out, 64, None, None)
    assert st["levels"] == n_levels and out[n_levels - 1] == n, (st, n_levels)
    assert_topk_parity(D, I, xb, xq, k, what=f"schedule {st}")


def test_fast_path_without_escalation_reports_certificate(fa):
    rng = np.random.default_rng(5)
    xb, xq = unit_rows(rng, 50000, 128), unit_rows(rng, 12, 128)
    D, I, st = build(fa, xb).search_ex(xq, 10, path=FAST)
    assert st["n_exact"] == 0 and st["n_fast"] == 12
    assert_topk_parity(D, I, xb, xq, 10, what="fast path")


def test_duplicates_lower_id_wins(fa):
    rng = np.random.default_rng(6)
    xb = unit_rows(rng, 30000, 128)
    src = rng.choice(30000, 300, replace=False)
    dst = rng.choice(30000, 300, replace=False)
    xb[dst] = xb[src]
    xq = xb[src[:8]] + 0.05 * rng.standard_normal((8, 128)).astype(np.float32)
    D, I, st = build(fa, xb).search_ex(xq, 10, path=AUTO)
    assert_topk_parity(D, I, xb, xq, 10, what=f"duplicates {st}")
    for r in range(8):
        ids, sc = I[r].tolist(), D[r].tolist()
        for a in range(9):
            if sc[a] == sc[a + 1]:
                assert ids[a] < ids[a + 1]


def test_clustered_data_escalates_and_stays_exact(fa, monkeypatch):
    """Clusters: rank-k and rank-4k scores are closer than the bf16 error bound, so the certificate
    must fail.  First escalation = one more bf16 pass with the provable threshold s_k - eps
    (n_rescan); if more rows than the buffer holds lie within eps, the exact fp32 scan answers
    (n_exact).  Results stay exact either way."""
    rng = np.random.default_rng(7)
    centers = unit_rows(rng, 8, 128)
    # moderately tight clusters: a few hundred rows within eps of the k-th score -> rescan succeeds
    xb = centers[rng.integers(0, 8, 40000)] + 0.004 * rng.standard_normal((40000, 128)).astype(np.float32)
    xb = (xb / np.linalg.norm(xb, axis=1, keepdims=True)).astype(np.float32)
    xq = (centers[:4] + 0.01 * unit_rows(rng, 4, 128)).astype(np.float32)
    ix = build(fa, xb)
    D, I, st = ix.search_ex(xq, 10, path=AUTO)
    assert st["n_cert_fail"] >= 1 and st["n_rescan"] + st["n_exact"] + st["n_retry"] == st["n_cert_fail"] + st["n_overflow"], st
    assert st["n_rescan"] >= 1, st
    assert_topk_parity(D, I, xb, xq, 10, what=f"clustered {st}")
    De, Ie, _ = ix.search_ex(xq, 10, path=EXACT)
    assert np.array_equal(I, Ie) and np.array_equal(D, De)
    # degenerate clusters: thousands of rows within eps -> the rescan buffer overflows -> exact scan
    xb2 = centers[rng.integers(0, 8, 80000)] + 1e-5 * rng.standard_normal((80000, 128)).astype(np.float32)
    xb2 = (xb2 / np.linalg.norm(xb2, axis=1, keepdims=True)).astype(np.float32)
    D, I, st = build(fa, xb2).search_ex(centers[:3], 10, path=AUTO)
    assert st["n_exact"] >= 1, st
    assert_topk_parity(D, I, xb2, centers[:3], 10, what=f"degenerate clusters {st}")
    # the rescan can be switched off: the same queries then go straight to the exact scan
    monkeypatch.setenv("KIRAG_NO_RESCAN", "1")
    D2, I2, st2 = ix.search_ex(xq, 10, path=AUTO)
    assert st2["n_rescan"] == 0 and st2["n_exact"] >= 1, st2
    assert np.array_equal(I2, Ie) and np.array_equal(D2, De)


def test_sorted_corpus_is_not_pathological(fa):
    """Rows sorted by similarity to the query (best last): the permuted tile walk keeps levels representative."""
    rng = np.random.default_rng(8)
    xb, xq = unit_rows(rng, 100000, 64), unit_rows(rng, 1, 64)
    order = np.argsort(xb @ xq[0])
    xb = np.ascontiguousarray(xb[order])
    D, I, st = build(fa, xb).search_ex(xq, 10, path=AUTO)
    assert_topk_parity(D, I, xb, xq, 10, what=f"sorted {st}")
    # position-sorted rows make every 128-row tile a narrow score band; an overflow is answered by
    # the exact scan (still correct), it must just not be the norm
    xq2 = unit_rows(rng, 8, 64)
    D, I, st = build(fa, xb).search_ex(xq2, 10, path=AUTO)
    assert st["n_overflow"] <= 1, st
    assert_topk_parity(D, I, xb, xq2, 10, what=f"sorted, other queries {st}")


def test_all_equal_scores_overflow_falls_back(fa):
    xb = np.ones((50000, 64), dtype=np.float32)
    xq = np.ones((2, 64), dtype=np.float32)
    D, I, st = build(fa, xb).search_ex(xq, 10, path=AUTO)
    assert I.tolist() == [list(range(10))] * 2 and np.all(D == 64.0)
    assert st["n_exact"] == 2, st


def test_planted_neighbours(fa):
    rng = np.random.default_rng(10)
    xb = unit_rows(rng, 80000, 256)
    tgt = rng.choice(80000, 20, replace=False)
    xq = xb[tgt] + 0.3 * unit_rows(rng, 20, 256)
    xq = (xq / np.linalg.norm(xq, axis=1, keepdims=True)).astype(np.float32)
    D, I, st = build(fa, xb).search_ex(xq, 20, path=AUTO)
    assert np.array_equal(I[:, 0], tgt)
    assert_topk_parity(D, I, xb, xq, 20, what=f"planted {st}")


# ----------------------------------------------------------- index plumbing ---
def test_incremental_add_growth_and_reconstruct(fa):
    rng = np.random.default_rng(11)
    xb = int_corpus(rng, 5000, 64)
    ix = fa.IndexFlatIP(64)
    for a, b in ((0, 1), (1, 130), (130, 131), (131, 3000), (3000, 5000)):
        ix.add(xb[a:b])
    assert ix.ntotal == 5000
    assert np.array_equal(ix.reconstruct_n(0, 5000), xb)
    assert np.array_equal(ix.reconstruct(4321), xb[4321])
    xq = int_corpus(rng, 6, 64)
    D, I, _ = ix.search_ex(xq, 10, path=AUTO)
    assert_topk_parity(D, I, xb, xq, 10, exact=True)


def test_id_offset(fa):
    rng = np.random.default_rng(12)
    xb, xq = int_corpus(rng, 2000, 64), int_corpus(rng, 3, 64)
    ix = build(fa, xb)
    D0, I0, _ = ix.search_ex(xq, 2040, path=EXACT)
    D1, I1, _ = ix.search_ex(xq, 2040, path=EXACT, id_offset=10**10)
    assert np.array_equal(D0, D1)
    assert np.array_equal(np.where(I0 >= 0, I0 + 10**10, -1), I1)


def test_save_load_roundtrip_and_container_is_ixfi(fa, tmp_path):
    rng = np.random.default_rng(13)
    xb, xq = unit_rows(rng, 3000, 64), unit_rows(rng, 4, 64)
    ix = build(fa, xb)
    p = str(tmp_path / "index.faiss")
    fa.write_index(ix, p)
    raw = open(p, "rb").read()
    assert raw[:4] == b"IxFI" and len(raw) == 45 + xb.nbytes
    ox = oracle._read_index(p)  # an independent reader of the same container
    assert np.array_equal(ox.reconstruct_n(), xb)
    ix2 = fa.read_index(p, fa.IO_FLAG_MMAP)
    assert ix2.ntotal == 3000 and ix2.d == 64
    D1, I1 = ix.search(xq, 10)
    D2, I2 = ix2.search(xq, 10)
    assert np.array_equal(I1, I2) and np.array_equal(D1, D2)
    # and the reverse: a file written by the independent writer loads here
    p2 = str(tmp_path / "other.faiss")
    oracle._write_index(ox, p2)
    assert np.array_equal(fa.read_index(p2).reconstruct_n(), xb)
    with pytest.raises(RuntimeError):
        fa.read_index(str(tmp_path / "missing.faiss"))


def test_search_golden_fixture(fa):
    z = load_search_golden()
    for name in ("unit_64", "unit_1024", "kgtn", "ties"):
        xb, xq, k = z[f"{name}_xb"], z[f"{name}_xq"], int(z[f"{name}_k"])
        ix = build(fa, xb)
        for path in (AUTO, EXACT):
            D, I, st = ix.search_ex(xq, k, path=path)
            assert np.array_equal(I, z[f"{name}_I"]), (name, path, st)
            np.testing.assert_allclose(D, z[f"{name}_D"], rtol=1e-5, atol=1e-6)
            if name == "ties":
                assert np.array_equal(D, z[f"{name}_D"])


def test_aligner_scoring_matches_reference_torch_golden(fa):
    from kirag_b200.scoring import filter_candidate_triples_scores

    z = np.load(os.path.join(GOLD, "aligner_golden.npz"))
    for name in ("s", "m", "few"):
        q, t, k = z[f"{name}_q"], z[f"{name}_t"], int(z[f"{name}_k"])
        idx, sc = filter_candidate_triples_scores(q, t, k)
        ref_s, ref_i = z[f"{name}_scores"], z[f"{name}_indices"]
        assert np.asarray(sc).shape == ref_s.shape
        np.testing.assert_allclose(np.asarray(sc, dtype=np.float32), ref_s, rtol=1e-5, atol=1e-6)
        for r in range(q.shape[0]):
            assert set(idx[r]) == set(ref_i[r].tolist())


@pytest.mark.parametrize("C,T,d,k", [(1, 137, 1024, 20), (2, 900, 1024, 20), (8, 5000, 256, 7), (2, 12, 64, 20),
                                     (3, 8192, 128, 50), (3, 8193, 128, 50)])
def test_aligner_real_shape_runs_on_the_callers_matrix(fa, C, T, d, k):
    """KiRAG's own aligner shape (1-2 chain queries x 10^2-10^3 triples, models.py:1514-1542): kirag_topk_ip scans the
    caller's matrix in place (no transient index) — same canonical scores and order as the index path, from host and
    from device buffers, ties by lower index, k > T clipped by the Python surface."""
    import torch

    from kirag_b200.scoring import topk_inner_product

    rng = np.random.default_rng(C * 1000 + T)
    t, q = unit_rows(rng, T, d), unit_rows(rng, C, d)
    t[T // 2] = t[T // 3]  # an exact tie
    D, I = topk_inner_product(q, t, k)
    kk = min(k, T)
    assert D.shape == (C, kk) and I.shape == (C, kk)
    assert_topk_parity(D, I, t, q, kk, what=f"aligner {C}x{T}")
    Dd, Id = topk_inner_product(torch.from_numpy(q).cuda(), torch.from_numpy(t).cuda(), k)
    assert np.array_equal(Id.cpu().numpy(), I) and np.array_equal(Dd.cpu().numpy(), D)
    ix = build(fa, t)  # the index path gives bit-identical scores
    Di, Ii, _ = ix.search_ex(q, kk, path=EXACT)
    assert np.array_equal(Ii, I) and np.array_equal(Di, D)


def test_aligner_scoring_accepts_unaligned_device_views(fa):
    """Views with a storage offset that is not a multiple of 16 bytes (ADVICE r1): copied, not faulted on."""
    import torch

    from kirag_b200.scoring import topk_inner_product

    rng = np.random.default_rng(91)
    t, q = unit_rows(rng, 20000, 64), unit_rows(rng, 3, 64)
    tb = torch.zeros(20000 * 64 + 1, dtype=torch.float32, device="cuda")
    qb = torch.zeros(3 * 64 + 3, dtype=torch.float32, device="cuda")
    tv, qv = tb[1:].view(20000, 64), qb[3:].view(3, 64)
    tv.copy_(torch.from_numpy(t))
    qv.copy_(torch.from_numpy(q))
    assert tv.data_ptr() % 16 != 0 and qv.data_ptr() % 16 != 0
    D, I = topk_inner_product(qv, tv, 20)
    assert_topk_parity(D.cpu().numpy(), I.cpu().numpy(), t, q, 20, what="unaligned views")
    D2, I2 = topk_inner_product(qv, tv[:500], 20)  # the in-place small-shape path
    assert_topk_parity(D2.cpu().numpy(), I2.cpu().numpy(), t[:500], q, 20, what="unaligned views, in place")


def test_config4_aligner_shape(fa):
    """BASELINE configs[4]: 256 chain queries x 50k candidate triples, top-20."""
    rng = np.random.default_rng(14)
    t, q = unit_rows(rng, 50000, 1024), unit_rows(rng, 256, 1024)
    from kirag_b200.scoring import topk_inner_product

    D, I = topk_inner_product(q, t, 20)
    assert_topk_parity(D, I, t, q, 20, what="aligner 256x50k")


def test_device_pointer_entry_points(fa):
    import torch

    rng = np.random.default_rng(15)
    xb, xq = unit_rows(rng, 40000, 128), unit_rows(rng, 10, 128)
    ix = fa.IndexFlatIP(128)
    ix.add_device(torch.from_numpy(xb).cuda())
    D, I = ix.search_device(torch.from_numpy(xq).cuda(), 10, id_offset=5)
    torch.cuda.synchronize()
    assert_topk_parity(D.cpu().numpy(), I.cpu().numpy() - 5, xb, xq, 10, what="device pointers")


# ------------------------------------------------- asynchronous search (async + finish) ---
def test_async_search_then_finish_equals_the_synchronous_call(fa):
    """kirag_index_search_async enqueues the first attempt without a host synchronisation;
    kirag_index_search_finish verifies the certificates and re-answers flagged queries in place."""
    import torch

    rng = np.random.default_rng(21)
    # (a) well-spread data: every certificate passes, finish() changes nothing
    xb, xq = unit_rows(rng, 60000, 256), unit_rows(rng, 40, 256)
    ix = build(fa, xb)
    q = torch.from_numpy(xq).cuda()
    Ds, Is = ix.search_device(q, 20)
    Da, Ia = ix.search_device_async(q, 20)
    assert ix.pending_flags_ptr() != 0
    changed = ix.finish()
    assert changed == 0 and ix.last_stats["n_fast"] == 40, ix.last_stats
    assert torch.equal(Ia, Is) and torch.equal(Da, Ds)
    assert ix.pending_flags_ptr() == 0 and ix.finish() == 0  # nothing pending any more
    # (b) clustered data: the certificates fail, finish() rewrites those rows and the result is the exact one
    centers = unit_rows(rng, 8, 128)
    xc = centers[rng.integers(0, 8, 40000)] + 0.004 * rng.standard_normal((40000, 128)).astype(np.float32)
    xc = (xc / np.linalg.norm(xc, axis=1, keepdims=True)).astype(np.float32)
    qc = torch.from_numpy((centers[:4] + 0.01 * unit_rows(rng, 4, 128)).astype(np.float32)).cuda()
    ic = build(fa, xc)
    De, Ie = ic.search_device(qc, 10, path=EXACT)
    Da, Ia = ic.search_device_async(qc, 10)
    changed = ic.finish()
    st = ic.last_stats
    assert changed >= 1 and st["n_cert_fail"] >= 1 and st["n_rescan"] + st["n_exact"] + st["n_retry"] == changed, st
    assert torch.equal(Ia, Ie) and torch.equal(Da, De)
    # (c) an unfinished asynchronous search is completed by the next call on the handle
    Da, Ia = ic.search_device_async(qc, 10)
    Ds2, Is2 = ic.search_device(qc[:2].contiguous(), 10)
    torch.cuda.synchronize()
    assert torch.equal(Ia, Ie) and torch.equal(Is2, Ie[:2])


def test_async_search_is_cuda_graph_capturable(fa):
    """Once the workspaces are warm the asynchronous half allocates nothing and never synchronises: it can be
    captured into a CUDA graph and replayed on new query contents."""
    import torch

    rng = np.random.default_rng(22)
    xb = unit_rows(rng, 80000, 128)
    ix = build(fa, xb)
    q = torch.from_numpy(unit_rows(rng, 8, 128)).cuda()
    ix.search_device(q, 10)  # warm the workspaces
    D = torch.empty((8, 10), dtype=torch.float32, device="cuda")
    I = torch.empty((8, 10), dtype=torch.int64, device="cuda")
    import ctypes

    from kirag_b200 import _lib

    lib = _lib.load()
    stream = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            _lib.check(lib.kirag_index_search_async(ix._h, ctypes.c_void_p(q.data_ptr()), 8, 10, ctypes.c_void_p(D.data_ptr()),
                                                    ctypes.c_void_p(I.data_ptr()), 0, ctypes.c_void_p(stream.cuda_stream)),
                       "search_async (captured)")
    for trial in range(3):
        q.copy_(torch.from_numpy(unit_rows(rng, 8, 128)))
        graph.replay()
        stream.synchronize()
        torch.cuda.synchronize()
        assert_topk_parity(D.cpu().numpy(), I.cpu().numpy(), xb, q.cpu().numpy(), 10, what=f"graph replay {trial}")
    assert ix.finish() == 0  # the captured call left a pending search behind: complete it


def test_graph_replayed_search_equals_the_plain_call_and_recaptures_when_the_index_changes(fa):
    """IndexFlatIP.search_device_graph: one CUDA-graph launch per call.  Same ids and scores as search_device on new
    query contents; adding rows changes the state token and forces a new capture; queries whose certificate fails
    in a replay are re-answered by finish() like in the plain call."""
    import torch

    rng = np.random.default_rng(31)
    xb = unit_rows(rng, 90000, 128)
    ix = build(fa, xb[:60000])
    for trial in range(3):
        q = torch.from_numpy(unit_rows(rng, 5, 128)).cuda()
        Dg, Ig = ix.search_device_graph(q, 10)
        Dg, Ig = Dg.clone(), Ig.clone()
        Dp, Ip = ix.search_device(q, 10)
        assert torch.equal(Ig, Ip) and torch.equal(Dg, Dp), trial
        assert_topk_parity(Dg.cpu().numpy(), Ig.cpu().numpy(), xb[:60000], q.cpu().numpy(), 10, what=f"graph {trial}")
    assert len(ix._graphs) == 1
    tok = ix.state_token()
    ix.add(xb[60000:])
    assert ix.state_token() != tok
    q = torch.from_numpy(unit_rows(rng, 5, 128)).cuda()
    Dg, Ig = ix.search_device_graph(q, 10)
    assert_topk_parity(Dg.cpu().numpy(), Ig.cpu().numpy(), xb, q.cpu().numpy(), 10, what="after add")
    # certificate failures inside a replay: tight clusters (rank k and rank 4k nearly tie)
    centers = unit_rows(rng, 64, 128)
    xc = centers[rng.integers(0, 64, 60000)] + 0.01 * unit_rows(rng, 60000, 128)
    xc = (xc / np.linalg.norm(xc, axis=1, keepdims=True)).astype(np.float32)
    ic = build(fa, xc)
    for trial in range(2):
        qc = torch.from_numpy((centers[trial * 4:trial * 4 + 4] + 0.01 * unit_rows(rng, 4, 128)).astype(np.float32)).cuda()
        Dg, Ig = ic.search_device_graph(qc, 10)
        st = ic.last_stats
        assert st["n_cert_fail"] + st["n_overflow"] >= 1, st
        De, Ie = ic.search_device(qc, 10, path=EXACT)
        assert torch.equal(Ig, Ie) and torch.equal(Dg, De), trial


def test_k_above_512_stays_on_the_filter_path(fa):
    """k' = min(4k, 2048): k up to 2048 is answered by the tcgen05 filter path, not by the fp32 scan."""
    rng = np.random.default_rng(23)
    xb, xq = unit_rows(rng, 150000, 128), unit_rows(rng, 3, 128)
    ix = build(fa, xb)
    for k in (600, 2048):
        D, I, st = ix.search_ex(xq, k, path=AUTO)
        assert st["levels"] >= 2 and st["n_fast"] + st["n_rescan"] + st["n_exact"] + st["n_retry"] == 3, st
        assert st["n_exact"] == 0, st
        assert_topk_parity(D, I, xb, xq, k, what=f"k={k} {st}")


# ------------------------------------------------------- centred shadow / escalation ladder ---
def e5_like_rows(rng, n, d, common=0.85):
    """Rows with a large common component, like E5 embeddings (random-pair cosine ~ common^2 = 0.72)."""
    mu = unit_rows(rng, 1, d)[0]
    noise = rng.standard_normal((n, d)).astype(np.float32)
    noise -= (noise @ mu)[:, None] * mu[None, :]
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    x = common * mu[None, :] + np.sqrt(1.0 - common * common) * noise
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32), mu


def test_e5_like_corpus_is_centred_and_certified(fa, monkeypatch):
    """Embeddings with a large common component: the shadow stores bf16(x - c), the certificate bound scales with
    ||x - c||, and (nearly) every query is certified on the first attempt; without centring the same corpus fails
    its certificates and pays a second pass.  Results are the exact ones either way."""
    rng = np.random.default_rng(31)
    common = 0.93  # random-pair cosine 0.86: the rank-100 / rank-400 gap (~0.0024) is below the uncentred bound (~0.0027)
    xb, mu = e5_like_rows(rng, 300_000, 512, common)
    noise = np.random.default_rng(32).standard_normal((64, 512)).astype(np.float32)
    noise -= (noise @ mu)[:, None] * mu[None, :]
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    xq = (common * mu[None, :] + np.sqrt(1.0 - common * common) * noise).astype(np.float32)
    xq /= np.linalg.norm(xq, axis=1, keepdims=True)
    assert float(np.mean(xb[:1000] @ xb[1000:2000].T)) > 0.8
    ix = build(fa, xb)
    D, I, st = ix.search_ex(xq, 100, path=AUTO)
    assert st["n_fast"] >= 62, f"centred shadow should certify on the first attempt: {st}"
    De, Ie, _ = ix.search_ex(xq, 100, path=EXACT)
    assert np.array_equal(I, Ie) and np.array_equal(D, De)
    assert_topk_parity(D[:8], I[:8], xb, xq[:8], 100, what=f"e5-like {st}")
    # the approximate scores the hook reports are still approximations of <q, x> (the centre is added back)
    approx = ix.debug_scores(xq[:4])[:5000]
    assert np.max(np.abs(approx - xb[:5000] @ xq[:4].T)) < 5e-3
    # the same corpus without centring: certificates fail (that is what the centre is for), answers stay exact
    monkeypatch.setenv("KIRAG_NO_CENTER", "1")
    raw = build(fa, xb)
    D2, I2, st2 = raw.search_ex(xq, 100, path=AUTO)
    assert st2["n_cert_fail"] > st["n_cert_fail"] + 16, (st, st2)
    assert np.array_equal(I2, Ie) and np.array_equal(D2, De)


def test_centre_is_decided_late_for_small_first_adds(fa):
    """The centring decision waits until 4096 rows are there; rows converted before it are re-converted."""
    rng = np.random.default_rng(33)
    xb, mu = e5_like_rows(rng, 20000, 128)
    ix = fa.IndexFlatIP(128)
    for a, b in ((0, 100), (100, 3000), (3000, 4096), (4096, 20000)):
        ix.add(xb[a:b])
    xq = xb[::1500] + 0.01 * rng.standard_normal((14, 128)).astype(np.float32)
    D, I, st = ix.search_ex(xq.astype(np.float32), 10, path=AUTO)
    De, Ie, _ = ix.search_ex(xq.astype(np.float32), 10, path=EXACT)
    assert np.array_equal(I, Ie) and np.array_equal(D, De), st
    approx = ix.debug_scores(xq[:2].astype(np.float32))
    assert np.max(np.abs(approx - xb @ xq[:2].T)) < 5e-3  # rows 0..4095 were re-converted with the centre


def test_overflow_is_retried_with_the_gentle_schedule(fa, monkeypatch):
    """A forced tiny candidate buffer overflows on the first attempt; the overflowed queries are re-answered by the
    filter path with the gentle level schedule (n_retry), not by the exact fp32 scan."""
    rng = np.random.default_rng(34)
    xb, xq = unit_rows(rng, 400_000, 64), unit_rows(rng, 5, 64)
    ix = build(fa, xb)
    monkeypatch.setenv("KIRAG_LEVEL_GROWTH", "32")
    monkeypatch.setenv("KIRAG_LEVEL1_GROWTH", "32")
    monkeypatch.setenv("KIRAG_CAND_CAP", "1024")  # k' = 128: survivors of a 32x level ~ 4096 > 1024
    D, I, st = ix.search_ex(xq, 32, path=AUTO)
    assert st["n_overflow"] >= 1 and st["n_retry"] >= 1, st
    assert_topk_parity(D, I, xb, xq, 32, what=f"retry {st}")


def test_growth_without_virtual_memory_api_still_works(fa, monkeypatch):
    """KIRAG_NO_VMM=1: the cudaMalloc + copy growth path (one buffer at a time) gives the same index."""
    rng = np.random.default_rng(41)
    xb, xq = unit_rows(rng, 30000, 128), unit_rows(rng, 5, 128)
    ref = build(fa, xb)
    D0, I0, _ = ref.search_ex(xq, 10)
    # the switch is read once per process: exercise it in a child process
    import subprocess
    import sys

    code = (
        "import numpy as np, sys\n"
        "sys.path.insert(0, %r)\n"
        "from kirag_b200 import faiss_api\n"
        "rng = np.random.default_rng(41)\n"
        "x = rng.standard_normal((30000, 128)).astype(np.float32); x /= np.linalg.norm(x, axis=1, keepdims=True)\n"
        "q = rng.standard_normal((5, 128)).astype(np.float32); q /= np.linalg.norm(q, axis=1, keepdims=True)\n"
        "ix = faiss_api.IndexFlatIP(128)\n"
        "for a in range(0, 30000, 7000): ix.add(x[a:a + 7000].astype(np.float32))\n"
        "D, I, st = ix.search_ex(q.astype(np.float32), 10)\n"
        "np.save(sys.argv[1], I)\n"
    ) % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import tempfile

    with tempfile.TemporaryDirectory() as td:
        out = os.path.join(td, "I.npy")
        env = dict(os.environ, KIRAG_NO_VMM="1")
        proc = subprocess.run([sys.executable, "-c", code, out], env=env, capture_output=True, text=True, timeout=300)
        assert proc.returncode == 0, proc.stderr[-2000:]
        assert np.array_equal(np.load(out), I0)


# ------------------------------------------------------------ streamed 256-query tiles ---
def test_streamed_pair_kernel_full_search(fa):
    rng = np.random.default_rng(52)
    xb, xq = unit_rows(rng, 90000, 256), unit_rows(rng, 700, 256)
    ix = build(fa, xb)
    D, I, st = ix.search_ex(xq, 20, path=AUTO)
    assert st["n_fast"] >= 690 and st["n_overflow"] == 0, st
    De, Ie, _ = ix.search_ex(xq[:64], 20, path=EXACT)
    assert np.array_equal(I[:64], Ie) and np.array_equal(D[:64], De)
    xi, qi = int_corpus(rng, 30000, 128), int_corpus(rng, 300, 128)
    D, I, st = build(fa, xi).search_ex(qi, 10, path=AUTO)
    Do, Io = oracle.flat_ip_search_blas(xi, qi, 10, use_torch=True)
    assert np.array_equal(I, Io) and np.array_equal(D, Do)
