"""The oracle itself: checked against fp64 brute force, hand-checkable cases and the golden fixtures."""
import os

import numpy as np
import pytest

from oracle import oracle
from tests.helpers import assert_topk_parity, exact_topk_f64, int_corpus, load_search_golden

GOLD = os.path.join(os.path.dirname(__file__), "golden")
LOWEST = np.float32(-3.4028234663852886e38)


def test_hand_checkable_ties_and_padding():
    # 5 rows in 2-D; scores against q=(1,0): 3, 1, 3, 0, 3 -> ties on 3 must come out id-ascending
    xb = np.array([[3, 0], [1, 5], [3, 9], [0, 1], [3, -2]], dtype=np.float32)
    xq = np.array([[1, 0]], dtype=np.float32)
    D, I = oracle.flat_ip_search(xb, xq, 3)
    assert I.tolist() == [[0, 2, 4]] and D.tolist() == [[3, 3, 3]]
    D, I = oracle.flat_ip_search(xb, xq, 2)  # tie straddles rank k: lower ids are kept
    assert I.tolist() == [[0, 2]]
    D, I = oracle.flat_ip_search(xb, xq, 1)
    assert I.tolist() == [[0]]
    D, I = oracle.flat_ip_search(xb, xq, 8)  # k > ntotal: FAISS padding
    assert I.tolist() == [[0, 2, 4, 1, 3, -1, -1, -1]]
    assert np.all(D[0, 5:] == LOWEST)


def test_empty_inputs():
    xb = np.zeros((0, 4), dtype=np.float32)
    D, I = oracle.flat_ip_search(xb, np.ones((2, 4), dtype=np.float32), 3)
    assert np.all(I == -1) and np.all(D == LOWEST)
    D, I = oracle.flat_ip_search(np.ones((3, 4), dtype=np.float32), np.zeros((0, 4), dtype=np.float32), 3)
    assert D.shape == (0, 3) and I.shape == (0, 3)


@pytest.mark.parametrize("n,d,nq,k", [(1000, 64, 5, 10), (300, 128, 3, 100), (50, 32, 4, 64), (4097, 16, 2, 7)])
def test_integer_data_is_exact_in_every_variant(n, d, nq, k):
    rng = np.random.default_rng(n + d)
    xb, xq = int_corpus(rng, n, d), int_corpus(rng, nq, d)
    for D, I in (oracle.flat_ip_search(xb, xq, k, accum="f32"), oracle.flat_ip_search(xb, xq, k, accum="f64"),
                 oracle.flat_ip_search_blas(xb, xq, k, q_block=3, db_block=257),
                 oracle.flat_ip_search_blas(xb, xq, k)):
        assert_topk_parity(D, I, xb, xq, k, exact=True)


@pytest.mark.parametrize("accum", ["f32", "f64"])
def test_random_unit_vectors_against_fp64(accum):
    rng = np.random.default_rng(3)
    xb = rng.standard_normal((5000, 96)).astype(np.float32)
    xb /= np.linalg.norm(xb, axis=1, keepdims=True)
    xq = rng.standard_normal((9, 96)).astype(np.float32)
    D, I = oracle.flat_ip_search(xb, xq, 20, accum=accum)
    assert_topk_parity(D, I, xb, xq, 20)
    Db, Ib = oracle.flat_ip_search_blas(xb, xq, 20, db_block=1024)
    assert_topk_parity(Db, Ib, xb, xq, 20)


def test_nan_and_duplicates():
    rng = np.random.default_rng(9)
    xb = int_corpus(rng, 64, 8)
    xb[10] = np.nan  # a NaN row never enters the heap (thresh < NaN is false)
    xb[20:24] = xb[3]
    xq = int_corpus(rng, 2, 8)
    D, I = oracle.flat_ip_search(xb, xq, 64)
    assert 10 not in I.tolist()[0] and I[0, -1] == -1
    row = I[0].tolist()
    assert row.index(3) < row.index(20) < row.index(21) < row.index(22) < row.index(23)


def test_merge_matches_unsharded():
    rng = np.random.default_rng(5)
    xb, xq = int_corpus(rng, 999, 32), int_corpus(rng, 6, 32)
    k, G = 12, 4
    per = (999 + G - 1) // G
    Ds, Is = [], []
    for g in range(G):
        lo, hi = g * per, min((g + 1) * per, 999)
        D, I = oracle.flat_ip_search(xb[lo:hi], xq, k, id_offset=lo)
        Ds.append(D), Is.append(I)
    D, I = oracle.merge_topk(np.stack(Ds), np.stack(Is))
    D1, I1 = oracle.flat_ip_search(xb, xq, k)
    assert np.array_equal(I, I1) and np.array_equal(D, D1)


def test_search_golden_fixture():
    z = load_search_golden()
    for name in ("unit_64", "unit_1024", "kgtn", "ties"):
        xb, xq, k = z[f"{name}_xb"], z[f"{name}_xq"], int(z[f"{name}_k"])
        D, I = oracle.flat_ip_search(xb, xq, k, accum="f64")
        assert np.array_equal(I, z[f"{name}_I"]) and np.array_equal(D, z[f"{name}_D"])
        assert_topk_parity(D, I, xb, xq, k, exact=(name == "ties"))
        # fp32 accumulation and the blocked path agree up to near-ties
        for D2, I2 in (oracle.flat_ip_search(xb, xq, k), oracle.flat_ip_search_blas(xb, xq, k)):
            assert_topk_parity(D2, I2, xb, xq, k, exact=(name == "ties"))


def test_aligner_golden_pins_oracle_to_reference_torch():
    """torch.matmul + torch.topk (models.py:1532-1538) outputs vs the oracle: same sets, same scores."""
    z = np.load(os.path.join(GOLD, "aligner_golden.npz"))
    for name in ("s", "m", "few"):
        q, t, k = z[f"{name}_q"], z[f"{name}_t"], int(z[f"{name}_k"])
        kk = min(k, t.shape[0])
        D, I = oracle.flat_ip_search(t, q, kk)
        ref_s, ref_i = z[f"{name}_scores"], z[f"{name}_indices"]
        assert D.shape == ref_s.shape
        np.testing.assert_allclose(D, ref_s, rtol=1e-5, atol=1e-6)
        for r in range(q.shape[0]):
            assert set(I[r].tolist()) == set(ref_i[r].tolist())


def test_pool_golden_pins_oracle_to_reference_torch():
    z = np.load(os.path.join(GOLD, "pool_golden.npz"))
    np.testing.assert_allclose(oracle.pool_normalize(z["a_hidden"], z["a_mask"], "mean", False), z["a_avg"], atol=2e-6)
    np.testing.assert_allclose(oracle.pool_normalize(z["a_hidden"], z["a_mask"], "mean", True), z["a_e5"], atol=1e-6)
    np.testing.assert_allclose(oracle.pool_normalize(z["a_hidden"], None, "cls", True), z["a_bge"], atol=1e-6)
    np.testing.assert_allclose(oracle.pool_normalize(z["b_hidden"], z["b_mask"], "mean", True), z["b_e5"], atol=1e-6)
    np.testing.assert_allclose(oracle.pool_normalize(z["c_hidden_f32"], z["c_mask"], "mean", True), z["c_e5_f32ref"],
                               atol=1e-6)
    # bf16 reference run (trainer autocast): within the 1e-3 the north star allows (bf16 has 8 mantissa bits)
    np.testing.assert_allclose(oracle.pool_normalize(z["c_hidden_f32"], z["c_mask"], "mean", True), z["c_e5_bf16ref"],
                               atol=1e-3)
    for name, mode in (("e5", "mean"), ("bge", "cls")):
        got = oracle.pool_normalize(z[f"d_{name}_hidden"], z["d_mask"], mode, True)
        np.testing.assert_allclose(got, z[f"d_{name}_out"], atol=1e-6)


def test_pool_all_zero_mask_row_is_nan_like_the_reference():
    import torch

    h = np.ones((2, 3, 4), dtype=np.float32)
    m = np.array([[1, 1, 0], [0, 0, 0]], dtype=np.int64)
    ref = oracle.pool_normalize_torch(torch.from_numpy(h), torch.from_numpy(m)).numpy()
    got = oracle.pool_normalize(h, m)
    assert np.all(np.isnan(ref[1])) and np.all(np.isnan(got[1]))
    np.testing.assert_allclose(got[0], ref[0], atol=1e-6)


def test_oracle_against_a_real_faiss_wheel_when_one_is_installed():
    """faiss-cpu is not installable in the build image (no wheel, no network), so the search oracle is unpinned
    (DESIGN.md §7).  Should a real wheel ever be importable, this test pins the restatement to it: ids identical
    on tie-free data, scores within fp32 summation-order noise, FAISS's padding for k > ntotal."""
    faiss = pytest.importorskip("faiss")
    if getattr(faiss, "__kirag_b200__", False):
        pytest.skip("sys.modules['faiss'] is the kirag_b200 stand-in, not a real faiss")
    rng = np.random.default_rng(42)
    xb = rng.standard_normal((5000, 64)).astype(np.float32)
    for nq in (3, 40):  # FAISS's n < 20 SIMD path and its blocked-sgemm path
        xq = rng.standard_normal((nq, 64)).astype(np.float32)
        ix = faiss.IndexFlatIP(64)
        ix.add(xb)
        for k in (10, 100):  # heap and reservoir result handlers
            Df, If = ix.search(xq, k)
            Do, Io = oracle.flat_ip_search(xb, xq, k)
            assert np.array_equal(If, Io)
            np.testing.assert_allclose(Df, Do, rtol=1e-5, atol=1e-6)
    small = faiss.IndexFlatIP(64)
    small.add(xb[:3])
    Df, If = small.search(xq[:2], 5)
    Do, Io = oracle.flat_ip_search(xb[:3], xq[:2], 5)
    assert np.array_equal(If, Io) and np.array_equal(Df[:, 3:], Do[:, 3:])
