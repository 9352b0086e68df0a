"""Shared comparison logic for the parity tests."""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# the search fixture is stored in two files to keep each under 1 MB (the 256 x 1024 case alone fills most of one)
SEARCH_GOLDEN_FILES = ("search_golden.npz", "search_golden_1024.npz")


def load_search_golden():
    """Every array of the search fixture, by name, from all its files."""
    z = {}
    for f in SEARCH_GOLDEN_FILES:
        z.update(np.load(os.path.join(GOLD, f)))
    return z


def exact_topk_f64(xb, xq, k):
    """Ground truth in fp64: ids by (score desc, id asc), scores as fp64."""
    s = xq.astype(np.float64) @ xb.astype(np.float64).T
    n = xb.shape[0]
    kk = min(k, n)
    order = np.lexsort((np.broadcast_to(np.arange(n), s.shape), -s), axis=1)[:, :kk]
    return np.take_along_axis(s, order, axis=1), order


def assert_topk_parity(D, I, xb, xq, k, rtol=1e-5, exact=False, what=""):
    """Check a search result against fp64 ground truth.

    * shape, padding: slots beyond ntotal hold (-FLT_MAX, -1)
    * scores: within rtol (relative to |q||x| scale) of the fp64 score of the returned id
    * order: rows sorted by (score desc, id asc) on the RETURNED fp32 scores
    * ids: identical to ground truth, except swaps explained by fp32 near-ties
      (|fp64 score difference| < 4 * rtol * scale); with exact=True no exception is allowed
    Returns the number of near-tie id differences (reported by the caller).
    """
    nq = xq.shape[0]
    n = xb.shape[0]
    assert D.shape == (nq, k) and I.shape == (nq, k), what
    assert D.dtype == np.float32 and I.dtype == np.int64, what
    kk = min(k, n)
    if kk < k:
        assert np.all(I[:, kk:] == -1), what + " padding ids"
        assert np.all(D[:, kk:] == np.float32(-3.4028234663852886e38)), what + " padding scores"
    if kk == 0 or nq == 0:
        return 0
    S_true, I_true = exact_topk_f64(xb, xq, k)
    Ik, Dk = I[:, :kk], D[:, :kk]
    assert np.all((Ik >= 0) & (Ik < n)), what + " id range"
    # no duplicates within a row
    assert all(len(set(r.tolist())) == kk for r in Ik), what + " duplicate ids"
    full = xq.astype(np.float64) @ xb.astype(np.float64).T
    scale = (np.linalg.norm(xq.astype(np.float64), axis=1)[:, None] *
             np.max(np.linalg.norm(xb.astype(np.float64), axis=1)))
    scale = np.maximum(scale, 1e-30)
    got_true_scores = np.take_along_axis(full, Ik, axis=1)
    err = np.abs(Dk.astype(np.float64) - got_true_scores)
    assert np.all(err <= rtol * scale), f"{what} score error {err.max():.3e} (scale {scale.max():.3e})"
    # order on returned scores
    d0, d1 = Dk[:, :-1], Dk[:, 1:]
    i0, i1 = Ik[:, :-1], Ik[:, 1:]
    assert np.all((d0 > d1) | ((d0 == d1) & (i0 < i1))), what + " row order (score desc, id asc)"
    diff = Ik != I_true
    n_diff = int(diff.sum())
    if exact:
        assert n_diff == 0, f"{what}: {n_diff} id mismatches on exactly representable data"
        assert np.array_equal(Dk.astype(np.float64), S_true), what + " scores must be exact"
        return 0
    if n_diff:
        # every id we returned that is not in the true set must be within a near-tie of the k-th true score
        tol = 4 * rtol * scale
        kth = S_true[:, -1:]
        assert np.all(got_true_scores >= kth - tol), f"{what}: returned an id that is not a near-tie of the true top-k"
        # and position-wise the true score sequence must agree within the same tolerance
        assert np.all(np.abs(got_true_scores - S_true) <= tol), what + " id swap not explained by a near-tie"
    return n_diff


def int_corpus(rng, n, d, lo=-3, hi=4):
    """Small-integer vectors: exactly representable in bf16, exact sums in fp32 -> every precision agrees."""
    return rng.integers(lo, hi, size=(n, d)).astype(np.float32)
