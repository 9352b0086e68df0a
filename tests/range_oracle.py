"""fp64 numpy restatement of IndexFlatIP.range_search for the range-search tests.

Every row with <q, x> > radius (strict), each query's list ordered by (score desc, id asc), FAISS's layout
(lims [nq+1], D float32, I int64).  On int_corpus data every product and partial sum is an exact small integer, so
the fp64 scores equal the library's canonical fp32 scores and the comparison can be exact.
"""
import numpy as np


def flat_ip_range_search(xb, xq, radius, id_offset=0):
    xb = np.asarray(xb, dtype=np.float32)
    xq = np.asarray(xq, dtype=np.float32)
    nq = xq.shape[0]
    s = xq.astype(np.float64) @ xb.astype(np.float64).T if xb.shape[0] else np.zeros((nq, 0))
    lims = np.zeros(nq + 1, dtype=np.int64)
    Ds, Is = [], []
    for i in range(nq):
        with np.errstate(invalid="ignore"):
            hit = np.nonzero(s[i] > radius)[0]
        order = np.lexsort((hit, -s[i][hit]))
        Ds.append(s[i][hit][order].astype(np.float32))
        Is.append(hit[order].astype(np.int64) + id_offset)
        lims[i + 1] = lims[i] + hit.size
    D = np.concatenate(Ds) if Ds else np.zeros(0, dtype=np.float32)
    I = np.concatenate(Is) if Is else np.zeros(0, dtype=np.int64)
    return lims, D, I
