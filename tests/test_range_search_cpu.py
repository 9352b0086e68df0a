"""Range search without a GPU: argument validation of the C ABI, and the sharded assembly (world size 2, gloo) with
oracle-backed local indexes in place of the CUDA library."""
import ctypes
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from kirag_b200 import _lib
from tests.helpers import int_corpus
from tests.range_oracle import flat_ip_range_search


def test_range_search_argument_validation():
    lib = _lib.load()
    lims = np.zeros(2, dtype=np.int64)
    q = np.zeros(64, dtype=np.float32)
    assert lib.kirag_index_range_search(None, q.ctypes.data, 1, 0.5, 0, 0, 0, lims.ctypes.data, None, None) != 0
    assert "null index" in _lib.last_error()
    assert lib.kirag_index_range_search(None, q.ctypes.data, -1, 0.5, 0, 0, 0, lims.ctypes.data, None, None) != 0
    assert "negative nq" in _lib.last_error()
    D = np.zeros(1, dtype=np.float32)
    I = np.zeros(1, dtype=np.int64)
    assert lib.kirag_index_range_fetch(None, D.ctypes.data, I.ctypes.data, 0, None) != 0
    assert "null index" in _lib.last_error()


def test_oracle_is_strict_and_ordered():
    xb = np.array([[1, 0], [2, 0], [2, 0], [0, 1], [-1, 0]], dtype=np.float32)
    xq = np.array([[1, 0], [0, 0]], dtype=np.float32)
    lims, D, I = flat_ip_range_search(xb, xq, 1.0, id_offset=10)
    assert lims.tolist() == [0, 2, 2]  # the row scoring exactly 1.0 is absent; the zero query has no hits
    assert I.tolist() == [11, 12] and D.tolist() == [2.0, 2.0]
    assert flat_ip_range_search(xb, xq, float("nan"))[0].tolist() == [0, 0, 0]


class _LocalOracleIndex:
    def __init__(self, d):
        self.d = d
        self.x = np.empty((0, d), dtype=np.float32)

    @property
    def ntotal(self):
        return self.x.shape[0]

    def add(self, x):
        self.x = np.concatenate([self.x, np.asarray(x, dtype=np.float32)])

    def range_search_device(self, q, radius, id_offset=0):
        lims, D, I = flat_ip_range_search(self.x, q.numpy(), radius, id_offset=id_offset)
        return torch.from_numpy(lims), torch.from_numpy(D), torch.from_numpy(I)


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from kirag_b200.sharded import ShardedFlatIP

        rng = np.random.default_rng(5)
        n, d = 301, 16
        xb, xq = int_corpus(rng, n, d), int_corpus(rng, 6, d)
        # rows of the second shard never reach the radius: that rank contributes no hits at all
        xb[151:] = 0.0
        xb[7] = xb[3]  # equal scores: ids ascending
        radius = 4.0
        ok = True
        sh = ShardedFlatIP(d, n, local_index=_LocalOracleIndex(d), merge_fn=lambda *a: None)
        sh.add_shard(xb[sh.lo:sh.hi])
        lims, D, I = sh.range_search(torch.from_numpy(xq), radius)
        lims1, D1, I1 = flat_ip_range_search(xb, xq, radius)
        ok = ok and sh.lo == (151 if rank else 0) and int(lims1[-1]) > 0
        ok = ok and np.array_equal(lims.numpy(), lims1) and np.array_equal(I.numpy(), I1) and np.array_equal(D.numpy(), D1)
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_sharded_range_search_world_size_2():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret[0] and ret[1]
