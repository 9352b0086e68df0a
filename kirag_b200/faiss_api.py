"""The part of the `faiss` Python surface that KiRAG touches, on the B200 library.

Reference call sites (all in /root/reference/retriever/index.py):
    faiss.IndexFlatIP(d)            :13, :23      -> IndexFlatIP
    faiss.IndexFlatL2               :14           -> exists, raises on construction
    faiss.IndexPQ, METRIC_INNER_PRODUCT :21       -> exist, IndexPQ raises on construction
    index.is_trained / index.train  :30-31        -> True / no-op
    index.add(x)                    :32           -> kirag_index_add
    index.search(x, k)              :47           -> kirag_index_search
    index.range_search(x, radius)   (no call site) -> kirag_index_range_search + kirag_index_range_fetch
    faiss.write_index(index, path)  :62           -> kirag_index_save   ("IxFI" container)
    faiss.read_index(path, flags)   :73           -> kirag_index_load
    index.ntotal                    :74, :79      -> kirag_index_ntotal

Error behaviour follows FAISS's SWIG wrapper: shape / k problems are
AssertionError, library failures are RuntimeError.  There is no CPU path.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Tuple

import numpy as np

from . import _lib

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
IO_FLAG_READ_ONLY = 2
IO_FLAG_SKIP_IVF_DATA = 8
IO_FLAG_MMAP = IO_FLAG_SKIP_IVF_DATA | 0x646F0000


def _ptr(a: np.ndarray) -> ctypes.c_void_p:
    return ctypes.c_void_p(a.ctypes.data)


class IndexFlatIP:
    """Exact inner-product index; corpus lives in HBM (fp32 master + bf16 shadow)."""

    metric_type = METRIC_INNER_PRODUCT
    is_trained = True

    def __init__(self, d: int, device: Optional[int] = None, _handle: Optional[int] = None):
        self._h = None
        self._pending = None
        self.last_stats: dict = {}
        self._lib = _lib.load()
        if _handle is not None:
            self._h = ctypes.c_void_p(_handle)
            self.d = int(self._lib.kirag_index_dim(self._h))
            self.device = _lib.default_device() if device is None else int(device)
            return
        d = int(d)
        assert d > 0, "dimension must be positive"
        self.d = d
        self.device = _lib.default_device() if device is None else int(device)
        h = ctypes.c_void_p()
        _lib.check(self._lib.kirag_index_create(d, METRIC_INNER_PRODUCT, self.device, ctypes.byref(h)),
                   "IndexFlatIP")
        self._h = h

    # -- faiss surface -----------------------------------------------------
    @property
    def ntotal(self) -> int:
        return int(self._lib.kirag_index_ntotal(self._h))

    def train(self, x) -> None:  # flat index: nothing to train (index.py:30-31 never reaches it)
        return None

    def reserve(self, n_total: int) -> None:
        _lib.check(self._lib.kirag_index_reserve(self._h, int(n_total)), "reserve")

    def add(self, x) -> None:
        x = np.ascontiguousarray(x, dtype=np.float32)
        assert x.ndim == 2, "add expects a 2-D array"
        n, d = x.shape
        assert d == self.d, f"add: vectors have dimension {d}, index has {self.d}"
        if n == 0:
            return
        _lib.check(self._lib.kirag_index_add(self._h, _ptr(x), n, 0, None), "add")

    def search(self, x, k: int) -> Tuple[np.ndarray, np.ndarray]:
        x = np.ascontiguousarray(x, dtype=np.float32)
        assert x.ndim == 2, "search expects a 2-D array"
        n, d = x.shape
        assert d == self.d, f"search: queries have dimension {d}, index has {self.d}"
        k = int(k)
        assert k > 0, "k must be positive"
        D = np.empty((n, k), dtype=np.float32)
        I = np.empty((n, k), dtype=np.int64)
        if n == 0:
            return D, I
        stats = _lib.SearchStats()
        path = int(os.environ.get("KIRAG_PATH", _lib.PATH_AUTO))
        _lib.check(
            self._lib.kirag_index_search_ex(self._h, _ptr(x), n, k, _ptr(D), _ptr(I), 0, 0, path,
                                            ctypes.byref(stats), None),
            "search",
        )
        self.last_stats = stats.as_dict()
        return D, I

    def search_ex(self, x, k: int, path: int = _lib.PATH_AUTO, id_offset: int = 0):
        """search() with an explicit path selector; returns (D, I, stats dict)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        assert x.ndim == 2 and x.shape[1] == self.d
        k = int(k)
        assert k > 0, "k must be positive"
        n = x.shape[0]
        D = np.empty((n, k), dtype=np.float32)
        I = np.empty((n, k), dtype=np.int64)
        stats = _lib.SearchStats()
        if n:
            _lib.check(
                self._lib.kirag_index_search_ex(self._h, _ptr(x), n, k, _ptr(D), _ptr(I), 0, int(id_offset),
                                                int(path), ctypes.byref(stats), None),
                "search_ex",
            )
        self.last_stats = stats.as_dict()
        return D, I, self.last_stats

    def range_search(self, x, radius: float) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """faiss IndexFlatIP.range_search: every row with score > radius.  Returns (lims int64 [n+1], D float32,
        I int64); query i owns D/I[lims[i]:lims[i+1]], ordered by (score desc, id asc).  Honours KIRAG_PATH."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        assert x.ndim == 2, "range_search expects a 2-D array"
        n, d = x.shape
        assert d == self.d, f"range_search: queries have dimension {d}, index has {self.d}"
        path = int(os.environ.get("KIRAG_PATH", _lib.PATH_AUTO))
        lims = np.zeros(n + 1, dtype=np.int64)
        stats = _lib.SearchStats()
        _lib.check(self._lib.kirag_index_range_search(self._h, _ptr(x), n, float(radius), 0, 0, path, _ptr(lims),
                                                      ctypes.byref(stats), None), "range_search")
        total = int(lims[n])
        D = np.empty(total, dtype=np.float32)
        I = np.empty(total, dtype=np.int64)
        _lib.check(self._lib.kirag_index_range_fetch(self._h, _ptr(D), _ptr(I), 0, None), "range_search")
        self.last_stats = stats.as_dict()
        return lims, D, I

    def reconstruct_n(self, i0: int = 0, n: int = -1) -> np.ndarray:
        if n < 0:
            n = self.ntotal - i0
        out = np.empty((n, self.d), dtype=np.float32)
        if n:
            _lib.check(self._lib.kirag_index_reconstruct(self._h, int(i0), int(n), _ptr(out), 0, None),
                       "reconstruct_n")
        return out

    def reconstruct(self, i: int) -> np.ndarray:
        return self.reconstruct_n(int(i), 1)[0]

    def reset(self) -> None:
        self._destroy()
        h = ctypes.c_void_p()
        _lib.check(self._lib.kirag_index_create(self.d, METRIC_INNER_PRODUCT, self.device, ctypes.byref(h)), "reset")
        self._h = h

    # -- device-resident entry points (additions, not part of faiss) --------
    def _own_tensor(self, t, what: str):
        """A contiguous float32 tensor ON THIS INDEX'S DEVICE with a 16-byte aligned base (the kernels use
        float4 loads); a tensor of another GPU is rejected instead of being handed to the kernels as a raw pointer."""
        import torch

        assert t.is_cuda and t.dim() == 2 and t.shape[1] == self.d, f"{what}: expected a CUDA tensor [n, {self.d}]"
        assert t.device.index == self.device, \
            f"{what}: tensor is on cuda:{t.device.index}, the index lives on cuda:{self.device}"
        t = t.contiguous()
        if t.dtype != torch.float32:
            t = t.float()
        if t.data_ptr() % 16:
            t = t.clone()
        return t

    def add_device(self, x) -> None:
        """x: float32 CUDA torch tensor [n, d] on this index's device."""
        import torch

        assert str(x.dtype) == "torch.float32", "add_device: float32 only (faiss add() semantics)"
        x = self._own_tensor(x, "add_device")
        st = torch.cuda.current_stream(x.device).cuda_stream
        _lib.check(self._lib.kirag_index_add(self._h, ctypes.c_void_p(x.data_ptr()), x.shape[0], 1,
                                             ctypes.c_void_p(st)), "add_device")

    def search_device(self, q, k: int, id_offset: int = 0, path: int = _lib.PATH_AUTO):
        """q: float32 CUDA tensor [n, d]; returns CUDA tensors (D [n,k] f32, I [n,k] i64).  The work is enqueued
        on the current stream; the call synchronises once to read the certificate flags (see the header)."""
        import torch

        q = self._own_tensor(q, "search_device")
        k = int(k)
        assert k > 0, "k must be positive"
        n = q.shape[0]
        D = torch.empty((n, k), dtype=torch.float32, device=q.device)
        I = torch.empty((n, k), dtype=torch.int64, device=q.device)
        stats = _lib.SearchStats()
        if n:
            st = torch.cuda.current_stream(q.device).cuda_stream
            _lib.check(
                self._lib.kirag_index_search_ex(self._h, ctypes.c_void_p(q.data_ptr()), n, k,
                                                ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()), 1,
                                                int(id_offset), int(path), ctypes.byref(stats), ctypes.c_void_p(st)),
                "search_device",
            )
        self.last_stats = stats.as_dict()
        return D, I

    def range_search_device(self, q, radius: float, id_offset: int = 0, path: int = _lib.PATH_AUTO):
        """range_search on a float32 CUDA tensor [n, d]; returns CUDA tensors (lims int64 [n+1], D f32, I i64).  The
        call is synchronous: the result size is only known once the survivors have been counted."""
        import torch

        q = self._own_tensor(q, "range_search_device")
        n = q.shape[0]
        lims = np.zeros(n + 1, dtype=np.int64)
        stats = _lib.SearchStats()
        st = ctypes.c_void_p(torch.cuda.current_stream(q.device).cuda_stream)
        _lib.check(self._lib.kirag_index_range_search(self._h, ctypes.c_void_p(q.data_ptr()), n, float(radius), 1,
                                                      int(id_offset), int(path), _ptr(lims), ctypes.byref(stats), st),
                   "range_search_device")
        total = int(lims[n])
        D = torch.empty(total, dtype=torch.float32, device=q.device)
        I = torch.empty(total, dtype=torch.int64, device=q.device)
        _lib.check(self._lib.kirag_index_range_fetch(self._h, ctypes.c_void_p(D.data_ptr()),
                                                     ctypes.c_void_p(I.data_ptr()), 1, st), "range_search_device")
        self.last_stats = stats.as_dict()
        return torch.from_numpy(lims).to(q.device), D, I

    def search_device_async(self, q, k: int, id_offset: int = 0):
        """Stream-ordered first half of search_device (kirag_index_search_async): no host synchronisation, CUDA-graph
        capturable once the workspaces are warm.  Returns (D, I); they are final for every query whose certificate
        passed.  Call finish() (after whatever else was enqueued behind it) to complete the search."""
        import torch

        q = self._own_tensor(q, "search_device_async")
        k = int(k)
        assert k > 0, "k must be positive"
        n = q.shape[0]
        D = torch.empty((n, k), dtype=torch.float32, device=q.device)
        I = torch.empty((n, k), dtype=torch.int64, device=q.device)
        if n:
            st = torch.cuda.current_stream(q.device).cuda_stream
            _lib.check(
                self._lib.kirag_index_search_async(self._h, ctypes.c_void_p(q.data_ptr()), n, k,
                                                   ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()),
                                                   int(id_offset), ctypes.c_void_p(st)),
                "search_device_async",
            )
        self._pending = (q, D, I)  # the library keeps raw pointers until finish()
        return D, I

    def pending_flags_ptr(self) -> int:
        """Device address of the pending search's per-query certificate flags (0 if there is nothing to verify)."""
        p = ctypes.c_void_p()
        _lib.check(self._lib.kirag_index_search_flags(self._h, ctypes.byref(p)), "search_flags")
        return int(p.value or 0)

    def finish(self) -> int:
        """Second half of search_device_async: verifies the certificates, re-answers flagged queries in place.
        Returns the number of queries whose rows of (D, I) were rewritten."""
        stats = _lib.SearchStats()
        changed = ctypes.c_int64(0)
        _lib.check(self._lib.kirag_index_search_finish(self._h, ctypes.byref(stats), ctypes.byref(changed)), "finish")
        self.last_stats = stats.as_dict()
        self._pending = None
        return int(changed.value)

    # -- CUDA-graph replay of the asynchronous search (small query batches: launches are what a call costs) -----
    def state_token(self) -> int:
        """Changes whenever something a captured search baked into its kernel arguments does (rows added, a workspace
        grown by a larger call): a graph is replayed only while the token is the one read after its capture."""
        tok = ctypes.c_uint64(0)
        _lib.check(self._lib.kirag_index_state_token(self._h, ctypes.byref(tok)), "state_token")
        return int(tok.value)

    def capture_search(self, nq: int, k: int, id_offset: int = 0, tail=None):
        """Capture kirag_index_search_async for a fixed (nq, k) into a CUDA graph.  `tail(D, I)` (optional) is called
        inside the capture with the search's output tensors and may enqueue more work on the capture stream (the
        multi-GPU exchange); what it returns is kept in the result.  Returns a dict with the static buffers
        (`q` to fill, `D`/`I` results), the graph, its stream and the state token."""
        import torch

        dev = torch.device("cuda", self.device)
        q = torch.nn.functional.normalize(torch.randn((nq, self.d), dtype=torch.float32, device=dev), dim=1)
        self.search_device(q, k, id_offset=id_offset)  # warm the workspaces: the capture itself must not allocate
        torch.cuda.synchronize(dev)
        stream = torch.cuda.Stream(device=dev)
        graph = torch.cuda.CUDAGraph()
        extra = None
        # nothing executes during the capture (in particular no cross-GPU rendez-vous of `tail`): ranks of a sharded
        # index may (re)capture independently of each other
        with torch.cuda.stream(stream):
            with torch.cuda.graph(graph, stream=stream):
                D, I = self.search_device_async(q, k, id_offset=id_offset)
                if tail is not None:
                    extra = tail(D, I)
        self.finish()  # the capture left a (never executed) pending search behind
        return {"q": q, "D": D, "I": I, "graph": graph, "stream": stream, "extra": extra, "token": self.state_token(),
                "nq": nq, "k": k, "id_offset": id_offset}

    def replay_search(self, cap) -> None:
        """Launch a captured search on its stream and mark it pending (finish() completes it)."""
        cap["graph"].replay()
        _lib.check(self._lib.kirag_index_search_rearm(self._h, ctypes.c_void_p(cap["stream"].cuda_stream)), "search_rearm")
        self._pending = (cap["q"], cap["D"], cap["I"])

    def search_device_graph(self, q, k: int, id_offset: int = 0):
        """search_device for small batches through a cached CUDA graph per (nq, k): one graph launch instead of a
        dozen kernel launches.  The returned tensors are the graph's static output buffers: they are overwritten by the
        next call with the same (nq, k)."""
        import torch

        q = self._own_tensor(q, "search_device_graph")
        key = (int(q.shape[0]), int(k), int(id_offset))
        cache = self.__dict__.setdefault("_graphs", {})
        cap = cache.get(key)
        if cap is None or cap["token"] != self.state_token():
            cap = cache[key] = self.capture_search(key[0], key[1], id_offset=key[2])
        cur = torch.cuda.current_stream(q.device)
        cap["stream"].wait_stream(cur)
        with torch.cuda.stream(cap["stream"]):
            cap["q"].copy_(q, non_blocking=True)
            self.replay_search(cap)
        self.finish()  # synchronises the graph's stream, verifies the certificates, re-answers flagged queries
        return cap["D"], cap["I"]

    def debug_scores(self, x) -> np.ndarray:
        """Dense approximate (bf16 tcgen05) scores [ntotal, nq] — test hook."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = np.empty((self.ntotal, x.shape[0]), dtype=np.float32)
        _lib.check(self._lib.kirag_index_debug_scores(self._h, _ptr(x), x.shape[0], _ptr(out)), "debug_scores")
        return out

    # -- lifetime -------------------------------------------------------------
    def _destroy(self) -> None:
        h, self._h = self._h, None
        if h is not None and self._lib is not None:
            self._lib.kirag_index_destroy(h)

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass


class IndexFlatL2:
    """Present because retriever/index.py:14 names it at import time; never constructed by KiRAG."""

    def __init__(self, *a, **kw):
        raise NotImplementedError("kirag_b200 implements the inner-product flat index only (IndexFlatL2 is unused "
                                  "by KiRAG: retrieve.py:112, faiss_index_corpus.py:29 pass 'inner_product')")


class IndexPQ:
    """Present because retriever/index.py:21 names it; only reached with n_subquantizers > 0 (no caller)."""

    def __init__(self, *a, **kw):
        raise NotImplementedError("kirag_b200 implements the exact flat index only (IndexPQ is unused by KiRAG)")


def write_index(index: IndexFlatIP, path) -> None:
    assert isinstance(index, IndexFlatIP), "write_index: not a kirag_b200 IndexFlatIP"
    _lib.check(index._lib.kirag_index_save(index._h, os.fspath(path).encode()), "write_index")


def read_index(path, flags: int = 0, device: Optional[int] = None) -> IndexFlatIP:
    lib = _lib.load()
    dev = _lib.default_device() if device is None else int(device)
    h = ctypes.c_void_p()
    _lib.check(lib.kirag_index_load(os.fspath(path).encode(), dev, ctypes.byref(h)), "read_index")
    return IndexFlatIP(0, device=dev, _handle=h.value)


def omp_get_max_threads() -> int:
    return 1


def get_num_gpus() -> int:
    return int(_lib.load().kirag_device_count())
