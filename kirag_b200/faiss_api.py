"""The part of the `faiss` Python surface that KiRAG touches, on the B200 library.

Reference call sites (all in /root/reference/retriever/index.py):
    faiss.IndexFlatIP(d)            :13, :23      -> IndexFlatIP
    faiss.IndexFlatL2               :14           -> exists, raises on construction
    faiss.IndexPQ, METRIC_INNER_PRODUCT :21       -> exist, IndexPQ raises on construction
    index.is_trained / index.train  :30-31        -> True / no-op
    index.add(x)                    :32           -> kirag_index_add
    index.remove_ids(x)             (no call site) -> kirag_index_remove_ids / kirag_index_remove_range
    index.search(x, k)              :47           -> kirag_index_search
    index.range_search(x, radius)   (no call site) -> kirag_index_range_search + kirag_index_range_fetch
    faiss.write_index(index, path)  :62           -> kirag_index_save   ("IxFI" container, "IxMp" for an IndexIDMap)
    faiss.read_index(path, flags)   :73           -> kirag_index_load   (IndexFlatIP, or IndexIDMap for an IxMp file)
    index.ntotal                    :74, :79      -> kirag_index_ntotal

FAISS's way of attaching the caller's ids to a flat index (no reference call site; the reference keeps its own
row -> passage table, retriever/index.py:24,82):
    faiss.IndexIDMap(faiss.IndexFlatIP(d))           -> IndexIDMap: the handle is recreated with KIRAG_INDEX_ID_MAP
    index.add_with_ids(x, ids)                       -> kirag_index_add_with_ids (int64 ids into the device id table)
    index.search / range_search                      -> the ids of the table, mapped by the kernels that write I
    index.remove_ids(x)                              -> selects by id value; nothing else shifts
    faiss.vector_to_array(index.id_map)              -> kirag_index_id_map

Error behaviour follows FAISS's SWIG wrapper: shape / k problems are
AssertionError, library failures are RuntimeError.  There is no CPU path.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
IO_FLAG_READ_ONLY = 2
IO_FLAG_SKIP_IVF_DATA = 8
IO_FLAG_MMAP = IO_FLAG_SKIP_IVF_DATA | 0x646F0000


def _ptr(a: np.ndarray) -> ctypes.c_void_p:
    return ctypes.c_void_p(a.ctypes.data)


def _master_flags(master: Optional[str]) -> int:
    """Index flags for where the fp32 master lives: "device" (HBM, the default) or "host" (pinned host memory mapped
    into the device; only the bf16 shadow takes HBM).  None reads KIRAG_MASTER, "device" when it is unset."""
    if master is None:
        master = os.environ.get("KIRAG_MASTER") or "device"
    assert master in ("device", "host"), f"master must be 'device' or 'host', got {master!r}"
    return _lib.INDEX_HOST_MASTER if master == "host" else 0


def _resolve_devices(device: Optional[int], devices) -> Optional[List[int]]:
    """The device list of a multi-device index, or None for a single-device one.  devices=None reads KIRAG_DEVICES
    (comma-separated device ids, e.g. "0,1,2,3") when no device is given either; unset means a single-device index."""
    if devices is None and device is None:
        env = os.environ.get("KIRAG_DEVICES")
        if env is not None:
            try:
                devices = [int(v) for v in env.split(",")]
            except ValueError:
                raise AssertionError(f"KIRAG_DEVICES must be comma-separated device ids, got {env!r}") from None
    if devices is None:
        return None
    assert device is None, "give either device or devices, not both"
    devices = [int(v) for v in devices]
    assert len(devices) >= 1, "devices must name at least one device"
    assert all(v >= 0 for v in devices), f"device ids must be non-negative, got {devices}"
    return devices


class IDSelectorRange:
    """faiss.IDSelectorRange: selects the ids imin <= id < imax."""

    def __init__(self, imin: int, imax: int):
        self.imin = int(imin)
        self.imax = int(imax)


class IDSelectorBatch:
    """faiss.IDSelectorBatch: selects the ids of an integer array (converted and flattened like remove_ids does)."""

    def __init__(self, ids):
        self.ids = _id_array(ids)


def _id_array(x) -> np.ndarray:
    """An integer array-like as FAISS converts it: np.ascontiguousarray(x, dtype=np.int64), flattened."""
    a = np.asarray(x)
    assert a.size == 0 or a.dtype.kind in "iu", f"expected an integer array or an IDSelector, got {type(x).__name__}"
    return np.ascontiguousarray(a, dtype=np.int64).ravel()


def _id_pairs(x, ids, d: int) -> Tuple[np.ndarray, np.ndarray]:
    """(x, ids) as FAISS's add_with_ids converts them: float32 [n, d] and int64 of shape (n,)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    assert x.ndim == 2, "add_with_ids expects a 2-D array"
    assert x.shape[1] == d, f"add_with_ids: vectors have dimension {x.shape[1]}, index has {d}"
    ids = np.ascontiguousarray(ids, dtype=np.int64)
    assert ids.shape == (x.shape[0],), "not same nb of vectors as ids"
    return x, ids


class IndexFlatIP:
    """Exact inner-product index; corpus lives in HBM (fp32 master + bf16 shadow).  master="host" keeps the fp32 master
    in pinned host memory instead (only the shadow in HBM), with bit-identical results.  devices=[...] stripes the rows
    over several GPUs (repeats allowed), searched at once and merged on devices[0]; results are bit-identical to a
    single-device index with the same rows."""

    metric_type = METRIC_INNER_PRODUCT
    is_trained = True

    def __init__(self, d: int, device: Optional[int] = None, master: Optional[str] = None,
                 devices: Optional[Sequence[int]] = None, _handle: Optional[int] = None):
        self._h = None
        self._pending = None
        self.last_stats: dict = {}
        self._flags = _master_flags(master)
        self._devices = _resolve_devices(device, devices)
        self._lib = _lib.load()
        if self._devices is not None:
            device = self._devices[0]
        self.device = _lib.default_device() if device is None else int(device)
        if _handle is not None:
            self._h = ctypes.c_void_p(_handle)
            self.d = int(self._lib.kirag_index_dim(self._h))
            return
        d = int(d)
        assert d > 0, "dimension must be positive"
        self.d = d
        self._h = self._create()

    def _create(self) -> ctypes.c_void_p:
        h = ctypes.c_void_p()
        if self._devices is None:
            rc = self._lib.kirag_index_create_ex(self.d, METRIC_INNER_PRODUCT, self.device, self._flags, ctypes.byref(h))
        else:
            devs = (ctypes.c_int * len(self._devices))(*self._devices)
            rc = self._lib.kirag_index_create_multi(self.d, METRIC_INNER_PRODUCT, devs, len(self._devices), self._flags,
                                                    ctypes.byref(h))
        _lib.check(rc, "IndexFlatIP")
        return h

    @property
    def devices(self) -> List[int]:
        """The devices of the shards, home device first ([device] for a single-device index)."""
        return list(self._devices) if self._devices is not None else [self.device]

    def _single_device(self, what: str) -> None:
        if self._devices is not None:
            raise RuntimeError(f"{what} is not supported on a multi-device index (no CUDA graph or asynchronous search "
                               "across devices)")

    @property
    def master(self) -> str:
        """Where the fp32 master lives: "device" or "host"."""
        return "host" if self._flags & _lib.INDEX_HOST_MASTER else "device"

    def storage_bytes(self) -> dict:
        """Corpus storage (fp32 master + bf16 shadow, no workspaces) now held: {"device": HBM bytes, "host": pinned
        host bytes}."""
        dev, host = ctypes.c_int64(0), ctypes.c_int64(0)
        _lib.check(self._lib.kirag_index_storage_bytes(self._h, ctypes.byref(dev), ctypes.byref(host)), "storage_bytes")
        return {"device": int(dev.value), "host": int(host.value)}

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

    def add_with_ids(self, x, ids) -> None:
        """Raises as FAISS's IndexFlat does: a flat index has no ids of its own (wrap it in IndexIDMap)."""
        x, ids = _id_pairs(x, ids, self.d)
        _lib.check(self._lib.kirag_index_add_with_ids(self._h, _ptr(x), _ptr(ids), x.shape[0], 0, None), "add_with_ids")

    def remove_ids(self, x) -> int:
        """faiss IndexFlatIP.remove_ids: removes every row whose id is selected by x (an integer array, an
        IDSelectorBatch or an IDSelectorRange); the remaining rows move down in order, so later ids shift.  Ids < 0 or
        >= ntotal select nothing, a repeated id counts once.  Returns the number of rows removed."""
        n = ctypes.c_int64(0)
        if isinstance(x, IDSelectorRange):
            _lib.check(self._lib.kirag_index_remove_range(self._h, x.imin, x.imax, ctypes.byref(n), None), "remove_ids")
        else:
            ids = x.ids if isinstance(x, IDSelectorBatch) else _id_array(x)
            _lib.check(self._lib.kirag_index_remove_ids(self._h, _ptr(ids), ids.size, ctypes.byref(n), None),
                       "remove_ids")
        return int(n.value)

    def remove_ids_device(self, ids) -> int:
        """remove_ids with the ids in an integer CUDA tensor on this index's (home) device, read on the current
        stream.  Selects by position on a plain index, by id value on an id map."""
        import torch

        assert ids.is_cuda and ids.device.index == self.device, \
            f"remove_ids_device: expected a CUDA tensor on cuda:{self.device}"
        assert not ids.dtype.is_floating_point and ids.dtype != torch.bool, "remove_ids_device: integer ids only"
        ids = ids.reshape(-1).to(torch.int64).contiguous()
        n = ctypes.c_int64(0)
        st = torch.cuda.current_stream(ids.device).cuda_stream
        _lib.check(self._lib.kirag_index_remove_ids_ex(self._h, ctypes.c_void_p(ids.data_ptr()), ids.numel(), 1,
                                                       ctypes.byref(n), ctypes.c_void_p(st)), "remove_ids_device")
        return int(n.value)

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
        self._h = self._create()

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

        self._single_device("search_device_async")
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
        self._single_device("pending_flags_ptr")
        p = ctypes.c_void_p()
        _lib.check(self._lib.kirag_index_search_flags(self._h, ctypes.byref(p)), "search_flags")
        return int(p.value or 0)

    def finish(self) -> int:
        """Second half of search_device_async: verifies the certificates, re-answers flagged queries in place.
        Returns the number of queries whose rows of (D, I) were rewritten."""
        self._single_device("finish")
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
        self._single_device("state_token")
        tok = ctypes.c_uint64(0)
        _lib.check(self._lib.kirag_index_state_token(self._h, ctypes.byref(tok)), "state_token")
        return int(tok.value)

    def capture_search(self, nq: int, k: int, id_offset: int = 0, tail=None):
        """Capture kirag_index_search_async for a fixed (nq, k) into a CUDA graph.  `tail(D, I)` (optional) is called
        inside the capture with the search's output tensors and may enqueue more work on the capture stream (the
        multi-GPU exchange); what it returns is kept in the result.  Returns a dict with the static buffers
        (`q` to fill, `D`/`I` results), the graph, its stream and the state token."""
        import torch

        self._single_device("capture_search")
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
        self._single_device("replay_search")
        cap["graph"].replay()
        _lib.check(self._lib.kirag_index_search_rearm(self._h, ctypes.c_void_p(cap["stream"].cuda_stream)), "search_rearm")
        self._pending = (cap["q"], cap["D"], cap["I"])

    def search_device_graph(self, q, k: int, id_offset: int = 0):
        """search_device for small batches through a cached CUDA graph per (nq, k): one graph launch instead of a
        dozen kernel launches.  The returned tensors are the graph's static output buffers: they are overwritten by the
        next call with the same (nq, k)."""
        import torch

        self._single_device("search_device_graph")
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
        self._single_device("debug_scores")
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


class IndexIDMap:
    """faiss.IndexIDMap over an IndexFlatIP: every row carries an int64 id of the caller's (any value, negative and
    repeated ones included), kept in a table on the device.  search / range_search return those ids (order as the
    plain index: score desc, then insertion order), remove_ids selects by id value and nothing else shifts,
    write_index writes FAISS's IxMp file.  The sub-index must be empty; its handle is recreated with the id table
    (device, devices and master kept) and shared with this object, which keeps it as `.index` (rows stay reachable
    by position through index.reconstruct_n; searches through either object return the ids)."""

    def __init__(self, index: IndexFlatIP, _loaded: bool = False):
        assert isinstance(index, IndexFlatIP), "IndexIDMap: the sub-index must be a kirag_b200 IndexFlatIP"
        if not _loaded:
            if index.ntotal != 0:
                raise RuntimeError("IndexIDMap: index must be empty on input")
            index._flags |= _lib.INDEX_ID_MAP
            index.reset()
        self.index = index

    metric_type = METRIC_INNER_PRODUCT
    is_trained = True

    @property
    def d(self) -> int:
        return self.index.d

    @property
    def ntotal(self) -> int:
        return self.index.ntotal

    @property
    def device(self) -> int:
        return self.index.device

    @property
    def devices(self) -> List[int]:
        return self.index.devices

    @property
    def last_stats(self) -> dict:
        return self.index.last_stats

    def train(self, x) -> None:
        return None

    def add(self, x) -> None:
        raise RuntimeError("add does not work on IndexIDMap, use add_with_ids")

    def add_with_ids(self, x, ids) -> None:
        x, ids = _id_pairs(x, ids, self.d)
        if x.shape[0]:
            _lib.check(self.index._lib.kirag_index_add_with_ids(self.index._h, _ptr(x), _ptr(ids), x.shape[0], 0, None),
                       "add_with_ids")

    def search(self, x, k: int) -> Tuple[np.ndarray, np.ndarray]:
        return self.index.search(x, k)

    def search_ex(self, x, k: int, path: int = _lib.PATH_AUTO):
        return self.index.search_ex(x, k, path=path)

    def range_search(self, x, radius: float) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        return self.index.range_search(x, radius)

    def remove_ids(self, x) -> int:
        """Removes every row whose id is selected by x (an integer array or IDSelectorBatch: membership;
        IDSelectorRange(imin, imax): imin <= id < imax), every row of a repeated id included.  Returns the rows
        removed."""
        return self.index.remove_ids(x)

    def reset(self) -> None:
        self.index.reset()

    def reconstruct(self, key: int):
        raise RuntimeError("reconstruct not implemented for this type of index (IndexIDMap has no reverse map; use "
                           "IndexIDMap.index.reconstruct_n for rows by position)")

    @property
    def id_map(self) -> np.ndarray:
        """The ids in row order (int64)."""
        n = self.ntotal
        out = np.empty(n, dtype=np.int64)
        if n:
            _lib.check(self.index._lib.kirag_index_id_map(self.index._h, 0, n, _ptr(out), 0, None), "id_map")
        return out

    def storage_bytes(self) -> dict:
        return self.index.storage_bytes()

    # -- device-resident entry points (as on IndexFlatIP) ---------------------------------------------------------
    def add_with_ids_device(self, x, ids) -> None:
        """x: float32 CUDA tensor [n, d], ids: integer CUDA tensor [n], both on this index's (home) device."""
        import torch

        assert str(x.dtype) == "torch.float32", "add_with_ids_device: float32 only (faiss add() semantics)"
        x = self.index._own_tensor(x, "add_with_ids_device")
        assert ids.is_cuda and ids.device == x.device, "add_with_ids_device: ids must be a CUDA tensor on the index's device"
        ids = ids.to(torch.int64).contiguous()
        assert tuple(ids.shape) == (x.shape[0],), "not same nb of vectors as ids"
        st = torch.cuda.current_stream(x.device).cuda_stream
        _lib.check(self.index._lib.kirag_index_add_with_ids(self.index._h, ctypes.c_void_p(x.data_ptr()),
                                                            ctypes.c_void_p(ids.data_ptr()), x.shape[0], 1,
                                                            ctypes.c_void_p(st)), "add_with_ids_device")

    def search_device(self, q, k: int, path: int = _lib.PATH_AUTO):
        return self.index.search_device(q, k, path=path)

    def range_search_device(self, q, radius: float, path: int = _lib.PATH_AUTO):
        return self.index.range_search_device(q, radius, path=path)

    def remove_ids_device(self, ids) -> int:
        return self.index.remove_ids_device(ids)

    def search_device_async(self, q, k: int):
        return self.index.search_device_async(q, k)

    def finish(self) -> int:
        return self.index.finish()

    def search_device_graph(self, q, k: int):
        return self.index.search_device_graph(q, k)

    def state_token(self) -> int:
        return self.index.state_token()


def vector_to_array(v) -> np.ndarray:
    """faiss.vector_to_array: a copy of the vector as a numpy array (IndexIDMap.id_map already is one)."""
    return np.array(v, copy=True)


class IndexFlatL2:
    """Present because retriever/index.py:14 names it at import time; never constructed by KiRAG."""

    def __init__(self, *a, **kw):
        raise NotImplementedError("kirag_b200 implements the inner-product flat index only (IndexFlatL2 is unused "
                                  "by KiRAG: retrieve.py:112, faiss_index_corpus.py:29 pass 'inner_product')")


class IndexPQ:
    """Present because retriever/index.py:21 names it; only reached with n_subquantizers > 0 (no caller)."""

    def __init__(self, *a, **kw):
        raise NotImplementedError("kirag_b200 implements the exact flat index only (IndexPQ is unused by KiRAG)")


def write_index(index, path) -> None:
    if isinstance(index, IndexIDMap):
        index = index.index
    assert isinstance(index, IndexFlatIP), "write_index: not a kirag_b200 IndexFlatIP or IndexIDMap"
    _lib.check(index._lib.kirag_index_save(index._h, os.fspath(path).encode()), "write_index")


def read_index(path, flags: int = 0, device: Optional[int] = None, master: Optional[str] = None,
               devices: Optional[Sequence[int]] = None):
    """`flags` are FAISS IO flags (IO_FLAG_MMAP is accepted and ignored); `master` and `devices` as for IndexFlatIP.
    An IxFI file gives an IndexFlatIP, an IxMp file an IndexIDMap over one."""
    index_flags = _master_flags(master)
    devs = _resolve_devices(device, devices)
    lib = _lib.load()
    h = ctypes.c_void_p()
    if devs is None:
        dev = _lib.default_device() if device is None else int(device)
        _lib.check(lib.kirag_index_load_ex(os.fspath(path).encode(), dev, index_flags, ctypes.byref(h)), "read_index")
        ix = IndexFlatIP(0, device=dev, master="host" if index_flags else "device", _handle=h.value)
    else:
        arr = (ctypes.c_int * len(devs))(*devs)
        _lib.check(lib.kirag_index_load_multi(os.fspath(path).encode(), arr, len(devs), index_flags, ctypes.byref(h)),
                   "read_index")
        ix = IndexFlatIP(0, master="host" if index_flags else "device", devices=devs, _handle=h.value)
    if lib.kirag_index_flags(ix._h) & _lib.INDEX_ID_MAP:
        ix._flags |= _lib.INDEX_ID_MAP  # reset() keeps the table
        return IndexIDMap(ix, _loaded=True)
    return ix


def omp_get_max_threads() -> int:
    return 1


def get_num_gpus() -> int:
    return int(_lib.load().kirag_device_count())
