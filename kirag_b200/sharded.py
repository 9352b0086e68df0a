"""Row-sharded exact search over the GPUs of one node.

No counterpart in the reference (its FAISS search is single-process CPU,
/root/reference/retriever/index.py:47); this is the multi-GPU form
BASELINE.json's north_star asks for.  One process per GPU (torchrun).  Rank g
owns the contiguous global rows [lo_g, hi_g); every rank answers every query
against its shard with GLOBAL ids (local row + lo_g); the k per-shard results
per query are then exchanged and merged into the global top-k by (score desc,
id asc).  Exactness: the global top-k is a subset of the union of the per-shard
top-k.

Two exchanges:
  "peer" (default on CUDA)  ONE kernel per rank (csrc/exchange.cu) stores its rows
         into every rank's exchange buffer over NVLink peer memory (CUDA IPC
         mappings), waits per query range for the peers' rows and merges them;
  "nccl"  one packed all_gather_into_tensor + kirag_merge_topk (the baseline the
         peer kernel replaces; also what the gloo CPU tests drive with the
         oracle plugged in).

The local search and the merge are injectable so that the plumbing (shard
ranges, id offsets, gather layout) is testable with gloo on CPU, where the
tests plug the oracle in; the defaults are the CUDA library and nothing else.
"""
from __future__ import annotations

import ctypes
import os
import warnings
from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib


def shard_range(n_total: int, world_size: int, rank: int, weights=None) -> Tuple[int, int]:
    """Contiguous row range of `rank`.  Default: ceil-sized shards, the last ones may be short/empty.  With
    `weights` (one positive number per rank, the same list on every rank): ranges proportional to the weights,
    boundaries rounded to whole 128-row tiles — a strong-scaling step is paced by its slowest GPU, and the GPUs of
    one box run at different power-capped clocks (measure_rank_weights)."""
    if weights is None:
        per = (n_total + world_size - 1) // world_size
        lo = min(rank * per, n_total)
        hi = min(lo + per, n_total)
        return lo, hi
    assert len(weights) == world_size and all(w > 0 for w in weights), "one positive weight per rank"
    total = float(sum(weights))
    bounds = [0]
    acc = 0.0
    for w in weights[:-1]:
        acc += float(w)
        b = int(round(acc / total * n_total / 128.0)) * 128
        bounds.append(min(max(b, bounds[-1]), n_total))
    bounds.append(n_total)
    return bounds[rank], bounds[rank + 1]


def measure_rank_weights(d: int, device: int, group=None, nq: int = 4096, k: int = 100, rows: int = 1 << 20,
                         seconds: float = 2.0):
    """Relative search speed of every rank's GPU (SPMD: all ranks call it together): each rank builds the same
    small probe index and runs the tensor-bound search for `seconds` at the same time as its peers (the power and
    thermal situation of the real job); returns the list of rates normalised to mean 1 (identical on every rank),
    ready for ShardedFlatIP(..., weights=...)."""
    import time

    from .faiss_api import IndexFlatIP

    dev = torch.device("cuda", device)
    g = torch.Generator(device=dev)
    g.manual_seed(20241)
    ix = IndexFlatIP(d, device=device)
    ix.reserve(rows)
    chunk = 1 << 18
    for r0 in range(0, rows, chunk):
        ix.add_device(torch.nn.functional.normalize(torch.randn(min(chunk, rows - r0), d, generator=g, device=dev), dim=1))
    q = torch.nn.functional.normalize(torch.randn(nq, d, generator=g, device=dev), dim=1)
    for _ in range(3):
        ix.search_device(q, k)
    torch.cuda.synchronize(dev)
    if dist.is_initialized():
        dist.barrier(group=group)
    times = []
    t_end = time.perf_counter() + seconds
    while time.perf_counter() < t_end or len(times) < 5:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ix.search_device(q, k)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    del ix
    torch.cuda.empty_cache()
    tail = sorted(times[len(times) // 2:])  # second half: clocks have settled under the power cap
    ms = tail[len(tail) // 2]
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    t = torch.tensor([1.0 / ms], dtype=torch.float64, device=dev)
    allt = [torch.zeros_like(t) for _ in range(world)]
    if world > 1:
        dist.all_gather(allt, t, group=group)
    else:
        allt = [t]
    rates = [float(x.item()) for x in allt]
    mean = sum(rates) / len(rates)
    return [r / mean for r in rates]


def merge_topk_device(D_all: torch.Tensor, I_all: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """D_all [G, nq, k] f32, I_all [G, nq, k] i64 (CUDA) -> (D [nq,k], I [nq,k]) via kirag_merge_topk."""
    if not D_all.is_cuda:
        raise RuntimeError("kirag_b200.sharded: merge needs CUDA tensors (no CPU fallback)")
    G, nq, k = D_all.shape
    D_all = D_all.contiguous()
    I_all = I_all.contiguous()
    D = torch.empty((nq, k), dtype=torch.float32, device=D_all.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=D_all.device)
    st = torch.cuda.current_stream(D_all.device).cuda_stream
    _lib.check(
        _lib.load().kirag_merge_topk(ctypes.c_void_p(D_all.data_ptr()), ctypes.c_void_p(I_all.data_ptr()), G, nq, k,
                                     ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()), 1,
                                     D_all.device.index, ctypes.c_void_p(st)),
        "merge_topk")
    return D, I


class PeerExchangeUnavailable(RuntimeError):
    """CUDA IPC mapping of a peer's exchange buffer failed on at least one rank (raised on EVERY rank)."""


class PeerExchange:
    """This rank's exchange buffer + the IPC mappings of every peer's (kirag_exchange_* C ABI).

    torch.distributed only carries the 64-byte IPC handles at construction time; the data path is
    the exchange kernel alone.  Every rank must call merge() in the same order with the same
    shapes (SPMD)."""

    def __init__(self, device: int, rank: int, world_size: int, max_nq: int, max_k: int, group=None):
        self._lib = _lib.load()
        self._h = None
        self.device, self.rank, self.world_size = int(device), int(rank), int(world_size)
        self.max_nq, self.max_k = int(max_nq), int(max_k)
        h = ctypes.c_void_p()
        status = self._lib.kirag_exchange_create(self.device, self.rank, self.world_size, self.max_nq, self.max_k,
                                                 ctypes.byref(h))
        err = _lib.last_error() if status else ""
        if self.world_size > 1:
            # agree on the outcome of the allocation before anyone waits for handles: a rank that failed here
            # would otherwise leave the others blocked in the handle exchange below
            created = [None] * self.world_size
            dist.all_gather_object(created, (int(status), err), group=group)
            bad = [(r, e) for r, (st, e) in enumerate(created) if st]
            if bad:
                if not status:
                    self._lib.kirag_exchange_destroy(h)
                raise PeerExchangeUnavailable("peer-memory exchange buffers could not be allocated: " +
                                              "; ".join(f"rank {r}: {e}" for r, e in bad))
        elif status:
            raise _lib.KiragError(f"exchange_create: {err}")
        self._h = h
        if self.world_size > 1:
            nb = int(self._lib.kirag_exchange_handle_bytes())
            mine = ctypes.create_string_buffer(nb)
            _lib.check(self._lib.kirag_exchange_export(self._h, mine), "exchange_export")
            handles = [None] * self.world_size
            dist.all_gather_object(handles, bytes(mine.raw), group=group)
            blob = b"".join(handles)
            assert len(blob) == nb * self.world_size
            # mapping a peer's buffer fails where the peer GPU is not visible / not P2P-reachable from this
            # process; every rank has to reach the same verdict, so the outcome is agreed on before anyone
            # raises (a half-connected group would dead-lock in the first exchange)
            status = self._lib.kirag_exchange_connect(self._h, blob)
            err = _lib.last_error() if status else ""
            outcomes = [None] * self.world_size
            dist.all_gather_object(outcomes, (int(status), err), group=group)  # also the "everyone has mapped" barrier
            bad = [(r, e) for r, (st, e) in enumerate(outcomes) if st]
            if bad:
                self.close()
                raise PeerExchangeUnavailable("peer-memory exchange could not be set up: " +
                                              "; ".join(f"rank {r}: {e}" for r, e in bad))

    def fits(self, nq: int, k: int) -> bool:
        return 0 < k <= self.max_k and nq * k <= self.max_nq * self.max_k

    def merge(self, D_loc: torch.Tensor, I_loc: torch.Tensor, flags_ptr: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        """D_loc [nq,k] f32, I_loc [nq,k] i64 (this rank's sorted per-shard result) -> global (D, I).
        `flags_ptr`: device address of this rank's per-query certificate flags (IndexFlatIP.pending_flags_ptr());
        when given on EVERY rank, the flags travel with the rows and any_flag() is valid after a stream sync."""
        nq, k = D_loc.shape
        D_loc = D_loc.contiguous()
        I_loc = I_loc.contiguous()
        D = torch.empty_like(D_loc)
        I = torch.empty_like(I_loc)
        st = torch.cuda.current_stream(D_loc.device).cuda_stream
        if flags_ptr:
            _lib.check(
                self._lib.kirag_exchange_merge_topk_flags(self._h, ctypes.c_void_p(D_loc.data_ptr()),
                                                          ctypes.c_void_p(I_loc.data_ptr()), ctypes.c_void_p(flags_ptr),
                                                          nq, k, ctypes.c_void_p(D.data_ptr()),
                                                          ctypes.c_void_p(I.data_ptr()), ctypes.c_void_p(st)),
                "exchange_merge_topk_flags")
        else:
            _lib.check(
                self._lib.kirag_exchange_merge_topk(self._h, ctypes.c_void_p(D_loc.data_ptr()),
                                                    ctypes.c_void_p(I_loc.data_ptr()), nq, k,
                                                    ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()),
                                                    ctypes.c_void_p(st)),
                "exchange_merge_topk")
        return D, I

    def any_flag(self) -> int:
        """OR over all ranks and queries of the flags carried by the last merge(..., flags_ptr) (after a stream
        synchronisation).  The same value on every rank."""
        v = int(self._lib.kirag_exchange_last_any_flag(self._h))
        if v < 0:
            raise _lib.KiragError(f"exchange: {_lib.last_error()}")
        return v

    def close(self) -> None:
        h, self._h = self._h, None
        if h is not None:
            self._lib.kirag_exchange_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ShardedFlatIP:
    """SPMD sharded index: every rank calls add_shard()/search() with the same arguments."""

    def __init__(self, d: int, n_total: int, rank: Optional[int] = None, world_size: Optional[int] = None,
                 device: Optional[int] = None, group=None,
                 local_index=None, merge_fn: Optional[Callable] = None, exchange: Optional[str] = None,
                 max_nq: int = 16384, max_k: int = 128, weights=None, master: Optional[str] = None):
        self.d = d
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world_size = dist.get_world_size(group) if world_size is None else world_size
        self.n_total = int(n_total)
        self.weights = None if weights is None else [float(w) for w in weights]
        self.lo, self.hi = shard_range(self.n_total, self.world_size, self.rank, self.weights)
        if local_index is None:
            from .faiss_api import IndexFlatIP

            local_index = IndexFlatIP(d, device=device, master=master)
            local_index.reserve(max(self.hi - self.lo, 1))
        from .faiss_api import IndexIDMap

        if isinstance(local_index, IndexIDMap) or getattr(local_index, "_flags", 0) & _lib.INDEX_ID_MAP:
            raise RuntimeError("ShardedFlatIP: the local index is an IndexIDMap; the row-sharded search returns global "
                               "row numbers and does not support id maps")
        self.index = local_index
        self.merge_fn = merge_fn or merge_topk_device
        # "peer": fused NVLink exchange+merge kernel; "nccl": all-gather + merge kernel.  An injected
        # local index / merge (the CPU gloo tests) always takes the collective path.
        injected = merge_fn is not None or not hasattr(self.index, "device")
        self.exchange = exchange or os.environ.get("KIRAG_EXCHANGE") or ("nccl" if injected else "peer")
        assert self.exchange in ("peer", "nccl"), f"unknown exchange {self.exchange!r}"
        self.peer: Optional[PeerExchange] = None
        if self.exchange == "peer" and self.world_size > 1:
            try:
                self.peer = PeerExchange(self.index.device, self.rank, self.world_size, max_nq, max_k, group=group)
            except PeerExchangeUnavailable as exc:
                if exchange == "peer" or os.environ.get("KIRAG_EXCHANGE") == "peer":
                    raise  # explicitly requested
                # every rank raised together: all of them fall back to the collective path
                warnings.warn(f"kirag_b200.sharded: {exc}; using the NCCL all-gather + merge path instead")
                self.exchange = "nccl"

    def close(self) -> None:
        """Collective teardown of the peer mappings: nobody unmaps or frees a buffer a peer may still be
        writing to.  Call it on every rank before destroying the process group (optional: process exit
        cleans up as well)."""
        if self.peer is not None:
            torch.cuda.synchronize(self.index.device)
            dist.barrier(group=self.group)
            self.peer.close()
            self.peer = None
            dist.barrier(group=self.group)

    @property
    def ntotal_local(self) -> int:
        return int(self.index.ntotal)

    def add_shard(self, x_local) -> None:
        """Append rows of THIS rank's range (in order).  Tensor (CUDA) or ndarray."""
        if isinstance(x_local, torch.Tensor) and x_local.is_cuda:
            self.index.add_device(x_local.contiguous().float())
        else:
            self.index.add(x_local.numpy() if isinstance(x_local, torch.Tensor) else x_local)
        assert self.index.ntotal <= self.hi - self.lo, "more rows added than this rank's shard holds"

    def search_local(self, q: torch.Tensor, k: int, path: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """Per-shard exact top-k with global ids.  `path`: a KIRAG_PATH_* selector (default AUTO; EXACT = the fp32
        CUDA-core scan, what bench.py's parity block and the large-config tests compare AUTO with)."""
        if path is None:
            return self.index.search_device(q, k, id_offset=self.lo)
        return self.index.search_device(q, k, id_offset=self.lo, path=path)

    def search(self, q: torch.Tensor, k: int, path: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """q [nq, d] replicated on every rank -> (D [nq,k], I [nq,k]) global result on every rank.

        With the peer exchange the certificate of the local search is verified AFTER the exchange: the local search
        is enqueued without a host synchronisation, its per-query flags travel with the rows, the exchange kernel
        ORs them over all ranks (the same word on every rank), and only if some rank had to re-answer a query do
        all ranks run the exchange a second time.  One stream synchronisation per search, at its very end."""
        nq = q.shape[0]
        if (path is None and self.peer is not None and self.world_size > 1 and self.peer.fits(nq, k)
                and 0 < nq <= min(self.peer.max_nq, 16384) and hasattr(self.index, "search_device_async")):
            D_loc, I_loc = self.index.search_device_async(q, k, id_offset=self.lo)
            flags_ptr = self.index.pending_flags_ptr()
            # ranks can only disagree on flags_ptr if one of them holds an empty shard: those carry zeros
            if not flags_ptr:
                self._zero_flags = getattr(self, "_zero_flags", None)
                if self._zero_flags is None or self._zero_flags.numel() < nq:
                    self._zero_flags = torch.zeros(max(nq, 1024), dtype=torch.int32, device=q.device)
                flags_ptr = self._zero_flags.data_ptr()
            D, I = self.peer.merge(D_loc, I_loc, flags_ptr)
            torch.cuda.current_stream(q.device).synchronize()
            redo = self.peer.any_flag()
            self.index.finish()  # re-answers this rank's flagged queries in place (no-op where none were flagged)
            if redo:
                D, I = self.peer.merge(D_loc, I_loc)
            return D, I
        D_loc, I_loc = self.search_local(q, k, path=path)
        return self.exchange_merge(D_loc, I_loc)

    def range_search(self, q: torch.Tensor, radius: float) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """q [nq, d] replicated on every rank -> (lims [nq+1], D, I) over the whole corpus, identical on every rank:
        every global row with score > radius, per query ordered by (score desc, id asc).  Each rank answers its shard
        (global ids), the per-query counts and the padded D/I arrays are all-gathered, and the lists are assembled
        here: shard ranges are contiguous and ascending in rank order, so a stable sort by score over the rank-ordered
        concatenation keeps equal scores in ascending id order."""
        lims_l, D_l, I_l = self.index.range_search_device(q, radius, id_offset=self.lo)
        if self.world_size == 1:
            return lims_l, D_l, I_l
        nq = q.shape[0]
        counts = (lims_l[1:] - lims_l[:-1]).contiguous()
        all_counts = [torch.empty_like(counts) for _ in range(self.world_size)]
        dist.all_gather(all_counts, counts, group=self.group)
        totals = [int(c.sum()) for c in all_counts]
        width = max(max(totals), 1)
        D_pad = torch.zeros(width, dtype=D_l.dtype, device=D_l.device)
        I_pad = torch.zeros(width, dtype=I_l.dtype, device=I_l.device)
        D_pad[:D_l.numel()] = D_l
        I_pad[:I_l.numel()] = I_l
        all_D = [torch.empty_like(D_pad) for _ in range(self.world_size)]
        all_I = [torch.empty_like(I_pad) for _ in range(self.world_size)]
        dist.all_gather(all_D, D_pad, group=self.group)
        dist.all_gather(all_I, I_pad, group=self.group)
        qids = torch.arange(nq, device=counts.device)
        D = torch.cat([d[:t] for d, t in zip(all_D, totals)])
        I = torch.cat([i[:t] for i, t in zip(all_I, totals)])
        owner = torch.cat([torch.repeat_interleave(qids, c) for c in all_counts])
        order = torch.sort(D, descending=True, stable=True).indices
        order = order[torch.sort(owner[order], stable=True).indices]
        per_query = torch.stack(all_counts).sum(dim=0)
        lims = torch.zeros(nq + 1, dtype=torch.int64, device=counts.device)
        lims[1:] = torch.cumsum(per_query, dim=0)
        return lims, D[order], I[order]

    def search_graph(self, q: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """search() for small query batches with the whole chain — local search, exchange+merge kernel, flag
        read-back — replayed from ONE CUDA graph per (nq, k): a graph launch and a stream synchronisation are all the
        host does per call (KiRAG's own shape is 1-2 queries per retrieval, knowledge_graph/models.py:1645).  Every
        rank must call it with the same shapes (SPMD).  The returned tensors are the graph's static output buffers
        (overwritten by the next call with the same shape)."""
        nq = int(q.shape[0])
        if not (self.peer is not None and self.world_size > 1 and self.peer.fits(nq, k) and 0 < nq <= 1024
                and hasattr(self.index, "capture_search")):
            return self.search(q, k)
        cache = self.__dict__.setdefault("_graphs", {})
        key = (nq, int(k))
        cap = cache.get(key)
        if cap is None or cap["token"] != self.index.state_token():
            # capturing executes nothing (no rendez-vous with the peers), so a rank may recapture on its own
            def tail(D_loc, I_loc):
                return self.peer.merge(D_loc, I_loc, self.index.pending_flags_ptr())

            cap = cache[key] = self.index.capture_search(nq, int(k), id_offset=self.lo, tail=tail)
        cur = torch.cuda.current_stream(q.device)
        cap["stream"].wait_stream(cur)
        with torch.cuda.stream(cap["stream"]):
            cap["q"].copy_(q, non_blocking=True)
            self.index.replay_search(cap)
            cap["stream"].synchronize()
            redo = self.peer.any_flag()
            self.index.finish()
            D, I = cap["extra"]
            if redo:
                D, I = self.peer.merge(cap["D"], cap["I"])
                cap["stream"].synchronize()
        return D, I

    def exchange_merge(self, D_loc: torch.Tensor, I_loc: torch.Tensor,
                       lists_sorted: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
        """Per-rank results [nq,k] with globally unique ids (padding id -1) -> the global top-k on every rank.
        `lists_sorted`: every row is ordered by (score desc, id asc) — what the peer kernel's sort-free merge
        relies on; pass False (same value on every rank) to take the collective path, whose merge kernel sorts."""
        if self.world_size == 1:
            return D_loc, I_loc
        nq, k = D_loc.shape
        if lists_sorted and self.peer is not None and self.peer.fits(nq, k):
            return self.peer.merge(D_loc, I_loc)
        # ONE collective for scores and ids: the payload is tiny (12*nq*k bytes per rank), so the
        # exchange is latency-bound and a second all-gather would double its cost.  Scores ride in
        # the same int64 tensor as the ids (bit-cast, zero-extended).
        packed = torch.empty((2, nq, k), dtype=torch.int64, device=I_loc.device)
        packed[0] = D_loc.contiguous().view(torch.int32).to(torch.int64)
        packed[1] = I_loc
        gathered = torch.empty((self.world_size, 2, nq, k), dtype=torch.int64, device=I_loc.device)
        dist.all_gather_into_tensor(gathered.view(-1, k), packed.view(-1, k), group=self.group)
        D_all = gathered[:, 0].to(torch.int32).view(torch.float32).contiguous()
        I_all = gathered[:, 1].contiguous()
        return self.merge_fn(D_all, I_all)
