#!/usr/bin/env python
"""bench.py — QPS of exact inner-product top-100 over a 21M x 1024 synthetic corpus on N B200s.

`python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.  A "step" is one search
of a batch of B queries against the whole corpus; the headline times K of them after W warm-up steps.
`--dump-outputs DIR` writes what the last timed step returned (scores.npy float32, ids.npy float64).

  value   QPS with queries and results resident in HBM (kirag_index_search, device pointers)
  e2e     QPS through the reference-facing call with HOST buffers: pinned-host queries in,
          host D/I out (faiss-shaped IndexFlatIP.search -> kirag_index_search_ex, host pointers)
  roofline  the tcgen05 filter scan (dominant kernel), timed live with CUDA events on its stream
            (kirag_profile_*): HBM GB/s for B <= 128, bf16 TFLOP/s above
  cpu_baseline  the FAISS-equivalent CPU restatement (oracle/, blocked sgemm + heap) on a bounded
            sample of the same workload, all host threads
  --impl reference   times that CPU restatement alone (FAISS itself is not installable here)

Synthetic data (SURVEY.md §8d): unit-norm Gaussian rows generated on device in 2^20-row chunks,
seed 1234 + chunk, so every GPU count sees the same global matrix; queries seed 4321.
Corpus (43 GB bf16 / 86 GB fp32) is far larger than the 126 MB L2, so no L2 flush is needed.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CHUNK = 1 << 20
D_MODEL = 1024


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--rows", type=int, default=int(os.environ.get("KIRAG_BENCH_ROWS", 21_000_000)))
    ap.add_argument("--batch", type=int, default=int(os.environ.get("KIRAG_BENCH_BATCH", 4096)))
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--sweep", type=str, default=os.environ.get("KIRAG_BENCH_SWEEP", "1,32,256,1024,16384"),
                    help="extra query batch sizes reported in `sweep` (comma separated, '' for none)")
    ap.add_argument("--cpu-sample-rows", type=int, default=0, help="rows of the CPU sample (0: 2^20)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the N=1 extras (other BASELINE configs, pooling, stress corpus, index I/O)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (scores, ids) as DIR/<name>.npy, "
                         "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 4096  # upper bound of one .npy header (numpy writes 128 bytes for these shapes)


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each [n, ...] array as out_dir/<name>.npy: float32 stays float32, everything else becomes float64 (exact
    for ids).  If the files would exceed DUMP_LIMIT_BYTES in all, headers included, the same fixed, seeded sample of
    rows is taken from every array and its row numbers are written as rows.npy."""
    import numpy as np

    arrays = {name: np.asarray(a) for name, a in arrays.items()}
    arrays = {name: a if a.dtype == np.float32 else a.astype(np.float64) for name, a in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    if sum(a.nbytes for a in arrays.values()) + NPY_HEADER_BYTES * len(arrays) > DUMP_LIMIT_BYTES:
        row_bytes = sum(a.nbytes for a in arrays.values()) // n + 8  # + 8: the row number in rows.npy
        keep = min(n, max(1, (DUMP_LIMIT_BYTES - NPY_HEADER_BYTES * (len(arrays) + 1)) // row_bytes))
        rows = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
                pw.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        pw.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w": pw[len(pw) // 2] if pw else None}


def workload_config(rows: int, batch: int, k: int) -> dict:
    """The `config` of the bench line: identical for both arms (ours and --impl reference) at every N — the workload
    is the same corpus, batch and k; how each arm runs it is described in `arm`."""
    return {"workload": f"DPR psgs_w100-scale {rows}x{D_MODEL} fp32 corpus (BASELINE configs[3]), query batch {batch}, "
                        f"exact inner-product top-{k}",
            "rows": rows, "dim": D_MODEL, "batch": batch, "k": k,
            "l2": "inputs (86 GB fp32 / 43 GB bf16) far larger than the 126 MB L2; no flush needed"}


# ------------------------------------------------------------------ reference arm ---
def cpu_baseline(batch: int, k: int, rows_total: int, sample_rows: int, steps: int = 1, warmup: int = 0):
    """FAISS-equivalent CPU search (oracle/) on a bounded sample, extrapolated linearly in N
    (flat search is exactly linear in the number of rows).  Returns (qps_at_rows_total, info)."""
    import numpy as np
    import torch

    from oracle import oracle

    oracle.build()
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    g = torch.Generator().manual_seed(1234)
    sample_rows = int(min(sample_rows, rows_total))
    xb = torch.nn.functional.normalize(torch.randn(sample_rows, D_MODEL, generator=g), dim=1).numpy()
    gq = torch.Generator().manual_seed(4321)
    b = int(min(batch, 1024))  # bounded: at most one FAISS query block of the batch
    xq = torch.nn.functional.normalize(torch.randn(b, D_MODEL, generator=gq), dim=1).numpy()
    # a real faiss-cpu wheel, should one ever be present on the box, IS the reference (SURVEY §8c/d): time the
    # unmodified library instead of the restatement.  (Never our own stand-in: that one is backed by the GPU.)
    real_faiss = None
    try:
        import faiss as _f

        if "kirag_b200" not in (getattr(_f, "__file__", "") or "") and hasattr(_f, "IndexFlatIP") and \
                not getattr(_f, "__kirag_b200__", False):
            real_faiss = _f
    except Exception:
        real_faiss = None
    if real_faiss is not None:
        try:
            real_faiss.omp_set_num_threads(cores)
        except Exception:
            pass
        ix = real_faiss.IndexFlatIP(D_MODEL)
        ix.add(xb)
        for _ in range(warmup):
            ix.search(xq, k)
        times = []
        for _ in range(max(1, steps)):
            t0 = time.perf_counter()
            out = ix.search(xq, k)
            times.append(time.perf_counter() - t0)
        t = sorted(times)[len(times) // 2]
        qps = b / (t * (rows_total / sample_rows))
        info = {"value": qps, "unit": "queries/s", "cores": cores, "kind": "reference",
                "sample": f"{b} queries x {sample_rows} rows x {D_MODEL} (of {batch} x {rows_total}), top-{k}, "
                          f"faiss {getattr(real_faiss, '__version__', '?')} IndexFlatIP.search, median of {len(times)} x "
                          f"{t:.3f}s, extrapolated linearly in rows"}
        return qps, info, t, out
    # pick the faster host BLAS for the blocked sgemm (MKL through torch, OpenBLAS through numpy)
    best = None
    for use_torch in (True, False):
        t0 = time.perf_counter()
        oracle.flat_ip_search_blas(xb[:16384], xq, k, use_torch=use_torch)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, use_torch)
    use_torch = best[1]
    for _ in range(warmup):
        oracle.flat_ip_search_blas(xb, xq, k, use_torch=use_torch)
    times = []
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        if b < 20:
            out = oracle.flat_ip_search(xb, xq, k)  # FAISS's n < 20 path: per-query scan, threads over queries
        else:
            out = oracle.flat_ip_search_blas(xb, xq, k, use_torch=use_torch)
        times.append(time.perf_counter() - t0)
    t = sorted(times)[len(times) // 2]
    qps = b / (t * (rows_total / sample_rows))
    info = {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"{b} queries x {sample_rows} rows x {D_MODEL} (of {batch} x {rows_total}), top-{k}, "
                      f"{'MKL(torch.mm)' if use_torch else 'OpenBLAS(numpy)'} sgemm 4096x1024 tiles + heap, "
                      f"median of {len(times)} x {t:.3f}s, extrapolated linearly in rows",
            "note": "FAISS-equivalent CPU restatement; faiss-cpu is not installable in this image"}
    return qps, info, t, out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    qps, info, t, (D, I) = cpu_baseline(args.batch, args.k, args.rows, args.cpu_sample_rows or (1 << 20),
                                        steps=args.steps, warmup=min(args.warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"scores": D, "ids": I})
    line = {
        "impl": "reference", "metric": "QPS, exact IP top-%d over %dx%d" % (args.k, args.rows, D_MODEL),
        "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        # a step of this arm is one pass over the bounded SAMPLE (what was actually timed); `value` is the metric of
        # the full workload, extrapolated linearly in rows and queries from it
        "ms_per_step": 1000.0 * t, "ms_per_full_step_extrapolated": 1000.0 * args.batch / qps if qps > 0 else None,
        "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.rows, args.batch, args.k),
        "arm": {"how": "FAISS-equivalent CPU flat search on all host cores, each step a bounded sample of the workload "
                       "(see cpu_baseline.sample), throughput extrapolated linearly in rows"},
        "cpu_baseline": info,
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------ our arm ---
def build_shard(index, lo: int, hi: int, device):
    """Fill `index` with global rows [lo, hi) of the synthetic corpus (chunk-seeded, device-generated)."""
    import torch

    g = torch.Generator(device=device)
    c0, c1 = lo // CHUNK, (hi + CHUNK - 1) // CHUNK
    for c in range(c0, c1):
        g.manual_seed(1234 + c)
        x = torch.randn(CHUNK, D_MODEL, generator=g, device=device)
        x = torch.nn.functional.normalize(x, dim=1)
        a, b = max(lo, c * CHUNK), min(hi, (c + 1) * CHUNK)
        index.add_device(x[a - c * CHUNK:b - c * CHUNK].contiguous())
        del x
    torch.cuda.synchronize(device)


def timed_steps(fn, steps, warmup, device, dist_ok):
    import torch
    import torch.distributed as dist

    for _ in range(warmup):
        fn()
    if dist_ok:
        dist.barrier()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(device)
    if dist_ok:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if dist_ok:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms / steps


def measure_batch(sh, lib, q_all, batch, k, steps, warmup, device, dist_ok, peaks, rows_total, world):
    """Device-resident QPS + live roofline of the filter scan for one query batch size."""
    import torch

    q = q_all[:batch].contiguous()
    stats_box = {}

    def step():
        D, I = sh.search(q, k)
        stats_box["stats"] = dict(sh.index.last_stats)
        stats_box["outputs"] = (D, I)
        return D, I

    ms = timed_steps(step, steps, warmup, device, dist_ok)
    outputs = stats_box["outputs"]  # what the last timed step returned (the roofline pass below computes it again)
    # roofline pass: same steps again with per-launch CUDA events on the launching stream
    lib.kirag_profile_enable(1)
    for _ in range(steps):
        step()
    torch.cuda.synchronize(device)
    scan_ms, launches, rows = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
    lib.kirag_profile_read(ctypes.byref(scan_ms), ctypes.byref(launches), ctypes.byref(rows))
    lib.kirag_profile_enable(0)
    scan_ms_step = scan_ms.value / steps
    rows_step = rows.value / steps  # rows streamed by this rank per step
    bytes_alg = rows_step * D_MODEL * 2 + batch * D_MODEL * 4 + batch * k * 12
    flops_alg = 2.0 * batch * rows_step * D_MODEL
    t_hbm = bytes_alg / (peaks["hbm_gbs"] * 1e9)
    t_tc = flops_alg / (peaks["bf16_tflops_sustained"] * 1e12)
    if t_hbm >= t_tc:
        ach = bytes_alg / (scan_ms_step * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"]}
    else:
        ach = flops_alg / (scan_ms_step * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["bf16_tflops_sustained"]}
    # dram__bytes_read.sum + dram__bytes_write.sum of the scan launches of one step.  DRAM counters cannot be read
    # from inside a run, so this is the figure of the committed `ncu --set full` capture of this very command
    # (profiles/r02_scan_traffic.json, produced by tools/profile_r2b.sh) when the workload matches it, else null.
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_scan_traffic.json")
    if world == 1 and rows_total == 21_000_000 and k == 100 and os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(str(batch), {}).get("dram_bytes_per_step")
    roof.update({"traffic": traffic, "traffic_note": "bytes per step (all scan launches of one step); NOT measured in this "
                 "run (DRAM counters cannot be read from inside a run): read from the committed single-pass ncu capture of the "
                 "same command (profiles/r02_scan_traffic.json, raw list profiles/r02_traffic_b4096.csv)",
                 "kernel": ("scan_tc_pair_kernel<256,streamed>" if batch > 128 else "scan_tc_pair_kernel<128,resident>"
                            if batch > 64 else "scan_tc_pair_kernel<64,resident>"), "kernel_ms_per_step": scan_ms_step,
                 "kernel_share_of_step": scan_ms_step / ms if ms > 0 else None,
                 "launches_per_step": launches.value / steps, "peak_source": peaks["source"],
                 "algorithmic_bytes_per_step": bytes_alg, "algorithmic_flops_per_step": flops_alg,
                 "frac_of_burst_peak": (ach / peaks["bf16_tflops"]) if roof["bound"] == "tensor" else None,
                 "frac_note": "peak = the driver-measured SUSTAINED figure (cuBLAS bf16 8192^3 back to back / torch copy): this "
                              "kernel is timed inside a long power-capped step; a frac above 1 means it outruns that "
                              "measurement under the same cap (a read-only stream beats a copy; the filter scan beats "
                              "cuBLAS's sustained rate), see frac_of_burst_peak / frac_of_nominal",
                 "frac_of_nominal": (ach / 7700.0) if roof["bound"] == "hbm" else (ach / 2250.0)})
    return {"batch": batch, "ms_per_step": ms, "qps": batch / (ms * 1e-3), "roofline": roof,
            "stats": stats_box.get("stats", {}), "outputs": outputs}


def parity_check(sh, q_all, batch, k, device, dist_ok, n_sample):
    """Outside every timed region: the certified filter path (KIRAG_PATH_AUTO, what was timed) against the exact
    fp32 CUDA-core scan (KIRAG_PATH_EXACT) on `n_sample` queries spread over the batch — ids and scores must be
    bit-equal — plus the row-order / id-range properties on the whole batch.  For N > 1 both sides go through the
    exchange+merge, and every rank must agree (MIN over ranks)."""
    import torch
    import torch.distributed as dist

    from kirag_b200 import _lib

    q = q_all[:batch].contiguous()
    D, I = sh.search(q, k)
    n_sample = min(n_sample, batch)
    idx = torch.unique(torch.linspace(0, batch - 1, n_sample, device=device).round().long())
    De, Ie = sh.search(q[idx].contiguous(), k, path=_lib.PATH_EXACT)
    torch.cuda.synchronize(device)
    mism = int((I[idx] != Ie).sum().item())
    sdiff = float((D[idx] - De).abs().max().item())
    ordered = bool((((D[:, :-1] > D[:, 1:]) | ((D[:, :-1] == D[:, 1:]) & (I[:, :-1] < I[:, 1:]))).all()).item())
    in_range = bool(((I >= 0) & (I < sh.n_total)).all().item())
    ok = mism == 0 and sdiff == 0.0 and ordered and in_range
    if dist_ok:
        t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        ok = bool(t.item())
    return {"batch": batch, "ok": ok, "checked_queries": int(idx.numel()), "mismatched_ids": mism,
            "max_abs_score_diff": sdiff, "rows_ordered": ordered, "ids_in_range": in_range}


# ------------------------------------------------- the other BASELINE configs, pooling, aligner, index I/O ---
def _event_time_ms(fn, iters, warmup, device):
    """Median and min of `iters` device-timed calls (CUDA events on the current stream), after `warmup` calls."""
    import torch

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(device)
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize(device)
        times.append(e0.elapsed_time(e1))
    times.sort()
    return times[len(times) // 2], times[0]


def _host_time_ms(fn, iters, warmup):
    """Median wall time of a SYNCHRONOUS host call (host buffers in, host buffers out)."""
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t0) * 1e3)
    times.sort()
    return times[len(times) // 2]


def e5_like_rows(n, device, seed, common=0.85):
    """Rows with a large common component, like E5 embeddings (random-pair cosine ~ common^2)."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(9000)
    mu = torch.nn.functional.normalize(torch.randn(1, D_MODEL, generator=g, device=device), dim=1)
    g.manual_seed(seed)
    x = torch.randn(n, D_MODEL, generator=g, device=device)
    x = torch.nn.functional.normalize(x - (x @ mu.T) * mu, dim=1)
    return torch.nn.functional.normalize(common * mu + (1.0 - common * common) ** 0.5 * x, dim=1)


def bench_other_configs(peaks, device):
    """BASELINE configs[0], [1], [2], [4] on one GPU, each through the faiss-shaped HOST call (host ndarray in,
    host ndarrays out: IndexFlatIP.search, what retriever/index.py:47 calls) and with device-resident queries."""
    import numpy as np
    import torch

    from kirag_b200 import faiss_api, scoring

    out = []
    hbm = peaks["hbm_gbs"] * 1e9
    tc = peaks["bf16_tflops_sustained"] * 1e12
    for name, rows, batch, k in (("configs[0] E5-shaped 100k x 1024, 1000 queries, top-10", 100_000, 1000, 10),
                                 ("configs[1] 2Wiki-scale 430k x 1024, batch 64, top-20", 430_000, 64, 20),
                                 ("configs[2] HotpotQA-scale 5.2M x 1024, batch 1024, top-100", 5_200_000, 1024, 100),
                                 ("KiRAG call shape: 5.2M x 1024, 2 queries, top-10", 5_200_000, 2, 10)):
        free, _ = torch.cuda.mem_get_info(device)
        if free < rows * D_MODEL * 6 + (6 << 30):
            out.append({"config": name, "skipped": f"{free >> 30} GiB free"})
            continue
        ix = faiss_api.IndexFlatIP(D_MODEL, device=device.index)
        ix.reserve(rows)
        build_shard(ix, 0, rows, device)
        g = torch.Generator(device=device)
        g.manual_seed(4321)
        q = torch.nn.functional.normalize(torch.randn(batch, D_MODEL, generator=g, device=device), dim=1)
        q_np = np.ascontiguousarray(q.cpu().numpy())
        dev_ms, dev_min = _event_time_ms(lambda: ix.search_device(q, k), 10, 5, device)
        host_ms = _host_time_ms(lambda: ix.search(q_np, k), 10, 3)
        # the whole asynchronous chain replayed from ONE CUDA graph (wall clock per call, stream sync included)
        graph_ms, graph_same = None, None
        if batch <= 1024:
            Dg, Ig = ix.search_device_graph(q, k)
            Dp, Ip = ix.search_device(q, k)
            graph_same = bool(torch.equal(Dg, Dp) and torch.equal(Ig, Ip))
            graph_ms = _host_time_ms(lambda: ix.search_device_graph(q, k), 20, 5)
        dev_call_ms = _host_time_ms(lambda: ix.search_device(q, k), 20, 5)
        D, I = ix.search_device(q, k)
        stats = dict(ix.last_stats)
        De, Ie = ix.search_device(q[:min(batch, 16)].contiguous(), k, path=1)
        t_roof = max(rows * D_MODEL * 2 / hbm, 2.0 * batch * rows * D_MODEL / tc) * 1e3
        out.append({"config": name, "rows": rows, "batch": batch, "k": k, "device_ms": dev_ms, "device_ms_min": dev_min,
                    "host_call_ms": host_ms, "device_call_wall_ms": dev_call_ms, "graph_call_wall_ms": graph_ms,
                    "graph_equals_plain": graph_same, "qps_device": batch / dev_ms * 1e3, "qps_host_call": batch / host_ms * 1e3,
                    "roofline_ms": t_roof, "frac_of_roofline": t_roof / dev_ms,
                    "parity_vs_exact": bool(torch.equal(I[:Ie.shape[0]], Ie) and torch.equal(D[:De.shape[0]], De)),
                    "stats": stats})
        del ix
        torch.cuda.empty_cache()
    # configs[4]: aligner triple scoring, 256 chain queries x 50k candidate triples, top-20, through kirag_topk_ip
    # (the transient candidate matrix is copied + converted on EVERY call: that is part of the measured time)
    g = torch.Generator(device=device)
    g.manual_seed(5)
    T = torch.nn.functional.normalize(torch.randn(50_000, D_MODEL, generator=g, device=device), dim=1)
    Q = torch.nn.functional.normalize(torch.randn(256, D_MODEL, generator=g, device=device), dim=1)
    ms, ms_min = _event_time_ms(lambda: scoring.topk_inner_product(Q, T, 20), 20, 5, device)
    ref_ms, _ = _event_time_ms(lambda: torch.topk(torch.matmul(Q, T.T), k=20, dim=1), 20, 5, device)
    Dk, Ik = scoring.topk_inner_product(Q, T, 20)
    ts, ti = torch.topk(torch.matmul(Q, T.T), k=20, dim=1)
    out.append({"config": "configs[4] aligner: 256 chain queries x 50k triples, top-20 (kirag_topk_ip, per-call setup included)",
                "rows": 50_000, "batch": 256, "k": 20, "device_ms": ms, "device_ms_min": ms_min,
                "torch_matmul_topk_same_gpu_ms": ref_ms,
                "ids_equal_torch_topk": float((Ik == ti).float().mean().item()),
                "max_abs_score_diff": float((Dk - ts).abs().max().item())})
    return out


def bench_pooling(peaks, device):
    """Mean-pool + L2-normalise epilogue on e5-large-v2-shaped hidden states [B, 512, 1024] (configs[4]); HBM roofline
    over the algorithmic bytes sum_b len_b*H*s + B*S*8 + B*H*4.  Inputs (537 MB fp32) exceed the 126 MB L2."""
    import torch

    from kirag_b200 import pooling

    out = []
    for B, dtype, ragged in ((256, torch.float32, False), (256, torch.bfloat16, False), (256, torch.float32, True)):
        S, H = 512, D_MODEL
        g = torch.Generator(device=device)
        g.manual_seed(777)
        h = torch.randn(B, S, H, generator=g, device=device, dtype=torch.float32).to(dtype)
        lens = torch.full((B,), S)
        if ragged:
            lens = torch.randint(1, S + 1, (B,), generator=torch.Generator().manual_seed(778))
        m = (torch.arange(S)[None, :] < lens[:, None]).to(torch.int64).to(device)
        alg = int(lens.sum()) * H * h.element_size() + B * S * 8 + B * H * 4
        # 10 calls per event pair: the kernel takes ~0.1 ms, so a single call between two events would mostly time
        # the host-side launch path of an idle GPU; the input (>= 268 MB) does not fit the 126 MB L2 between calls
        def many(fn, n=10):
            return lambda: [fn() for _ in range(n)]

        ms, ms_min = (t / 10 for t in _event_time_ms(many(lambda: pooling.e5_embed(h, m)), 10, 3, device))
        ref = lambda: torch.nn.functional.normalize(
            h.masked_fill(~m[..., None].bool(), 0.0).sum(dim=1) / m.sum(dim=1)[..., None], p=2, dim=1)
        ref_ms = _event_time_ms(many(ref), 5, 2, device)[0] / 10
        err = float((pooling.e5_embed(h, m).float() - ref().float()).abs().max().item())
        gbs = alg / (ms * 1e-3) / 1e9
        out.append({"shape": [B, S, H], "dtype": str(dtype).replace("torch.", ""), "ragged": ragged, "ms": ms, "ms_min": ms_min,
                    "algorithmic_bytes": alg, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peaks["hbm_gbs"],
                    "reference_aten_ms_same_gpu": ref_ms, "max_abs_diff_vs_reference_expression": err})
        del h
        torch.cuda.empty_cache()
    return out


def bench_stress(device, k):
    """The certificate on an E5-like corpus (rows = normalize(0.85 mu + noise): random-pair cosine 0.72) against the
    i.i.d. corpus of the same size: step time, certificate failures, second passes; answers checked against EXACT."""
    import torch

    from kirag_b200 import faiss_api

    rows = 2_000_000
    out = []
    for kind in ("iid", "e5_like"):
        ix = faiss_api.IndexFlatIP(D_MODEL, device=device.index)
        ix.reserve(rows)
        for c in range(0, rows, 500_000):
            if kind == "iid":
                g = torch.Generator(device=device)
                g.manual_seed(600 + c)
                x = torch.nn.functional.normalize(torch.randn(500_000, D_MODEL, generator=g, device=device), dim=1)
            else:
                x = e5_like_rows(500_000, device, 700 + c)
            ix.add_device(x)
            del x
        for batch in (32, 1024):
            if kind == "iid":
                g = torch.Generator(device=device)
                g.manual_seed(4321)
                q = torch.nn.functional.normalize(torch.randn(batch, D_MODEL, generator=g, device=device), dim=1)
            else:
                q = e5_like_rows(batch, device, 4321)
            ms, _ = _event_time_ms(lambda: ix.search_device(q, k), 10, 5, device)
            D, I = ix.search_device(q, k)
            st = dict(ix.last_stats)
            De, Ie = ix.search_device(q[:16].contiguous(), k, path=1)
            out.append({"corpus": kind, "rows": rows, "batch": batch, "ms_per_step": ms, "n_cert_fail": st["n_cert_fail"],
                        "n_rescan": st["n_rescan"], "n_retry": st["n_retry"], "n_exact": st["n_exact"], "n_overflow": st["n_overflow"],
                        "parity_vs_exact": bool(torch.equal(I[:16], Ie) and torch.equal(D[:16], De))})
        del ix
        torch.cuda.empty_cache()
    return out


def bench_index_io(device):
    """faiss.write_index / faiss.read_index (retriever/index.py:62,73) on the largest corpus the scratch disk takes
    (at most 4M rows = 16 GB): seconds and GB/s of the IxFI file, and the search result before == after."""
    import shutil
    import tempfile

    import torch

    from kirag_b200 import faiss_api

    tmp = tempfile.mkdtemp(prefix="kirag_io_")
    try:
        free_disk = shutil.disk_usage(tmp).free
        rows = 4_000_000
        while rows * D_MODEL * 4 > free_disk * 0.5 and rows > 250_000:
            rows //= 2
        if rows * D_MODEL * 4 > free_disk * 0.5:
            return {"skipped": f"{free_disk >> 30} GiB free on {tmp}"}
        ix = faiss_api.IndexFlatIP(D_MODEL, device=device.index)
        ix.reserve(rows)
        build_shard(ix, 0, rows, device)
        g = torch.Generator(device=device)
        g.manual_seed(4321)
        q = torch.nn.functional.normalize(torch.randn(8, D_MODEL, generator=g, device=device), dim=1)
        D0, I0 = ix.search_device(q, 10)
        path = os.path.join(tmp, "index.faiss")
        t0 = time.perf_counter()
        faiss_api.write_index(ix, path)
        write_s = time.perf_counter() - t0
        del ix
        torch.cuda.empty_cache()
        t0 = time.perf_counter()
        ix2 = faiss_api.read_index(path, faiss_api.IO_FLAG_MMAP, device=device.index)
        load_s = time.perf_counter() - t0
        D1, I1 = ix2.search_device(q, 10)
        gb = rows * D_MODEL * 4 / 1e9
        return {"rows": rows, "file_gb": gb, "write_s": write_s, "write_gbs": gb / write_s, "load_s": load_s,
                "load_gbs": gb / load_s, "note": "load = read the IxFI file (page cache warm from the write) through two "
                "pinned 64 MB buffers + one convert pass; includes building the bf16 shadow",
                "same_results_after_reload": bool(torch.equal(I0, I1) and torch.equal(D0, D1))}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from kirag_b200 import _build, _lib
    from kirag_b200.sharded import ShardedFlatIP, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist_ok = world > 1
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if dist_ok:
        dist.init_process_group("nccl", device_id=device)
    if rank == 0:
        _build.build()
    if dist_ok:
        dist.barrier()
    lib = _lib.load()
    peaks = load_peaks()
    k, B = args.k, args.batch

    # N > 1: a strong-scaling step is paced by the slowest GPU, and the GPUs of one box sit at different power-capped
    # clocks (rank_diag of the r01 / r02 runs: 18.0 ... 19.9 ms of local search on equal shards).  Every rank's speed
    # is measured on a small probe index (all ranks at the same time, ~2 s, outside every timed region) and the row
    # ranges are made proportional to it.  KIRAG_BENCH_EQUAL_SHARDS=1 keeps equal shards.
    weights = None
    measured_weights = None
    if dist_ok and os.environ.get("KIRAG_BENCH_EQUAL_SHARDS", "0") != "1":
        from kirag_b200.sharded import measure_rank_weights

        weights = measure_rank_weights(D_MODEL, local_rank, nq=min(B, 4096), k=k)
        measured_weights = list(weights)
        if max(weights) / min(weights) < 1.03:  # within the noise of the probe: equal shards
            weights = None
    sh = ShardedFlatIP(D_MODEL, args.rows, rank=rank, world_size=world, device=local_rank, weights=weights)
    t_build = time.perf_counter()
    build_shard(sh.index, sh.lo, sh.hi, device)
    build_s = time.perf_counter() - t_build
    gq = torch.Generator(device=device)
    gq.manual_seed(4321)
    sweep = [int(s) for s in args.sweep.split(",") if s.strip()] if args.sweep else []
    max_b = max([B] + sweep)
    q_all = torch.nn.functional.normalize(torch.randn(max_b, D_MODEL, generator=gq, device=device), dim=1)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    head = measure_batch(sh, lib, q_all, B, k, args.steps, args.warmup, device, dist_ok, peaks, args.rows, world)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        D, I = head.pop("outputs")
        dump_outputs(args.dump_outputs, {"scores": D.cpu().numpy(), "ids": I.cpu().numpy()})

    # where a multi-GPU step goes: every rank's LOCAL search time (no exchange) and the exchange alone.  The step
    # is paced by the slowest rank (GPUs of one box sit at different power-capped clocks), so max(local) + exchange
    # ~ ms_per_step explains the scaling loss that is not kernel time.
    rank_diag = None
    if dist_ok:
        qh = q_all[:B].contiguous()
        # all ranks time their local search AT THE SAME TIME (rank 0 arrives late: it stops the clock sampler first):
        # the GPUs of one chassis share its power and cooling, a GPU that runs while its neighbours idle is ~10 %
        # faster (rank 0 looked like that in every earlier rank_diag)
        dist.barrier()
        local_ms = timed_steps(lambda: sh.search_local(qh, k), max(3, min(args.steps, 5)), 2, device, False)
        D_loc, I_loc = sh.search_local(qh, k)
        exch = (lambda: sh.peer.merge(D_loc, I_loc)) if sh.peer is not None else (lambda: sh.search(qh, k))
        exch_ms = timed_steps(exch, 10, 3, device, True) if sh.peer is not None else None
        t = torch.tensor([local_ms], dtype=torch.float64, device=device)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        rank_diag = {"local_search_ms_per_rank": [round(float(x.item()), 3) for x in allt],
                     "exchange_merge_ms": exch_ms,
                     "shard_weights": None if weights is None else [round(w, 4) for w in weights],
                     "measured_rank_speeds": None if measured_weights is None else [round(w, 4) for w in measured_weights],
                     "shard_rows": [b_ - a_ for a_, b_ in (shard_range(args.rows, world, r_, weights) for r_ in range(world))]}

    # end to end through the reference-facing call with HOST buffers (rank-local shard; for N > 1 the
    # exchange + merge are included through the device path and the final result is copied out)
    q_host = torch.empty((B, D_MODEL), dtype=torch.float32, pin_memory=True)
    q_host.copy_(q_all[:B].cpu())
    q_np = q_host.numpy()
    launches_box = {}

    def e2e_step():
        if world == 1:
            D, I = sh.index.search(q_np, k)  # faiss-shaped call: host ndarray in, host ndarrays out
            launches_box["n"] = sh.index.last_stats.get("kernel_launches", 0)
        else:
            qd = q_host.to(device, non_blocking=True)
            D, I = sh.search(qd, k)
            D, I = D.cpu(), I.cpu()
            launches_box["n"] = sh.index.last_stats.get("kernel_launches", 0) + 1
        return D, I

    e2e_steps = max(2, min(args.steps, 5))
    e2e_ms = timed_steps(e2e_step, e2e_steps, min(args.warmup, 2), device, dist_ok)

    sweep_out = []
    for b in sweep:
        if b == B:
            continue
        # short steps right after the power-capped headline phase: warm up longer so that the clocks have settled
        sw_sampler = ClockSampler(local_rank)
        if rank == 0:
            sw_sampler.start()
        # a step of a small batch takes ~1 ms on an 8-GPU shard: time enough of them (>= ~0.1 s) for a stable figure
        sw_steps = 100 if b <= 128 else 20 if b <= 1024 else max(3, min(args.steps, 5))
        r = measure_batch(sh, lib, q_all, b, k, sw_steps, 10 if b <= 1024 else 3, device, dist_ok,
                          peaks, args.rows, world)
        sw_clocks = sw_sampler.stop() if rank == 0 else None
        sweep_out.append({"batch": b, "qps": r["qps"], "ms_per_step": r["ms_per_step"],
                          "sm_mhz": (sw_clocks or {}).get("sm_mhz"), "power_w": (sw_clocks or {}).get("power_w"),
                          "throttle_reasons": (sw_clocks or {}).get("reasons"),
                          "roofline_bound": r["roofline"]["bound"], "roofline_frac": r["roofline"]["frac"],
                          "roofline_achieved": r["roofline"]["achieved"], "roofline_unit": r["roofline"]["unit"],
                          "n_fast": r["stats"].get("n_fast"), "n_exact": r["stats"].get("n_exact"), "steps": sw_steps})

    # parity where the numbers are quoted (outside every timed region; every rank takes part for N > 1)
    checks = [parity_check(sh, q_all, B, k, device, dist_ok, 64)]
    for b in sweep:
        if b != B:
            checks.append(parity_check(sh, q_all, b, k, device, dist_ok, 16))
    parity = {"ok": all(c["ok"] for c in checks), "checked_queries": sum(c["checked_queries"] for c in checks),
              "method": "KIRAG_PATH_AUTO (timed path) vs KIRAG_PATH_EXACT (fp32 CUDA-core scan of the master) on sampled "
                        "queries of every measured batch size: ids and scores bit-equal; all rows ordered by (score desc, "
                        "id asc); for N > 1 both through the exchange+merge, MIN over ranks",
              "per_batch": checks}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the CPU leg runs in its own process (own thread-pool settings), through the reference arm
        try:
            env = {k_: v for k_, v in os.environ.items() if not k_.endswith("_NUM_THREADS")}
            proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3",
                                   "--warmup", "1", "--batch", str(B), "--k", str(k), "--rows", str(args.rows),
                                   "--cpu-sample-rows", str(args.cpu_sample_rows or (1 << 20))],
                                  capture_output=True, text=True, timeout=600, env=env)
            cpu = json.loads(proc.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as exc:  # the baseline is a reported number, never a reason to lose the line
            cpu = {"value": None, "unit": "queries/s", "cores": len(os.sched_getaffinity(0)), "kind": "port",
                   "sample": f"failed: {exc}"}
    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        # everything below needs the HBM the 21M-row index occupies
        sh.index._destroy()
        torch.cuda.empty_cache()
        extras = {}
        for name, fn in (("configs", lambda: bench_other_configs(peaks, device)), ("pooling", lambda: bench_pooling(peaks, device)),
                         ("stress", lambda: bench_stress(device, k)), ("index_io", lambda: bench_index_io(device))):
            try:
                extras[name] = fn()
            except Exception as exc:  # an extra is a reported number, never a reason to lose the line
                extras[name] = {"failed": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()
    if rank == 0:
        line = {
            "metric": "QPS, exact IP top-%d over %dx%d" % (k, args.rows, D_MODEL),
            "value": head["qps"], "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16 filter + f32 rescoring", "data": "synthetic",
            "config": workload_config(args.rows, B, k),
            "arm": {"k_prime": min(4 * k, 2048),
                    "parallelism": (f"row-shard x{world} + " + ("fused NVLink peer-memory exchange+merge kernel"
                                                                 if sh.peer is not None else "all_gather(k) + merge"))
                    if world > 1 else "single GPU"},
            "roofline": head["roofline"],
            "cpu_baseline": cpu,
            "e2e": {"value": B / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": B * D_MODEL * 4, "d2h_bytes_per_step": B * k * 12},
            "gpu_launches": (int(head["stats"].get("kernel_launches", 0)) + (1 if world > 1 else 0)) * args.steps,
            "clocks": clocks,
            "search_stats": head["stats"],
            "parity": parity,
            "rank_diag": rank_diag,
            "sweep": sweep_out,
            "build_s": build_s,
            "build_note": f"rank 0's shard ({sh.hi - sh.lo} rows) from device-generated 2^20-row chunks through "
                          "IndexFlatIP.add_device (fp32 copy + bf16 shadow convert), storage reserved up front",
        }
        if extras is not None:
            line.update(extras)
        emit(line)
    if dist_ok:
        sh.close()
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, warnings) to stderr."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _REAL_STDOUT
    args = parse_args()
    # libraries (NCCL's version banner, for one) print to fd 1: keep the contract's single JSON line clean
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1; the CPU arm must use every host core (set before torch/numpy load)
        cores = str(len(os.sched_getaffinity(0)))
        for var in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
            os.environ[var] = cores
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
