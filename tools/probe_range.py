"""Range search against top-k search at equal result counts, one GPU, one process (the corpus is built once):
   python tools/probe_range.py [OUT_DIR]
The bench corpus (bench.build_shard: PROBE_ROWS rows x 1024, default 21M) and the bench queries (seed 4321).  Per batch
B (PROBE_BATCHES, default 1,32,128,1024,4096) the radius is the median over the batch of the 100th-best score of
search(k=100), so both calls return ~100 rows per query.  Reported per B: ms per call of range_search_device and of
search_device(k=100) (CUDA events around PROBE_STEPS calls after warm-up, the two alternated PROBE_REPS times), the
filter scan's roofline fraction from the kirag_profile_* scan events (same formula and peaks as bench.py: MEASURED_PEAKS.json,
else bench.py's fallback figures; the header line records which), a host-clock split of one range call into its two C calls
(search, fetch), the stats of the range
call, and whether AUTO equals EXACT (lims, D, I) on 32 sampled queries.  One JSON line per batch, also written to
OUT_DIR/probe.jsonl, after a line with the card name and power limit."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from kirag_b200 import _lib, faiss_api  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else None
rows = int(os.environ.get("PROBE_ROWS", 21_000_000))
batches = [int(b) for b in os.environ.get("PROBE_BATCHES", "1,32,128,1024,4096").split(",")]
steps = int(os.environ.get("PROBE_STEPS", 5))
reps = int(os.environ.get("PROBE_REPS", 2))
K = 100
dev = torch.device("cuda", 0)
D_MODEL = bench.D_MODEL
peaks = bench.load_peaks()
lib = _lib.load()
lines = []


def emit(rec):
    print(json.dumps(rec), flush=True)
    lines.append(rec)


card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
emit({"card": card, "rows": rows, "d": D_MODEL, "k": K, "steps": steps, "reps": reps, "peak_source": peaks["source"],
      "peak_hbm_gbs": peaks["hbm_gbs"], "peak_bf16_tflops_sustained": peaks["bf16_tflops_sustained"]})

ix = faiss_api.IndexFlatIP(D_MODEL, device=0)
ix.reserve(rows)
bench.build_shard(ix, 0, rows, dev)
g = torch.Generator(device=dev)
g.manual_seed(4321)
q_all = torch.nn.functional.normalize(torch.randn(max(batches), D_MODEL, generator=g, device=dev), dim=1)


def timed(fn):
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / steps


def scan_roofline(fn, batch):
    lib.kirag_profile_enable(1)
    for _ in range(steps):
        fn()
    torch.cuda.synchronize(dev)
    scan_ms, launches, srows = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
    lib.kirag_profile_read(ctypes.byref(scan_ms), ctypes.byref(launches), ctypes.byref(srows))
    lib.kirag_profile_enable(0)
    ms = scan_ms.value / steps
    r = srows.value / steps
    bytes_alg = r * D_MODEL * 2 + batch * D_MODEL * 4
    flops_alg = 2.0 * batch * r * D_MODEL
    if bytes_alg / (peaks["hbm_gbs"] * 1e9) >= flops_alg / (peaks["bf16_tflops_sustained"] * 1e12):
        frac, bound = bytes_alg / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "hbm"
    else:
        frac, bound = flops_alg / (ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"], "tensor"
    return {"scan_ms": ms, "scan_launches": launches.value / steps, "bound": bound, "frac": frac}


def host(t):
    return t.cpu().numpy()


def split_call(q, radius):
    """Host-clock ms of the two C calls behind range_search_device: the search (synchronous, returns lims) and the
    fetch of D / I into device tensors."""
    import time

    n = q.shape[0]
    lims = np.zeros(n + 1, dtype=np.int64)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    _lib.check(lib.kirag_index_range_search(ix._h, ctypes.c_void_p(q.data_ptr()), n, radius, 1, 0, 0,
                                            ctypes.c_void_p(lims.ctypes.data), None, st), "range_search")
    t1 = time.perf_counter()
    D = torch.empty(int(lims[n]), dtype=torch.float32, device=dev)
    I = torch.empty(int(lims[n]), dtype=torch.int64, device=dev)
    _lib.check(lib.kirag_index_range_fetch(ix._h, ctypes.c_void_p(D.data_ptr()), ctypes.c_void_p(I.data_ptr()), 1, st),
               "range_fetch")
    t2 = time.perf_counter()
    return {"search_ms": (t1 - t0) * 1e3, "fetch_ms": (t2 - t1) * 1e3}


for B in batches:
    q = q_all[:B].contiguous()
    Dk, _ = ix.search_device(q, K)
    radius = float(torch.median(Dk[:, K - 1]).item())

    def rng_call():
        return ix.range_search_device(q, radius)

    def topk_call():
        return ix.search_device(q, K)

    for _ in range(2):
        rng_call()
        topk_call()
    t_range, t_topk = [], []
    for _ in range(reps):
        t_range.append(timed(rng_call))
        t_topk.append(timed(topk_call))
    split = [split_call(q, radius) for _ in range(3)]
    lims, D, I = rng_call()
    stats = dict(ix.last_stats)
    lims_h, D_h, I_h = host(lims), host(D), host(I)
    roof_range = scan_roofline(rng_call, B)
    roof_topk = scan_roofline(topk_call, B)
    # AUTO == EXACT on sampled queries, and the sampled queries' lists equal their rows of the whole batch's answer
    idx = np.sort(np.random.default_rng(B).choice(B, min(32, B), replace=False))
    qs = q[torch.from_numpy(idx).to(dev)].contiguous()
    a = [host(t) for t in ix.range_search_device(qs, radius, path=_lib.PATH_AUTO)]
    e = [host(t) for t in ix.range_search_device(qs, radius, path=_lib.PATH_EXACT)]
    same = all(np.array_equal(x, y) for x, y in zip(a, e))
    for j, i in enumerate(idx):
        same = same and np.array_equal(a[1][a[0][j]:a[0][j + 1]], D_h[lims_h[i]:lims_h[i + 1]]) \
            and np.array_equal(a[2][a[0][j]:a[0][j + 1]], I_h[lims_h[i]:lims_h[i + 1]])
    counts = np.diff(lims_h)
    emit({"batch": B, "radius": radius, "range_ms": t_range, "topk_ms": t_topk,
          "range_over_topk": min(t_range) / min(t_topk), "range_call_split": split, "results_per_query_mean": float(counts.mean()),
          "results_per_query_max": int(counts.max()), "stats": stats, "range_scan": roof_range,
          "topk_scan": roof_topk, "auto_equals_exact_sampled": bool(same), "sampled_queries": int(len(idx))})

if out_dir:
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "probe.jsonl"), "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
