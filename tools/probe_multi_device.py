"""Multi-device index (IndexFlatIP(devices=[...])) against a single-device index, one process:
   python tools/probe_multi_device.py [OUT_DIR]          (default OUT_DIR: profiles/r06_multi_device)
The bench corpus (bench.build_shard: seeded, d = 1024), PROBE_ROWS rows (default 21M), is built once per configuration:
a single-device index on cuda:0, then multi-device indexes over G = 1, 2, 4 and 8 distinct GPUs (as many as are
visible; PROBE_GS overrides the list), and G shards on cuda:0 alone for G in PROBE_SAME_GPU_GS (default 2, 8: no
speed-up is possible there; it prices the worker threads and the merge).  Per configuration and batch B in
PROBE_BATCHES (default 1, 32, 4096), k = 100:
  ms            host clock around PROBE_STEPS synchronised search_device calls after a warm-up call;
  merge_ms      device time of multi_merge_kernel in one profiled call (torch.profiler, CUDA activities);
  shard_ms_max  the slowest device: first kernel start to last kernel end of the same profiled call, the merge kernel left
                out (host gaps inside that span count as shard time; with several shards on one device, their sum);
  equal         whether D / I equal the single-device index's bit for bit (all B queries).
The first line holds every visible card's name and power limit, read in the same run.  One JSON line per record, also
written (as it comes) to OUT_DIR/probe.jsonl."""
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from kirag_b200 import faiss_api  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r06_multi_device")
D_MODEL = bench.D_MODEL
rows = int(os.environ.get("PROBE_ROWS", 21_000_000))
batches = [int(b) for b in os.environ.get("PROBE_BATCHES", "1,32,4096").split(",")]
steps = int(os.environ.get("PROBE_STEPS", 10))
K = 100
n_gpus = torch.cuda.device_count()
gs = [int(g) for g in os.environ.get("PROBE_GS", "1,2,4,8").split(",") if int(g) <= n_gpus]
same_gpu_gs = [int(g) for g in os.environ.get("PROBE_SAME_GPU_GS", "2,8").split(",") if g]
dev = torch.device("cuda", 0)
os.makedirs(out_dir, exist_ok=True)
out_file = open(os.path.join(out_dir, "probe.jsonl"), "w")


def emit(rec):
    # written as it comes: a run cut short keeps what it measured
    print(json.dumps(rec), flush=True)
    out_file.write(json.dumps(rec) + "\n")
    out_file.flush()


cards = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
emit({"cards": cards, "visible": n_gpus, "rows": rows, "d": D_MODEL, "k": K, "batches": batches, "steps": steps,
      "configs": ["single"] + [f"G={g}" for g in gs] + [f"G={g} on cuda:0" for g in same_gpu_gs]})

g = torch.Generator(device=dev)
g.manual_seed(4321)
q_all = torch.nn.functional.normalize(torch.randn(max(batches), D_MODEL, generator=g, device=dev), dim=1)


def sync_all():
    for i in range(n_gpus):
        torch.cuda.synchronize(i)


def profiled(fn):
    """merge kernel ms and the slowest device's kernel span (ms) of one call."""
    from torch.profiler import ProfilerActivity, profile

    sync_all()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        sync_all()
    merge_us, span = 0.0, {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        if "multi_merge_kernel" in e.name:
            merge_us += e.time_range.elapsed_us()
            continue
        lo, hi = span.get(e.device_index, (float("inf"), 0.0))
        span[e.device_index] = (min(lo, e.time_range.start), max(hi, e.time_range.end))
    per_dev = {int(d): (hi - lo) / 1e3 for d, (lo, hi) in span.items()}
    return merge_us / 1e3, per_dev


reference = {}
summary = {}
configs = [("single", None)] + [(f"G={g}", list(range(g))) for g in gs]
configs += [(f"G={g} on cuda:0", [0] * g) for g in same_gpu_gs]
for name, devices in configs:
    gc.collect()
    sync_all()
    t0 = time.perf_counter()
    ix = faiss_api.IndexFlatIP(D_MODEL, device=0) if devices is None else faiss_api.IndexFlatIP(D_MODEL, devices=devices)
    ix.reserve(rows)
    bench.build_shard(ix, 0, rows, dev)
    sync_all()
    emit({"config": name, "devices": ix.devices, "build_s": time.perf_counter() - t0, "storage": ix.storage_bytes()})
    for B in batches:
        q = q_all[:B].contiguous()

        def call():
            return ix.search_device(q, K)

        D, I = call()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(steps):
            call()
        sync_all()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        merge_ms, per_dev = profiled(call) if devices is not None else (None, None)
        if devices is None:
            reference[B] = (D.cpu(), I.cpu())
            equal = True
        else:
            equal = bool(torch.equal(D.cpu(), reference[B][0]) and torch.equal(I.cpu(), reference[B][1]))
        rec = {"config": name, "batch": B, "k": K, "ms": ms, "qps": B / (ms * 1e-3), "merge_ms": merge_ms,
               "shard_ms_max": max(per_dev.values()) if per_dev else None, "device_span_ms": per_dev,
               "stats": {key: ix.last_stats[key] for key in ("n_fast", "n_exact", "n_cert_fail", "levels")},
               "equal_to_single": equal}
        emit(rec)
        summary.setdefault(f"B={B}", {})[name] = round(ms, 3)
    del ix
    gc.collect()
    torch.cuda.empty_cache()
emit({"summary_ms": summary})
out_file.close()
