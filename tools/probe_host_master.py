"""Host-resident fp32 master against device master, one GPU, one process:
   python tools/probe_host_master.py [OUT_DIR]          (default OUT_DIR: profiles/r05_host_master)
The bench corpus (bench.build_shard, d = 1024) with 21M rows when /proc/meminfo's MemAvailable leaves room for the 86 GB
of pinned master plus PROBE_HEADROOM_GB (default 24) of headroom, else the largest whole number of millions of rows
that does (recorded).  Both arms cannot sit in HBM together, so each round builds the device-master index, measures it,
frees it, then does the same with the host-master index; PROBE_ROUNDS (default 2) rounds alternate them.  Per arm and
round: add time; per cell B x k (PROBE_BATCHES, default 1,2,32,128,1024,4096; k in 10, 100): ms per search_device call
(CUDA events around PROBE_STEPS calls after a warm-up), the scan ms and the tail (last scan -> final) and rescoring ms
from one call's phase timeline (kirag_profile_*; a device-master call of at most 128 queries runs the fused tail, which
has no separate rescoring mark), and one KIRAG_PATH_EXACT call of 256 queries.  Also: the cudaMemcpyAsync rate of a
1 GiB pinned buffer to the device (the PCIe reference), the bytes rescoring could read at most (B x k' x d x 4: the
s~_k - 2 eps skip reads fewer; the count actually read is not instrumented), whether AUTO equals EXACT on 16 sampled
queries, and whether the host arm's D / I equal the device arm's for every cell's sampled queries.  One JSON line per
record, also written (as it comes) to OUT_DIR/probe.jsonl, after a line with the card name and power limit."""
import ctypes
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from kirag_b200 import _lib, faiss_api  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r05_host_master")
D_MODEL = bench.D_MODEL
batches = [int(b) for b in os.environ.get("PROBE_BATCHES", "1,2,32,128,1024,4096").split(",")]
ks = (10, 100)
steps = int(os.environ.get("PROBE_STEPS", 5))
rounds = int(os.environ.get("PROBE_ROUNDS", 2))
headroom = float(os.environ.get("PROBE_HEADROOM_GB", 24)) * 1e9
dev = torch.device("cuda", 0)
lib = _lib.load()
os.makedirs(out_dir, exist_ok=True)
out_file = open(os.path.join(out_dir, "probe.jsonl"), "w")


def emit(rec):
    # written as it comes: a run cut short keeps what it measured
    print(json.dumps(rec), flush=True)
    out_file.write(json.dumps(rec) + "\n")
    out_file.flush()


def mem_available() -> int:
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    raise RuntimeError("no MemAvailable in /proc/meminfo")


avail = mem_available()
fit = int((avail - headroom) // (D_MODEL * 4) // 1_000_000 * 1_000_000)
rows = int(os.environ.get("PROBE_ROWS", min(21_000_000, fit)))
assert rows > 0, f"MemAvailable {avail / 1e9:.1f} GB leaves no room for a host master"
card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
emit({"card": card, "rows": rows, "d": D_MODEL, "mem_available_gb": avail / 1e9, "rows_that_fit": fit,
      "reduced": rows < 21_000_000, "steps": steps, "rounds": rounds, "batches": batches, "k": list(ks)})


def timed(fn, n):
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / n


# PCIe reference: 1 GiB pinned host -> device with cudaMemcpyAsync (torch's copy_ of a pinned tensor)
h_buf = torch.empty(1 << 28, dtype=torch.float32, pin_memory=True)
d_buf = torch.empty(1 << 28, dtype=torch.float32, device=dev)
d_buf.copy_(h_buf, non_blocking=True)
h2d_ms = timed(lambda: d_buf.copy_(h_buf, non_blocking=True), 5)
emit({"h2d_pinned_1gib_ms": h2d_ms, "h2d_gbs": (1 << 30) / (h2d_ms * 1e-3) / 1e9})
del h_buf, d_buf

g = torch.Generator(device=dev)
g.manual_seed(4321)
q_all = torch.nn.functional.normalize(torch.randn(max(batches + [256]), D_MODEL, generator=g, device=dev), dim=1)


def phases(fn):
    """scan ms, tail ms (last scan mark -> final) and rescoring ms (mark 50 - the mark before it) of one call."""
    lib.kirag_profile_enable(1)
    fn()
    torch.cuda.synchronize(dev)
    tags = (ctypes.c_int * 256)()
    ms = (ctypes.c_double * 256)()
    n = lib.kirag_profile_read_timeline(tags, ms, 256)
    scan_ms, launches, srows = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
    lib.kirag_profile_read(ctypes.byref(scan_ms), ctypes.byref(launches), ctypes.byref(srows))
    lib.kirag_profile_enable(0)
    t = [(tags[i], ms[i]) for i in range(n)]
    last_scan = max((m for tg, m in t if 10 <= tg < 30), default=None)
    final = next((m for tg, m in t if tg == 51), None)
    resc = None
    for i, (tg, m) in enumerate(t):
        if tg == 50 and i > 0:
            resc = m - t[i - 1][1]
    return {"scan_ms": scan_ms.value, "scan_launches": launches.value,
            "tail_ms": None if last_scan is None or final is None else final - last_scan, "rescore_ms": resc}


def host(x):
    return x.cpu().numpy()


samples = {}   # (B, k) -> {arm: (D, I)} of 16 sampled queries
results = []
for r in range(rounds):
    for arm in ("device", "host"):
        gc.collect()
        torch.cuda.empty_cache()
        t0 = time.perf_counter()
        ix = faiss_api.IndexFlatIP(D_MODEL, device=0, master=arm)
        ix.reserve(rows)
        t1 = time.perf_counter()
        bench.build_shard(ix, 0, rows, dev)
        t2 = time.perf_counter()
        emit({"round": r, "arm": arm, "reserve_s": t1 - t0, "add_s": t2 - t1, "storage_bytes": ix.storage_bytes()})
        for B in batches:
            q = q_all[:B].contiguous()
            idx = torch.from_numpy(np.sort(np.random.default_rng(B).choice(B, min(16, B), replace=False))).to(dev)
            for k in ks:
                def call():
                    return ix.search_device(q, k)

                call()
                ms = timed(call, steps)
                st = dict(ix.last_stats)
                ph = phases(call)
                kprime = min(max(4 * k, 32), 2048)
                qs = q[idx].contiguous()
                Da, Ia = ix.search_device(qs, k, path=_lib.PATH_AUTO)
                De, Ie = ix.search_device(qs, k, path=_lib.PATH_EXACT)
                auto_eq_exact = bool(torch.equal(Da, De) and torch.equal(Ia, Ie))
                samples.setdefault((B, k), {})[arm] = (host(Da), host(Ia))
                rb_max = B * kprime * D_MODEL * 4
                rec = {"round": r, "arm": arm, "batch": B, "k": k, "ms": ms, **ph,
                       "rescore_bytes_at_most": rb_max if arm == "host" else None,
                       "rescore_gbs_at_most": (rb_max / (ph["rescore_ms"] * 1e-3) / 1e9
                                               if arm == "host" and ph["rescore_ms"] else None),
                       "stats": {key: st[key] for key in ("n_fast", "n_exact", "n_cert_fail", "n_overflow", "levels")},
                       "auto_equals_exact_sampled": auto_eq_exact}
                emit(rec)
                results.append(rec)
        q = q_all[:256].contiguous()
        ix.search_device(q[:8], 10, path=_lib.PATH_EXACT)
        t0 = time.perf_counter()
        De, Ie = ix.search_device(q, 10, path=_lib.PATH_EXACT)
        torch.cuda.synchronize(dev)
        emit({"round": r, "arm": arm, "exact_256_queries_s": time.perf_counter() - t0,
              "exact_stats": {key: ix.last_stats[key] for key in ("n_exact",)}})
        samples.setdefault(("exact", 256), {})[arm] = (host(De), host(Ie))
        del ix, q
        gc.collect()
        torch.cuda.synchronize(dev)

same = {f"{key[0]}x{key[1]}": bool(np.array_equal(v["device"][0], v["host"][0]) and np.array_equal(v["device"][1], v["host"][1]))
        for key, v in samples.items() if len(v) == 2}
emit({"host_equals_device_sampled": same, "all_equal": all(same.values())})
summary = {}
for rec in results:
    key = f"B={rec['batch']} k={rec['k']}"
    summary.setdefault(key, {"device_ms": [], "host_ms": []})[rec["arm"] + "_ms"].append(round(rec["ms"], 3))
emit({"summary_ms": summary})
out_file.close()
