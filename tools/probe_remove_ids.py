"""IndexFlatIP.remove_ids on the bench corpus, one process:
   python tools/probe_remove_ids.py [OUT_DIR]          (default OUT_DIR: profiles/r07_remove_ids)
The bench corpus (bench.build_shard: seeded, d = 1024), PROBE_ROWS rows (default 21M), is built once per configuration:
a device master on cuda:0, a host master on cuda:0, and G = 2 shards on cuda:0.  After a warm-up removal (the last
row), each configuration times three removals in turn, host clock around a synchronised call:
  row0    row 0: every row after it moves (the whole master is read and written through staging, one convert pass)
  last    the last row: nothing moves
  p1      1 % of the rows at random (seeded)
Afterwards, on PROBE_Q sampled queries (k = 100): AUTO equals EXACT bit for bit, and the queries that were copies of
removed rows (taken before the removal) no longer find their row: the returned ids' rows differ from the query.
The first line holds every visible card's name and power limit, read in the same run.  One JSON line per record, also
written (as it comes) to OUT_DIR/probe.jsonl."""
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
from kirag_b200 import faiss_api  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r07_remove_ids")
D_MODEL = bench.D_MODEL
rows = int(os.environ.get("PROBE_ROWS", 21_000_000))
n_q = int(os.environ.get("PROBE_Q", 64))
configs = os.environ.get("PROBE_CONFIGS", "device,host,G=2 on cuda:0").split(",")
K = 100
dev = torch.device("cuda", 0)
os.makedirs(out_dir, exist_ok=True)
out_file = open(os.path.join(out_dir, "probe.jsonl"), "w")


def emit(rec):
    print(json.dumps(rec), flush=True)
    out_file.write(json.dumps(rec) + "\n")
    out_file.flush()


cards = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
emit({"cards": cards, "rows": rows, "d": D_MODEL, "k": K, "queries": n_q, "configs": configs})

for name in configs:
    gc.collect()
    torch.cuda.synchronize(dev)
    try:
        if name == "device":
            ix = faiss_api.IndexFlatIP(D_MODEL, device=0)
        elif name == "host":
            ix = faiss_api.IndexFlatIP(D_MODEL, device=0, master="host")
        else:
            ix = faiss_api.IndexFlatIP(D_MODEL, devices=[0, 0])
        ix.reserve(rows)
        t0 = time.perf_counter()
        bench.build_shard(ix, 0, rows, dev)
        torch.cuda.synchronize(dev)
    except Exception as e:  # e.g. not enough pinned host memory for the host master
        emit({"config": name, "error": str(e)[:300]})
        continue
    emit({"config": name, "build_s": time.perf_counter() - t0, "ntotal": ix.ntotal, "storage": ix.storage_bytes()})
    rng = np.random.default_rng(77)
    ix.remove_ids([ix.ntotal - 1])  # warm-up: workspaces and staging allocated
    n = ix.ntotal
    sel_p1 = np.sort(rng.choice(n - 1, size=n // 100, replace=False)) + 1  # old row 0 is gone by then
    probe_rows = sel_p1[rng.choice(sel_p1.size, size=n_q, replace=False)]
    xq = np.stack([ix.reconstruct(int(r)) for r in probe_rows])
    for case in ("row0", "last", "p1"):
        n0 = ix.ntotal
        ids = [0] if case == "row0" else [n0 - 1] if case == "last" else sel_p1 - 1  # p1 in the ids after row0
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        removed = ix.remove_ids(ids)
        torch.cuda.synchronize(dev)
        ms = (time.perf_counter() - t0) * 1e3
        emit({"config": name, "case": case, "ms": round(ms, 3), "removed": removed, "ntotal_before": n0,
              "ntotal_after": ix.ntotal})
    Da, Ia, st_a = ix.search_ex(xq, K, path=0)
    De, Ie, _ = ix.search_ex(xq, K, path=1)
    top = np.stack([ix.reconstruct(int(i)) for i in Ia[:, 0]])
    emit({"config": name, "auto_equals_exact": bool(np.array_equal(Ia, Ie) and np.array_equal(Da.view(np.uint32),
                                                                                           De.view(np.uint32))),
          "removed_rows_found": int(np.sum(np.all(top == xq, axis=1))), "stats": st_a})
    del ix
    gc.collect()
    torch.cuda.empty_cache()
out_file.close()
