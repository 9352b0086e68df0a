"""IndexIDMap against a plain IndexFlatIP on the bench corpus, one process:
   python tools/probe_id_map.py [OUT_DIR]          (default OUT_DIR: profiles/r08_id_map)
The bench corpus (bench.build_shard: seeded, d = 1024), PROBE_ROWS rows (default 10M: the plain index and the id map
are held at once, 2 x 61 GB), is built into a plain index and an id map whose ids are a seeded random int64 permutation.
  search    B = 1 / 32 / 4096 queries, k = 100, device pointers: the two indexes alternate, PROBE_REPS rounds of
            PROBE_STEPS calls each after a warm-up; the outputs are checked equal (D bit-equal, I = ids[I_plain])
  remove    1 % of the rows at random: by external id on the id map, by position on the plain index (the same rows);
            host clock around a synchronised call; afterwards the two indexes are checked equal again
  io        write_index / read_index of both (IxMp against IxFI) under PROBE_IO_DIR (default: a temporary directory)
The first line holds every visible card's name and power limit, read in the same run.  One JSON line per record, also
written (as it comes) to OUT_DIR/probe.jsonl."""
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from kirag_b200 import faiss_api  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r08_id_map")
D_MODEL = bench.D_MODEL
rows = int(os.environ.get("PROBE_ROWS", 10_000_000))
steps = int(os.environ.get("PROBE_STEPS", 20))
reps = int(os.environ.get("PROBE_REPS", 3))
K = 100
dev = torch.device("cuda", 0)
os.makedirs(out_dir, exist_ok=True)
out_file = open(os.path.join(out_dir, "probe.jsonl"), "w")


def emit(rec):
    print(json.dumps(rec), flush=True)
    out_file.write(json.dumps(rec) + "\n")
    out_file.flush()


def timed(fn):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(dev)
    return (time.perf_counter() - t0) * 1e3, out


cards = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
emit({"cards": cards, "rows": rows, "d": D_MODEL, "k": K, "steps": steps, "reps": reps})

rng = np.random.default_rng(88)
ids = rng.permutation(rows).astype(np.int64) * 1_000_003 - (1 << 40)
plain = faiss_api.IndexFlatIP(D_MODEL, device=0)
plain.reserve(rows)
t_build = timed(lambda: bench.build_shard(plain, 0, rows, dev))[0]
idmap = faiss_api.IndexIDMap(faiss_api.IndexFlatIP(D_MODEL, device=0))
idmap.index.reserve(rows)
piece = 1 << 20
t_copy = 0.0
for r in range(0, rows, piece):  # the same rows, copied from the plain index
    x = torch.from_numpy(plain.reconstruct_n(r, min(piece, rows - r))).to(dev)
    t_copy += timed(lambda: idmap.add_with_ids_device(x, torch.from_numpy(ids[r:r + x.shape[0]]).to(dev)))[0]
emit({"build_plain_ms": round(t_build, 1), "add_with_ids_ms": round(t_copy, 1), "storage_plain": plain.storage_bytes(),
      "storage_id_map": idmap.storage_bytes()})
ids_dev = torch.from_numpy(ids).to(dev)


def check(B):
    q = torch.nn.functional.normalize(torch.randn((B, D_MODEL), device=dev, generator=torch.Generator(dev).manual_seed(B)),
                                      dim=1)
    Dp, Ip = plain.search_device(q, K)
    Dm, Im = idmap.search_device(q, K)
    want = torch.where(Ip >= 0, ids_dev[Ip.clamp(min=0)], torch.full_like(Ip, -1))
    return bool(torch.equal(Dp, Dm) and torch.equal(Im, want)), q


for B in (1, 32, 4096):
    equal, q = check(B)
    times = {"plain": [], "id_map": []}
    for ix in (plain, idmap):
        for _ in range(3):
            ix.search_device(q, K)
    for _ in range(reps):
        for name, ix in (("plain", plain), ("id_map", idmap)):
            ms = timed(lambda: [ix.search_device(q, K) for _ in range(steps)])[0] / steps
            times[name].append(round(ms, 4))
    emit({"case": "search", "B": B, "equal": equal, "ms_per_call": times})

sel = np.sort(rng.choice(rows, size=rows // 100, replace=False))
ms_map, n_map = timed(lambda: idmap.remove_ids(ids[sel]))
ms_plain, n_plain = timed(lambda: plain.remove_ids(sel))
ids = np.delete(ids, sel)
ids_dev = torch.from_numpy(ids).to(dev)
equal = all(check(B)[0] for B in (1, 32, 4096)) and np.array_equal(idmap.id_map, ids)
emit({"case": "remove_p1", "ms_id_map_by_id": round(ms_map, 2), "ms_plain_by_position": round(ms_plain, 2),
      "removed": [n_map, n_plain], "equal_after": bool(equal)})

io_dir = os.environ.get("PROBE_IO_DIR") or tempfile.mkdtemp(prefix="probe_id_map_")
paths, n_rows = {}, idmap.ntotal
for name, ix in (("IxFI", plain), ("IxMp", idmap)):
    paths[name] = os.path.join(io_dir, f"{name}.faiss")
    emit({"case": "io_write", "format": name, "write_ms": round(timed(lambda: faiss_api.write_index(ix, paths[name]))[0], 1),
          "bytes": os.path.getsize(paths[name])})
del plain, idmap  # the reads below need the HBM
gc.collect()
for name, path in paths.items():
    ms_r, back = timed(lambda: faiss_api.read_index(path, device=0))
    ok = back.ntotal == n_rows and (name == "IxFI" or np.array_equal(back.id_map, ids))
    emit({"case": "io_read", "format": name, "read_ms": round(ms_r, 1), "ok": bool(ok)})
    del back
    gc.collect()
    os.remove(path)
out_file.close()
