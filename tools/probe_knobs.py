"""A/B of scan-kernel knobs on one GPU inside ONE process (the corpus is built once):
   python tools/probe_knobs.py ROWS B1,B2,... "ENV1=a,ENV2=b;ENV1=c,..."  — prints ms/step per (setting, batch).
PROBE_D: corpus width (default: the bench corpus, d = 1024); other widths are seeded unit rows generated on the device.
PROBE_SAVE: directory; the first result of each batch is saved there as d{D}_b{B}.npz (D, I), so that two builds,
each run in its own process, can be compared bit for bit."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from kirag_b200 import faiss_api  # noqa: E402

rows = int(sys.argv[1])
batches = [int(b) for b in sys.argv[2].split(",")]
settings = [dict(kv.split("=") for kv in s.split(",") if kv) for s in sys.argv[3].split(";")]
steps = int(os.environ.get("PROBE_STEPS", 5))
reps = int(os.environ.get("PROBE_REPS", 2))
dev = torch.device("cuda", 0)
d = int(os.environ.get("PROBE_D", bench.D_MODEL))
save = os.environ.get("PROBE_SAVE")
ix = faiss_api.IndexFlatIP(d, device=0)
ix.reserve(rows)
g = torch.Generator(device=dev)
if d == bench.D_MODEL:
    bench.build_shard(ix, 0, rows, dev)
else:
    chunk = max(1, (1 << 28) // d)  # 1 GB of fp32 per chunk
    for c, a in enumerate(range(0, rows, chunk)):
        g.manual_seed(1234 + c)
        ix.add_device(torch.nn.functional.normalize(torch.randn(min(chunk, rows - a), d, generator=g, device=dev), dim=1))
    torch.cuda.synchronize()
g.manual_seed(4321)
q_all = torch.nn.functional.normalize(torch.randn(max(batches), d, generator=g, device=dev), dim=1)
ref = {}
for rep in range(reps):
    for st in settings:
        for k_, v in st.items():
            os.environ[k_] = v
        for B in batches:
            q = q_all[:B].contiguous()
            for _ in range(3):
                D, I = ix.search_device(q, 100)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                D, I = ix.search_device(q, 100)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            key = B
            same = ""
            if key in ref:
                same = " same" if (torch.equal(ref[key][1], I) and torch.equal(ref[key][0], D)) else " DIFFERENT RESULT"
            else:
                ref[key] = (D.clone(), I.clone())
                if save:
                    os.makedirs(save, exist_ok=True)
                    np.savez(os.path.join(save, f"d{d}_b{B}.npz"), D=D.cpu().numpy(), I=I.cpu().numpy())
            print(f"rep {rep} {st} B={B:6d} {ms:9.3f} ms/step  {B / ms * 1e3:10.1f} qps{same}", flush=True)
