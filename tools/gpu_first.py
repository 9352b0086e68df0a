"""First-contact checks on a B200, each stage in its own process with a timeout so that a hang or a
trap in one kernel does not hide the others.  Prints one line per stage."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGES = {
    "device": """
import torch, ctypes
from kirag_b200 import _lib
lib=_lib.load(); print('devices', lib.kirag_device_count(), torch.cuda.get_device_name(0), torch.cuda.get_device_properties(0).multi_processor_count)
""",
    "exact_small": """
import numpy as np
from kirag_b200 import faiss_api
from oracle import oracle
rng=np.random.default_rng(0)
xb=rng.integers(-3,4,size=(20000,128)).astype(np.float32); xq=rng.integers(-3,4,size=(9,128)).astype(np.float32)
ix=faiss_api.IndexFlatIP(128); ix.add(xb)
D,I,st=ix.search_ex(xq,10,path=1); Do,Io=oracle.flat_ip_search(xb,xq,10)
print('exact ids equal', np.array_equal(I,Io), 'scores equal', np.array_equal(D,Do), st)
""",
    "tc_scores_resident": """
import numpy as np
from kirag_b200 import faiss_api
rng=np.random.default_rng(0)
for (n,d,nq) in ((256,64,4),(1000,128,32),(4096,1024,8)):
    xb=rng.integers(-3,4,size=(n,d)).astype(np.float32); xq=rng.integers(-3,4,size=(nq,d)).astype(np.float32)
    ix=faiss_api.IndexFlatIP(d); ix.add(xb)
    got=ix.debug_scores(xq); ref=(xb.astype(np.float64)@xq.astype(np.float64).T).astype(np.float32)
    bad=np.argwhere(got!=ref)
    print('tc resident', (n,d,nq), 'exact' if len(bad)==0 else f'MISMATCH {len(bad)} of {got.size}; first {bad[:5].tolist()} got {got[tuple(bad[0])]} ref {ref[tuple(bad[0])]}' )
""",
    "tc_scores_streamed": """
import numpy as np
from kirag_b200 import faiss_api
rng=np.random.default_rng(0)
for (n,d,nq) in ((300,64,40),(1000,128,100),(2000,1024,200),(1000,256,600)):
    xb=rng.integers(-3,4,size=(n,d)).astype(np.float32); xq=rng.integers(-3,4,size=(nq,d)).astype(np.float32)
    ix=faiss_api.IndexFlatIP(d); ix.add(xb)
    got=ix.debug_scores(xq); ref=(xb.astype(np.float64)@xq.astype(np.float64).T).astype(np.float32)
    bad=np.argwhere(got!=ref)
    print('tc streamed', (n,d,nq), 'exact' if len(bad)==0 else f'MISMATCH {len(bad)} of {got.size}; first {bad[:5].tolist()} got {got[tuple(bad[0])]} ref {ref[tuple(bad[0])]}' )
""",
    "tc_scores_pair": """
import os, numpy as np
os.environ['KIRAG_DEBUG_BQ']='256s'
from kirag_b200 import faiss_api
rng=np.random.default_rng(0)
for (n,d,nq) in ((256,64,256),(300,64,40),(1000,128,300),(2100,1024,520),(128,64,256),(129,256,1)):
    xb=rng.integers(-3,4,size=(n,d)).astype(np.float32); xq=rng.integers(-3,4,size=(nq,d)).astype(np.float32)
    ix=faiss_api.IndexFlatIP(d); ix.add(xb)
    got=ix.debug_scores(xq); ref=(xb.astype(np.float64)@xq.astype(np.float64).T).astype(np.float32)
    bad=np.argwhere(got!=ref)
    print('tc pair', (n,d,nq), 'exact' if len(bad)==0 else f'MISMATCH {len(bad)} of {got.size}; first {bad[:5].tolist()} got {got[tuple(bad[0])]} ref {ref[tuple(bad[0])]}' )
""",
    "auto_small": """
import numpy as np
from kirag_b200 import faiss_api
from oracle import oracle
rng=np.random.default_rng(1)
xb=rng.standard_normal((100000,128)).astype(np.float32); xb/=np.linalg.norm(xb,axis=1,keepdims=True)
xq=rng.standard_normal((16,128)).astype(np.float32); xq/=np.linalg.norm(xq,axis=1,keepdims=True)
ix=faiss_api.IndexFlatIP(128); ix.add(xb)
D,I,st=ix.search_ex(xq,10); Do,Io=oracle.flat_ip_search(xb,xq,10,accum='f64')
print('auto ids equal', np.array_equal(I,Io), 'max score err', float(np.max(np.abs(D-Do))), st)
""",
    "pool": """
import numpy as np, torch
from kirag_b200 import pooling
from oracle import oracle
h=torch.randn(8,512,1024); m=(torch.arange(512)[None,:]<torch.randint(1,513,(8,))[:,None]).to(torch.int64)
got=pooling.e5_embed(h.cuda(),m.cuda()).cpu(); ref=oracle.pool_normalize_torch(h,m)
print('pool max err', float((got-ref).abs().max()))
""",
    "smoke": "import __graft_entry__ as g; g.smoke()",
}

if __name__ == "__main__":
    names = sys.argv[1:] or list(STAGES)
    rc_all = 0
    for name in names:
        try:
            p = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r)\n" % ROOT + STAGES[name]],
                               cwd=ROOT, capture_output=True, text=True, timeout=240)
            tail = (p.stdout + p.stderr).strip().splitlines()[-12:]
            print(f"[{name}] rc={p.returncode}")
            for line in tail:
                print("   ", line)
            rc_all |= p.returncode != 0
        except subprocess.TimeoutExpired:
            print(f"[{name}] TIMEOUT")
            rc_all |= 1
    sys.exit(int(rc_all))
