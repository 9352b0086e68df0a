"""`import kirag_b200.as_faiss` makes `import faiss` resolve to the B200 library.

The reference has no plugin registry for its index: the seam is the
`import faiss` line of /root/reference/retriever/index.py:6.  Importing this
module BEFORE the reference's `retriever.index` puts a module object exposing
the symbols KiRAG uses into `sys.modules["faiss"]`, so `retriever/index.py`,
`retriever/retrievers.py`, `faiss_index_corpus.py` and `retrieve.py` run
byte-for-byte unmodified on the sm_100a search path.
"""
from __future__ import annotations

import sys
import types

from . import faiss_api

_EXPORTED = [
    "IndexFlatIP", "IndexFlatL2", "IndexPQ", "IndexIDMap", "IDSelectorBatch", "IDSelectorRange", "METRIC_INNER_PRODUCT",
    "METRIC_L2", "IO_FLAG_MMAP", "IO_FLAG_READ_ONLY", "write_index", "read_index", "vector_to_array",
    "omp_get_max_threads", "get_num_gpus",
]


def make_module() -> types.ModuleType:
    mod = types.ModuleType("faiss")
    mod.__doc__ = "kirag_b200 stand-in for the subset of faiss used by KiRAG (sm_100a, no CPU path)"
    for name in _EXPORTED:
        setattr(mod, name, getattr(faiss_api, name))
    mod.__version__ = "1.8.0+kirag_b200"
    mod.__kirag_b200__ = True
    return mod


def install(force: bool = True) -> types.ModuleType:
    """Install the stand-in as sys.modules['faiss'] (replacing a real faiss only if force)."""
    cur = sys.modules.get("faiss")
    if cur is not None and not force and not getattr(cur, "__kirag_b200__", False):
        return cur
    mod = make_module()
    sys.modules["faiss"] = mod
    return mod


install()
