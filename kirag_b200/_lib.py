"""ctypes binding of the C ABI declared in include/kirag_b200.h.

There is no Python/CPU implementation behind these symbols: if the shared
library is missing the import fails, and if no B200 is visible every call
raises.  (The oracle under /oracle is test infrastructure and is never
imported from here.)
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
# KIRAG_B200_LIB: load another build of the SAME ABI (same-box A/B of kernel changes); default: the in-tree library
LIB_PATH = os.environ.get("KIRAG_B200_LIB") or os.path.join(HERE, "libkirag_b200.so")

# constants mirrored from the header
ABI_VERSION = 11
INDEX_HOST_MASTER = 1
INDEX_ID_MAP = 16
METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
PATH_AUTO, PATH_EXACT, PATH_FAST = 0, 1, 2
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
MASK_I64, MASK_I32, MASK_U8 = 0, 1, 2
POOL_MEAN, POOL_CLS = 0, 1


class SearchStats(ctypes.Structure):
    _fields_ = [
        ("nq", c_int64),
        ("n_fast", c_int64),
        ("n_exact", c_int64),
        ("n_cert_fail", c_int64),
        ("n_overflow", c_int64),
        ("levels", c_int32),
        ("path", c_int32),
        ("kernel_launches", c_int64),
        ("n_rescan", c_int64),
        ("n_retry", c_int64),
    ]

    def as_dict(self):
        return {name: int(getattr(self, name)) for name, _ in self._fields_}


class KiragError(RuntimeError):
    """A C-ABI call returned a non-zero status (CUDA failure, bad handle...)."""


# every exported symbol: name -> (restype, argtypes).  tests/test_abi.py checks
# this table against include/kirag_b200.h and against the built library.
SIGNATURES = {
    "kirag_abi_version": (c_int, []),
    "kirag_last_error": (c_char_p, []),
    "kirag_device_count": (c_int, []),
    "kirag_profile_enable": (c_int, [c_int]),
    "kirag_profile_read": (c_int, [POINTER(ctypes.c_double), POINTER(c_int64), POINTER(ctypes.c_double)]),
    "kirag_profile_read_launches": (c_int, [POINTER(ctypes.c_double), POINTER(ctypes.c_double), c_int64]),
    "kirag_profile_read_timeline": (c_int, [POINTER(c_int), POINTER(ctypes.c_double), c_int64]),
    "kirag_index_create": (c_int, [c_int, c_int, c_int, POINTER(c_void_p)]),
    "kirag_index_create_ex": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_void_p)]),
    "kirag_index_create_multi": (c_int, [c_int, c_int, POINTER(c_int), c_int, c_int, POINTER(c_void_p)]),
    "kirag_index_load_multi": (c_int, [c_char_p, POINTER(c_int), c_int, c_int, POINTER(c_void_p)]),
    "kirag_index_shards": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int64), c_int]),
    "kirag_debug_stripe_map": (c_int, [c_int, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "kirag_debug_stripe_rows": (c_int, [c_int64, c_int, POINTER(c_int64)]),
    "kirag_index_destroy": (c_int, [c_void_p]),
    "kirag_index_reserve": (c_int, [c_void_p, c_int64]),
    "kirag_index_add": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "kirag_index_add_with_ids": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "kirag_index_flags": (c_int, [c_void_p]),
    "kirag_index_remove_ids_ex": (c_int, [c_void_p, c_void_p, c_int64, c_int, POINTER(c_int64), c_void_p]),
    "kirag_index_id_map": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int, c_void_p]),
    "kirag_index_remove_ids": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_int64), c_void_p]),
    "kirag_index_remove_range": (c_int, [c_void_p, c_int64, c_int64, POINTER(c_int64), c_void_p]),
    "kirag_debug_remove_plan": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_int64, c_void_p, c_void_p,
                                        c_int64]),
    "kirag_index_ntotal": (c_int64, [c_void_p]),
    "kirag_index_dim": (c_int, [c_void_p]),
    "kirag_index_search": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_int64, c_void_p]),
    "kirag_index_search_ex": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_int64, c_int,
                                      POINTER(SearchStats), c_void_p]),
    "kirag_index_range_search": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_int, c_int64, c_int, c_void_p,
                                         POINTER(SearchStats), c_void_p]),
    "kirag_index_range_fetch": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "kirag_index_search_async": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "kirag_index_search_finish": (c_int, [c_void_p, POINTER(SearchStats), POINTER(c_int64)]),
    "kirag_index_search_flags": (c_int, [c_void_p, POINTER(c_void_p)]),
    "kirag_index_search_rearm": (c_int, [c_void_p, c_void_p]),
    "kirag_index_state_token": (c_int, [c_void_p, POINTER(ctypes.c_uint64)]),
    "kirag_index_reconstruct": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int, c_void_p]),
    "kirag_index_save": (c_int, [c_void_p, c_char_p]),
    "kirag_index_load": (c_int, [c_char_p, c_int, POINTER(c_void_p)]),
    "kirag_index_load_ex": (c_int, [c_char_p, c_int, c_int, POINTER(c_void_p)]),
    "kirag_index_storage_bytes": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "kirag_index_device_ptrs": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p)]),
    "kirag_debug_level_schedule": (c_int, [c_int64, c_int64, c_int, c_int, POINTER(c_int64), c_int, POINTER(c_int),
                                           POINTER(c_int)]),
    "kirag_index_debug_scores": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "kirag_merge_topk": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "kirag_exchange_create": (c_int, [c_int, c_int, c_int, c_int64, c_int, POINTER(c_void_p)]),
    "kirag_exchange_destroy": (c_int, [c_void_p]),
    "kirag_exchange_handle_bytes": (c_int, []),
    "kirag_exchange_export": (c_int, [c_void_p, c_void_p]),
    "kirag_exchange_connect": (c_int, [c_void_p, c_void_p]),
    "kirag_exchange_connect_ptrs": (c_int, [c_void_p, POINTER(c_void_p)]),
    "kirag_exchange_buffer": (c_void_p, [c_void_p]),
    "kirag_exchange_merge_topk": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "kirag_exchange_merge_topk_flags": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p,
                                                c_void_p]),
    "kirag_exchange_last_any_flag": (c_int, [c_void_p]),
    "kirag_topk_ip": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                              c_void_p]),
    "kirag_topk_ip_release": (c_int, []),
    "kirag_pool_normalize": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_int64,
                                     c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "kirag_pool_normalize_fwd_saved": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                               c_int64, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "kirag_pool_normalize_typed": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                           c_int64, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "kirag_pool_normalize_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                              c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load libkirag_b200.so (once).  Raises ImportError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m kirag_b200._build` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "kirag_b200 has no CPU or pure-Python fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = restype
        fn.argtypes = argtypes
    got = lib.kirag_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libkirag_b200.so has ABI version {got}, the Python host expects {ABI_VERSION}")
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().kirag_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int, what: str) -> None:
    if status != 0:
        raise KiragError(f"{what}: {last_error()}")


def default_device() -> int:
    """KIRAG_DEVICE, else torch's current CUDA device if torch is already in use, else 0."""
    env = os.environ.get("KIRAG_DEVICE")
    if env:
        return int(env)
    import sys

    torch = sys.modules.get("torch")
    if torch is not None:
        try:
            if torch.cuda.is_available():
                return int(torch.cuda.current_device())
        except Exception:
            pass
    return 0
