"""ctypes binding of libb2ip.so (C ABI: include/b2ip.h).

There is deliberately no fallback: if the shared library is missing or no B200 is visible the
import of the library / creation of an engine raises, it never degrades to a CPU path.
"""
from __future__ import annotations

import ctypes
import os

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG_ROOT, "lib", "libb2ip.so")

B2IP_OK = 0
B2IP_F32, B2IP_F16, B2IP_BF16 = 0, 1, 2
STORE_F32, STORE_F16, STORE_BF16 = 0, 1, 2
MEM_HOST, MEM_DEVICE = 0, 1
MODE_AUTO, MODE_TENSOR, MODE_EXACT = 0, 1, 2
MAX_K = 2048

# every symbol include/b2ip.h declares (tests check the .so exports all of them)
SYMBOLS = (
    "b2ip_create", "b2ip_create_ex", "b2ip_destroy", "b2ip_set_stream", "b2ip_set_option", "b2ip_reserve", "b2ip_add", "b2ip_ntotal",
    "b2ip_dim", "b2ip_set_row_offset", "b2ip_set_row_segments", "b2ip_search", "b2ip_search_ex", "b2ip_search_filtered", "b2ip_range_search", "b2ip_range_fetch", "b2ip_search_exchange", "b2ip_enable_peer_access", "b2ip_group_create", "b2ip_group_destroy", "b2ip_group_search", "b2ip_group_last_error",
    "b2ip_merge_topk", "b2ip_merge_topk_strided", "b2ip_export_rows",
    "b2ip_copy_to_device", "b2ip_copy_to_host", "b2ip_stats", "b2ip_last_error", "b2ip_debug_coarse_scores", "b2ip_debug_plan_bootstrap", "b2ip_version",
)


class Stats(ctypes.Structure):
    _fields_ = [
        ("nq", ctypes.c_int64), ("ntotal", ctypes.c_int64),
        ("k", ctypes.c_int32), ("mode_used", ctypes.c_int32),
        ("coarse_launches", ctypes.c_int32), ("total_launches", ctypes.c_int32),
        ("coarse_ms", ctypes.c_float), ("total_ms", ctypes.c_float),
        ("coarse_flops", ctypes.c_double),
        ("candidates", ctypes.c_int64), ("rescored", ctypes.c_int64),
        ("fallback_queries", ctypes.c_int64),
        ("slabs", ctypes.c_int32), ("query_batches", ctypes.c_int32),
        ("refresh_ms", ctypes.c_float), ("finalize_ms", ctypes.c_float),
        ("max_err_over_eps", ctypes.c_double), ("bound_violations", ctypes.c_int64),
        ("graph_mode", ctypes.c_int32), ("sample_rows", ctypes.c_int32),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


MAX_PEERS = 8
GATHER_ALL, GATHER_OWNER = 0, 1
XF_WORDS = 4              # uint32 flag words per publishing rank (csrc/select_kernels.cuh)


class Exchange(ctypes.Structure):
    """b2ip_exchange_t (include/b2ip.h): peer-mapped gather buffers and flag arrays of one parity."""
    _fields_ = [("world", ctypes.c_int32), ("rank", ctypes.c_int32), ("slot_bytes", ctypes.c_int64),
                ("gather", ctypes.c_void_p * MAX_PEERS), ("flags", ctypes.c_void_p * MAX_PEERS),
                ("gthr", ctypes.c_void_p * MAX_PEERS), ("thr_stride", ctypes.c_int64),
                ("gather_mode", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class B2ipError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libb2ip error {code}: {msg}")
        self.code = code


_lib = None


def load() -> ctypes.CDLL:
    """dlopen libb2ip.so and declare the prototypes.  Raises if it has not been built
    (`python -c "import __graft_entry__ as g; g.build()"` or `make -C czech-contriever_b200/csrc`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA library first "
            "(make -C czech-contriever_b200/csrc). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.b2ip_create.argtypes = [i32, i32, ctypes.POINTER(vp)]
    lib.b2ip_create_ex.argtypes = [i32, i32, i32, ctypes.POINTER(vp)]
    lib.b2ip_destroy.argtypes = [vp]
    lib.b2ip_destroy.restype = None
    lib.b2ip_set_stream.argtypes = [vp, vp]
    lib.b2ip_set_option.argtypes = [vp, ctypes.c_char_p, i64]
    lib.b2ip_reserve.argtypes = [vp, i64]
    lib.b2ip_add.argtypes = [vp, i64, vp, i32, i32]
    lib.b2ip_ntotal.argtypes = [vp]
    lib.b2ip_ntotal.restype = i64
    lib.b2ip_dim.argtypes = [vp]
    lib.b2ip_set_row_offset.argtypes = [vp, i64]
    lib.b2ip_set_row_segments.argtypes = [vp, i32, vp, vp]
    lib.b2ip_search.argtypes = [vp, i64, vp, i32, vp, vp, i32, i32]
    lib.b2ip_search_ex.argtypes = [vp, i64, vp, i32, i32, vp, vp, i32, i32]
    lib.b2ip_search_filtered.argtypes = [vp, i64, vp, i32, i32, vp, i64, vp, vp, i32, i32]
    lib.b2ip_range_search.argtypes = [vp, i64, vp, i32, ctypes.c_float, i32, i32, vp]
    lib.b2ip_range_fetch.argtypes = [vp, vp, vp, i32]
    lib.b2ip_search_exchange.argtypes = [vp, i64, vp, i32, ctypes.POINTER(Exchange), ctypes.c_uint32, vp, vp,
                                         ctypes.POINTER(ctypes.c_int64)]
    lib.b2ip_enable_peer_access.argtypes = [vp, i32]
    lib.b2ip_group_create.argtypes = [i32, ctypes.POINTER(vp), ctypes.POINTER(vp)]
    lib.b2ip_group_create.restype = i32
    lib.b2ip_group_destroy.argtypes = [vp]
    lib.b2ip_group_destroy.restype = None
    lib.b2ip_group_search.argtypes = [vp, i64, vp, i32, i32, vp, vp, ctypes.POINTER(ctypes.c_int64)]
    lib.b2ip_group_search.restype = i32
    lib.b2ip_group_last_error.argtypes = [vp]
    lib.b2ip_group_last_error.restype = ctypes.c_char_p
    lib.b2ip_merge_topk.argtypes = [i32, vp, i64, i32, i32, vp, vp, vp, vp]
    lib.b2ip_merge_topk_strided.argtypes = [i32, vp, i64, i32, i32, vp, vp, i64, i64, vp, vp]
    lib.b2ip_export_rows.argtypes = [vp, i64, i64, vp, i32]
    lib.b2ip_copy_to_device.argtypes = [vp, vp, vp, i64]
    lib.b2ip_copy_to_host.argtypes = [vp, vp, vp, i64]
    lib.b2ip_stats.argtypes = [vp, ctypes.POINTER(Stats)]
    lib.b2ip_last_error.argtypes = [vp]
    lib.b2ip_last_error.restype = ctypes.c_char_p
    lib.b2ip_debug_coarse_scores.argtypes = [vp, i64, vp, i64, i64, vp]
    lib.b2ip_debug_plan_bootstrap.argtypes = [i64, i32, i32, i32, i32, i32, ctypes.POINTER(ctypes.c_int32),
                                              ctypes.POINTER(ctypes.c_int64)]
    lib.b2ip_debug_plan_bootstrap.restype = i32
    lib.b2ip_version.restype = ctypes.c_char_p
    for name in ("b2ip_create", "b2ip_create_ex", "b2ip_set_stream", "b2ip_set_option", "b2ip_reserve", "b2ip_add", "b2ip_dim",
                 "b2ip_set_row_offset", "b2ip_set_row_segments", "b2ip_search", "b2ip_search_ex", "b2ip_search_filtered", "b2ip_range_search", "b2ip_range_fetch", "b2ip_search_exchange", "b2ip_enable_peer_access", "b2ip_merge_topk", "b2ip_merge_topk_strided",
                 "b2ip_export_rows", "b2ip_stats", "b2ip_debug_coarse_scores", "b2ip_copy_to_device",
                 "b2ip_copy_to_host"):
        getattr(lib, name).restype = i32
    _lib = lib
    return lib


_hostmap = None


def load_hostmap():
    """The CPython extension csrc/hostmap.c (`map_ids`: the row -> external id loop of
    reference src/index.py:44-45 in C).  Built next to libb2ip.so by `make -C csrc`."""
    global _hostmap
    if _hostmap is None:
        import glob
        import importlib.util
        hits = sorted(glob.glob(os.path.join(_PKG_ROOT, "lib", "_b2ip_hostmap*.so")))
        if not hits:
            raise ImportError(
                f"{os.path.join(_PKG_ROOT, 'lib')}/_b2ip_hostmap*.so not found: build the native "
                "pieces first (make -C czech-contriever_b200/csrc)")
        spec = importlib.util.spec_from_file_location("_b2ip_hostmap", hits[-1])
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _hostmap = mod
    return _hostmap


def check(rc: int, handle=None) -> None:
    if rc != B2IP_OK:
        msg = load().b2ip_last_error(handle)
        raise B2ipError(rc, msg.decode() if msg else "")
