"""ctypes binding of ``include/rpk.h`` -- the same C-ABI a cgo binding would call (INTEGRATION.md).

There is no CPU implementation behind this module: if ``librpk.so`` is missing, or no sm_100 GPU is
present, construction fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "librpk.so")

RPK_OK, RPK_EINVAL, RPK_ECUDA, RPK_ENOMEM, RPK_ESTATE, RPK_ENODEV = 0, -1, -2, -3, -4, -5
ERR_NAMES = {0: "RPK_OK", -1: "RPK_EINVAL", -2: "RPK_ECUDA", -3: "RPK_ENOMEM", -4: "RPK_ESTATE", -5: "RPK_ENODEV"}

# every symbol include/rpk.h declares (tests assert the library exports all of them)
SYMBOLS = [
    "rpk_create", "rpk_destroy", "rpk_last_error", "rpk_abi_version", "rpk_host_alloc", "rpk_host_free",
    "rpk_offers_upload", "rpk_select", "rpk_select_device", "rpk_select_device_gather", "rpk_best_device_ptr",
    "rpk_status_diff", "rpk_status_seed", "rpk_status_reset", "rpk_status_diff_device", "rpk_stats_get",
    "rpk_launch_count", "rpk_ipc_alloc", "rpk_ipc_open", "rpk_ipc_close", "rpk_ipc_free", "rpk_peer_fence",
    "rpk_peer_bind", "rpk_peer_wait", "rpk_peer_inline_wait", "rpk_status_diff_codes", "rpk_status_seed_slots", "rpk_tick",
    "rpk_status_diff_device_codes", "rpk_xchg_bytes", "rpk_status_diff_device_gather",
    "rpk_offer_sets_upload", "rpk_select_sets", "rpk_select_sets_device",
]

RPK_MAX_OFFER_SETS = 256
RPK_SET_ALL = 0xFFFF


class RpkStats(C.Structure):
    _fields_ = [
        ("select_calls", C.c_uint64), ("offer_scores", C.c_uint64), ("status_calls", C.c_uint64),
        ("status_records", C.c_uint64), ("last_select_kernel_ms", C.c_float), ("last_select_total_ms", C.c_float),
        ("last_status_kernel_ms", C.c_float), ("last_status_total_ms", C.c_float),
        ("select_kernel_kind", C.c_uint32), ("n_gpus", C.c_uint32), ("distinct_mem", C.c_uint32),
        ("distinct_vcpu", C.c_uint32), ("distinct_ram", C.c_uint32), ("packed_bits", C.c_uint32),
    ]


class RpkError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


_lib = None


def load():
    """Load ``librpk.so`` (built in-tree by ``__graft_entry__.build()`` / ``make -C csrc``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `make -C {os.path.join(_PKG, 'csrc')}` "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u32, i32p, f64p, u8p, u32p, u64p = (C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p)
    L.rpk_create.restype = C.c_int
    L.rpk_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(vp)]
    L.rpk_destroy.restype = None
    L.rpk_destroy.argtypes = [vp]
    L.rpk_last_error.restype = C.c_char_p
    L.rpk_last_error.argtypes = [vp]
    L.rpk_abi_version.restype = C.c_int
    L.rpk_host_alloc.restype = vp
    L.rpk_host_alloc.argtypes = [C.c_size_t]
    L.rpk_host_free.restype = None
    L.rpk_host_free.argtypes = [vp]
    L.rpk_offers_upload.restype = C.c_int
    L.rpk_offers_upload.argtypes = [vp, u32, i32p, i32p, i32p, f64p, f64p, u8p]
    L.rpk_select.restype = C.c_int
    L.rpk_select.argtypes = [vp, u32, i32p, i32p, i32p, f64p, u8p, i32p, i32p]
    L.rpk_select_device.restype = C.c_int
    L.rpk_select_device.argtypes = [vp, C.c_int, u32, i32p, i32p, i32p, f64p, u8p, i32p, i32p, vp]
    L.rpk_select_device_gather.restype = C.c_int
    L.rpk_select_device_gather.argtypes = [vp, C.c_int, u32, i32p, i32p, i32p, f64p, u8p, C.c_int, C.POINTER(vp), u32,
                                           i32p, vp]
    L.rpk_offer_sets_upload.restype = C.c_int
    L.rpk_offer_sets_upload.argtypes = [vp, u32, u32, u32p]
    L.rpk_select_sets.restype = C.c_int
    L.rpk_select_sets.argtypes = [vp, u32, i32p, i32p, i32p, f64p, u8p, vp, i32p, i32p]
    L.rpk_select_sets_device.restype = C.c_int
    L.rpk_select_sets_device.argtypes = [vp, C.c_int, u32, i32p, i32p, i32p, f64p, u8p, vp, i32p, i32p, vp]
    L.rpk_best_device_ptr.restype = vp
    L.rpk_best_device_ptr.argtypes = [vp, C.c_int]
    L.rpk_status_diff.restype = C.c_int
    L.rpk_status_diff.argtypes = [vp, u32, u8p, u32, u32p, u32p, u64p]
    L.rpk_status_seed.restype = C.c_int
    L.rpk_status_seed.argtypes = [vp, u32, u8p, u32]
    L.rpk_status_reset.restype = C.c_int
    L.rpk_status_reset.argtypes = [vp, u32]
    L.rpk_status_diff_device.restype = C.c_int
    L.rpk_status_diff_device.argtypes = [vp, C.c_int, u32, u8p, u32, u64p, u32p, u32p, vp]
    L.rpk_status_diff_codes.restype = C.c_int
    L.rpk_status_diff_codes.argtypes = [vp, u32, u8p, u32, u32p, vp, u32p, u64p]
    L.rpk_status_seed_slots.restype = C.c_int
    L.rpk_status_seed_slots.argtypes = [vp, u32, u32p, u8p, u32]
    L.rpk_tick.restype = C.c_int
    L.rpk_tick.argtypes = [vp, u32, i32p, i32p, i32p, f64p, u8p, i32p, i32p, u32, u8p, u32, u32p, vp, u32p]
    L.rpk_status_diff_device_codes.restype = C.c_int
    L.rpk_status_diff_device_codes.argtypes = [vp, C.c_int, u32, u8p, u32, u64p, u32p, vp, u32p, vp]
    L.rpk_xchg_bytes.restype = C.c_size_t
    L.rpk_xchg_bytes.argtypes = [C.c_int, u32]
    L.rpk_status_diff_device_gather.restype = C.c_int
    L.rpk_status_diff_device_gather.argtypes = [vp, C.c_int, u32, u8p, u32, u64p, u32, C.c_int, C.POINTER(vp), u32, C.c_int, u32p, vp]
    L.rpk_stats_get.restype = C.c_int
    L.rpk_stats_get.argtypes = [vp, C.POINTER(RpkStats)]
    for name in ("rpk_ipc_alloc", "rpk_ipc_open", "rpk_ipc_close", "rpk_ipc_free"):
        getattr(L, name).restype = C.c_int
    L.rpk_ipc_alloc.argtypes = [vp, C.c_int, C.c_size_t, C.POINTER(vp), C.c_char_p]
    L.rpk_ipc_open.argtypes = [vp, C.c_int, C.c_char_p, C.POINTER(vp)]
    L.rpk_ipc_close.argtypes = [vp, C.c_int, vp]
    L.rpk_ipc_free.argtypes = [vp, C.c_int, vp]
    L.rpk_peer_fence.restype = C.c_int
    L.rpk_peer_fence.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp), C.c_int, C.c_uint32, vp]
    L.rpk_peer_bind.restype = C.c_int
    L.rpk_peer_bind.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp), C.c_int]
    L.rpk_peer_inline_wait.restype = C.c_int
    L.rpk_peer_inline_wait.argtypes = [vp, C.c_int, C.c_int]
    L.rpk_peer_wait.restype = C.c_int
    L.rpk_peer_wait.argtypes = [vp, C.c_int, C.c_uint, vp]
    L.rpk_launch_count.restype = C.c_uint64
    L.rpk_launch_count.argtypes = [vp]
    _lib = L
    return L
