"""ctypes binding of include/modulate_b200.h (one entry per exported symbol).

The shared library is the product; this module only loads it.  If it is missing it is built
with nvcc (``modulate_b200.build``); if that fails the import raises -- there is no Python or
CPU fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes
import os

from . import build as _build

# MODULATE_B200_LIB selects an alternative build of the same library (kernel tuning variants)
_LIB_PATH = os.environ.get("MODULATE_B200_LIB") or _build.LIB


class ModDesc(ctypes.Structure):
    """``mod_desc`` (24 bytes): {src_off u64, dst_off u64, len u32, key i32}."""
    _fields_ = [("src_off", ctypes.c_uint64), ("dst_off", ctypes.c_uint64),
                ("len", ctypes.c_uint32), ("key", ctypes.c_int32)]


assert ctypes.sizeof(ModDesc) == 24

# symbol -> (restype, argtypes); must list EVERY function include/modulate_b200.h declares
# (tests/test_abi_symbols.py parses the header and checks this table and the .so against it).
SIGNATURES = {
    "mod_abi_version": (ctypes.c_int, []),
    "mod_device_count": (ctypes.c_int, []),
    "mod_init": (ctypes.c_int, [ctypes.c_int]),
    "mod_current_device": (ctypes.c_int, []),
    "mod_is_device_pointer": (ctypes.c_int, [ctypes.c_void_p]),
    "mod_shutdown": (None, []),
    "mod_last_error": (ctypes.c_char_p, []),
    "mod_launch_count": (ctypes.c_uint64, []),
    "mod_host_alloc": (ctypes.c_void_p, [ctypes.c_uint64]),
    "mod_host_free": (ctypes.c_int, [ctypes.c_void_p]),
    "mod_device_alloc": (ctypes.c_void_p, [ctypes.c_uint64]),
    "mod_device_free": (ctypes.c_int, [ctypes.c_void_p]),
    "mod_memcpy_h2d": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]),
    "mod_memcpy_d2h": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]),
    "mod_stream_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "mod_stream_create": (ctypes.c_void_p, []),
    "mod_stream_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "mod_cycle": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32]),
    "mod_cycle_sharded": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32, ctypes.c_uint64]),
    "mod_cycle_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32,
                                        ctypes.c_void_p]),
    "mod_key_jump": (ctypes.c_int32, [ctypes.c_int32, ctypes.c_uint64]),
    "mod_plan_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64,
                                       ctypes.c_uint32, ctypes.POINTER(ctypes.c_void_p)]),
    "mod_plan_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "mod_plan_payload_bytes": (ctypes.c_uint64, [ctypes.c_void_p]),
    "mod_plan_num_tiles": (ctypes.c_uint64, [ctypes.c_void_p]),
    "mod_plan_run": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "mod_plan_tile_range": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64,
                                           ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]),
    "mod_plan_run_window": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p,
                                           ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                           ctypes.c_uint64, ctypes.c_void_p]),
    "mod_cycle_batch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                       ctypes.c_void_p, ctypes.c_uint64]),
    "mod_cycle_batch_sharded": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                               ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64]),
    "mod_plan_find": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
    "mod_plan_find_window": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p,
                                            ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint32,
                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p,
                                            ctypes.c_void_p]),
    "mod_find_batch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p,
                                      ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]),
    "mod_plan_find_masked": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32,
                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
    "mod_plan_find_masked_window": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p,
                                                   ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p,
                                                   ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                                   ctypes.c_void_p, ctypes.c_void_p]),
    "mod_find_masked_batch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p,
                                             ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64,
                                             ctypes.c_void_p]),
    "mod_pattern_set_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.POINTER(ctypes.c_void_p)]),
    "mod_pattern_set_create_nocase": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32,
                                                     ctypes.POINTER(ctypes.c_void_p)]),
    "mod_pattern_set_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "mod_plan_find_set": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
    "mod_plan_find_set_window": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64,
                                                ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
    "mod_find_set_batch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_uint64, ctypes.c_void_p]),
    # include/modulate_ark.h: C binding of the archive-level facade
    "mod_ark_unpack": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int32]),
    "mod_ark_pack": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int,
                                    ctypes.c_int, ctypes.c_int, ctypes.c_int32]),
    "mod_ark_find": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_int32,
                                    ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]),
    "mod_ark_find_set": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32,
                                        ctypes.c_int32, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.POINTER(ctypes.c_uint64), ctypes.c_void_p]),
    "mod_ark_find_masked": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint32,
                                           ctypes.c_int32, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.POINTER(ctypes.c_uint64)]),
    "mod_ark_find_set_nocase": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32,
                                               ctypes.c_int32, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                               ctypes.POINTER(ctypes.c_uint64), ctypes.c_void_p]),
    "mod_dta_set_int": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int32]),
    "mod_shard_range": (ctypes.c_int, [ctypes.c_uint64, ctypes.c_int, ctypes.c_int,
                                       ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]),
    "mod_shard_descs": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_void_p, ctypes.c_uint64]),
    "mod_group_descs": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]),
}

_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load() -> ctypes.CDLL:
    """Load (building first if needed) libmodulate_b200.so and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if _LIB_PATH == _build.LIB and _build.stale(_LIB_PATH):
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this box: a prebuilt .so is still acceptable
            if not os.path.exists(_LIB_PATH):
                raise ImportError(
                    "modulate_b200: libmodulate_b200.so is missing and could not be built "
                    f"({exc}); there is no CPU fallback") from exc
    L = ctypes.CDLL(_LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(L, name)
        except AttributeError:
            if _LIB_PATH != _build.LIB:  # an older tuning variant selected through MODULATE_B200_LIB
                continue
            raise  # header / library mismatch in the product build: fail loudly
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = L
    return L


class ModError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"modulate_b200 error {code}: {message}")
        self.code = code


def check(rc: int) -> int:
    if rc < 0:
        raise ModError(rc, load().mod_last_error().decode("utf-8", "replace"))
    return rc
