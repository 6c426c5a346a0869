"""oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes handles onto the CPU checkers:

* ``liboracle.so``         -- plain-C restatement (``cycle_oracle.c``) of
  ``CEncryptionCycler::Cycle`` (reference ``CEncryptionCycler.cpp:4-25``) and of the
  gather/scatter data movement of ``CArk::ExtractFiles`` / ``CArk::BuildArk``
  (``CArk.cpp:494``, ``:807-811``).
* ``_ref/libcycle_ref.so`` -- the UNMODIFIED reference ``CEncryptionCycler.cpp`` compiled by
  ``oracle/Makefile`` (present when built in the dev container; travels to the GPU box).
* ``_ref/libark_ref.so``   -- the reference's own ``CArk.cpp`` / ``CDtaFile.cpp`` / ``Utils.cpp`` behind
  ``ref_ark/ark_ref_shim.cpp`` (Win32 stand-ins in ``ref_ark/``); used only by
  ``tests/golden/make_ark_golden.py`` to write the HDR / ARK / DTB fixtures under ``tests/golden/``.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package.  Parity status: pinned (see
``cycle_oracle.c`` header).
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")
_REF = os.path.join(_HERE, "_ref", "libcycle_ref.so")
_ARK_REF = os.path.join(_HERE, "_ref", "libark_ref.so")

M = 0x7FFFFFFF
A = 16807


class Desc(ctypes.Structure):
    """Same 24-byte layout as ``mod_desc`` in include/modulate_b200.h."""
    _fields_ = [("src_off", ctypes.c_uint64), ("dst_off", ctypes.c_uint64),
                ("len", ctypes.c_uint32), ("key", ctypes.c_int32)]


DESC_DTYPE = np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("len", "<u4"), ("key", "<i4")])


class RefPart(ctypes.Structure):
    _fields_ = [("off", ctypes.c_uint64), ("len", ctypes.c_uint32), ("key", ctypes.c_int32)]


PART_DTYPE = np.dtype([("off", "<u8"), ("len", "<u4"), ("key", "<i4")])


def build(force: bool = False) -> None:
    """Compile liboracle.so and (when /root/reference is present) _ref/libcycle_ref.so."""
    # staleness by content, not modification time: a copied tree keeps its build and is never written to
    with open(os.path.join(_HERE, "cycle_oracle.c"), "rb") as f:
        fp = hashlib.sha256(f.read()).hexdigest()
    stamp = _LIB + ".stamp"
    if force or not os.path.exists(_LIB) or not os.path.exists(stamp) or open(stamp).read().strip() != fp:
        subprocess.check_call(["make", "-B", "-C", _HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
        with open(stamp, "w") as f:
            f.write(fp)
    if os.path.exists("/root/reference/Modulate/CEncryptionCycler.cpp") and \
            (force or not os.path.exists(_REF)):
        subprocess.check_call(["make", "-C", _HERE, "ref"], stdout=subprocess.DEVNULL)
    # the reference's own CArk / CDtaFile (fixture generator tests/golden/make_ark_golden.py only)
    if os.path.exists("/root/reference/Modulate/CArk.cpp") and (force or not os.path.exists(_ARK_REF)):
        subprocess.check_call(["make", "-C", _HERE, "ark_ref"], stdout=subprocess.DEVNULL)


_lib = None
_ref = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB)
        L.oracle_cycle_key.argtypes = [ctypes.c_int32]
        L.oracle_cycle_key.restype = ctypes.c_int32
        L.oracle_cycle.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int32]
        L.oracle_cycle.restype = None
        L.oracle_pow_a.argtypes = [ctypes.c_uint64]
        L.oracle_pow_a.restype = ctypes.c_uint32
        L.oracle_key_residue.argtypes = [ctypes.c_int32]
        L.oracle_key_residue.restype = ctypes.c_uint32
        L.oracle_key_jump.argtypes = [ctypes.c_int32, ctypes.c_uint64]
        L.oracle_key_jump.restype = ctypes.c_int32
        L.oracle_keystream_byte.argtypes = [ctypes.c_int32, ctypes.c_uint64]
        L.oracle_keystream_byte.restype = ctypes.c_ubyte
        L.oracle_cycle_at.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32, ctypes.c_uint64]
        L.oracle_cycle_at.restype = None
        L.oracle_cycle_batch.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]
        L.oracle_cycle_batch.restype = None
        L.oracle_fnv1a64.argtypes = [ctypes.c_void_p, ctypes.c_uint64]
        L.oracle_fnv1a64.restype = ctypes.c_uint64
        _lib = L
    return _lib


def have_ref() -> bool:
    build()
    return os.path.exists(_REF)


def ref() -> ctypes.CDLL:
    """The unmodified reference cipher (raises if it was never built)."""
    global _ref
    if _ref is None:
        build()
        if not os.path.exists(_REF):
            raise FileNotFoundError("oracle/_ref/libcycle_ref.so not built (reference sources absent)")
        R = ctypes.CDLL(_REF)
        R.ref_cycle.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.c_int]
        R.ref_cycle.restype = None
        R.ref_cycle_parts.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int]
        R.ref_cycle_parts.restype = None
        R.ref_hardware_threads.argtypes = []
        R.ref_hardware_threads.restype = ctypes.c_int
        _ref = R
    return _ref


def _i32(key: int) -> int:
    key &= 0xFFFFFFFF
    return key - (1 << 32) if key & 0x80000000 else key


def _ptr(a: np.ndarray) -> int:
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data


def cycle(data: np.ndarray, key: int, *, use_ref: bool = False) -> np.ndarray:
    """Return Cycle(data, len(data), key) as a new uint8 array (input untouched)."""
    out = np.ascontiguousarray(data, dtype=np.uint8).copy()
    assert out.size < (1 << 32)
    if out.size:
        (ref().ref_cycle if use_ref else lib().oracle_cycle)(_ptr(out), out.size, _i32(key))
    return out


def cycle_at(data: np.ndarray, key: int, pos: int) -> np.ndarray:
    """Cycle a window that starts `pos` bytes into a longer stream (closed-form jump)."""
    out = np.ascontiguousarray(data, dtype=np.uint8).copy()
    if out.size:
        lib().oracle_cycle_at(_ptr(out), out.size, _i32(key), pos)
    return out


def keystream(key: int, n: int, *, use_ref: bool = False) -> np.ndarray:
    return cycle(np.zeros(n, dtype=np.uint8), key, use_ref=use_ref)


def key_jump(key: int, pos: int) -> int:
    return lib().oracle_key_jump(_i32(key), pos)


def key_residue(key: int) -> int:
    return lib().oracle_key_residue(_i32(key))


def pow_a(e: int) -> int:
    return lib().oracle_pow_a(e)


def cycle_batch(descs: np.ndarray, src: np.ndarray, dst: np.ndarray) -> np.ndarray:
    """Apply every descriptor (gather/scatter + per-entry Cycle) into `dst` in place."""
    descs = np.ascontiguousarray(descs, dtype=DESC_DTYPE)
    assert dst.dtype == np.uint8 and src.dtype == np.uint8
    if len(descs):
        assert int((descs["src_off"] + descs["len"]).max()) <= src.size
        assert int((descs["dst_off"] + descs["len"]).max()) <= dst.size
    lib().oracle_cycle_batch(_ptr(descs), len(descs), _ptr(src), _ptr(dst))
    return dst


def fnv1a64(data: np.ndarray) -> int:
    data = np.ascontiguousarray(data, dtype=np.uint8)
    return lib().oracle_fnv1a64(_ptr(data), data.size)


def ref_cycle_parts(buf: np.ndarray, parts: np.ndarray, threads: int) -> None:
    """In place: one unmodified-reference Cycle() per (off, len, key) part over `threads` threads."""
    parts = np.ascontiguousarray(parts, dtype=PART_DTYPE)
    ref().ref_cycle_parts(_ptr(buf), _ptr(parts), len(parts), threads)
