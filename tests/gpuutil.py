"""Helpers of the GPU tests, built on the C ABI only (no torch needed): device memory, search result buffers, and
sources whose entries decipher to given bytes."""
from __future__ import annotations

import ctypes
import functools
import os
import tempfile

import numpy as np

import kernel_model as km
import modulate_b200 as mb
import oracle
import synth
from modulate_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "modulate_b200", "bin", "modulate")
EDGE_KEYS = [0, 0x7FFFFFFF, -0x80000000, -1, 1]


class DeviceBuffer:
    def __init__(self, nbytes: int):
        self.lib = _abi.load()
        self.nbytes = int(nbytes)
        self.ptr = self.lib.mod_device_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError(self.lib.mod_last_error().decode())

    @classmethod
    def from_numpy(cls, a: np.ndarray) -> "DeviceBuffer":
        a = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        b = cls(a.nbytes)
        b.upload(a)
        return b

    def upload(self, a: np.ndarray, offset: int = 0) -> None:
        a = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        assert offset + a.nbytes <= self.nbytes
        if a.nbytes:
            _abi.check(self.lib.mod_memcpy_h2d(self.ptr + offset, a.ctypes.data, a.nbytes, None))
            _abi.check(self.lib.mod_stream_sync(None))

    def download(self, offset: int = 0, nbytes: int | None = None) -> np.ndarray:
        n = self.nbytes - offset if nbytes is None else nbytes
        out = np.empty(n, dtype=np.uint8)
        if n:
            _abi.check(self.lib.mod_memcpy_d2h(out.ctypes.data, self.ptr + offset, n, None))
            _abi.check(self.lib.mod_stream_sync(None))
        return out

    def fill_payload(self, seed_offset: int = 0, chunk: int = 64 << 20) -> None:
        """Fill with the synthetic stream synth.payload(seed_offset + i)."""
        import synth
        for o in range(0, self.nbytes, chunk):
            n = min(chunk, self.nbytes - o)
            self.upload(synth.payload(seed_offset + o, n), o)

    def free(self) -> None:
        if self.ptr:
            self.lib.mod_device_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def sync() -> None:
    _abi.check(_abi.load().mod_stream_sync(None))


def aligned_buffer(a: np.ndarray) -> DeviceBuffer:
    b = DeviceBuffer.from_numpy(a)
    assert b.ptr % 16 == 0  # the model's addresses are offsets from 16-byte aligned bases
    return b


class Results:
    """total (u64), counts (u32 per descriptor) and a list of `cap` matches in one device buffer; the list is
    16-byte aligned, as mod_match stores need."""

    def __init__(self, n: int, cap: int):
        self.n, self.cap = n, cap
        self.list_at = (16 + 4 * n + 15) & ~15
        self.buf = DeviceBuffer(self.list_at + 8 * max(cap, 1))
        self.buf.upload(np.zeros(self.buf.nbytes, np.uint8))
        self.total, self.counts, self.matches = self.buf.ptr, self.buf.ptr + 16, self.buf.ptr + self.list_at

    def read(self):
        raw = self.buf.download()
        total = int(raw[:8].view(np.uint64)[0])
        counts = raw[16:16 + 4 * self.n].view(np.uint32).copy()
        m = raw[self.list_at:].view(mb.MATCH_DTYPE)[:min(total, self.cap)]
        return total, counts, [(int(a), int(b)) for a, b in zip(m["desc"], m["pos"])]


def as_list(matches):
    """mb.SET_MATCH_DTYPE records -> [(desc, pos, pattern)]."""
    return [(int(a), int(b), int(c)) for a, b, c in zip(matches["desc"], matches["pos"], matches["pattern"])]


def build_source(plain_entries, keys, phase):
    """Byte-packed source whose entries decipher to `plain_entries` (Cycle is its own inverse)."""
    sizes = np.array([e.size for e in plain_entries], np.int64)
    src_off = synth.packed_offsets(sizes) + phase
    src = np.zeros(int(phase + sizes.sum() + 64), np.uint8)
    for e, o, k in zip(plain_entries, src_off, keys):
        src[o:o + e.size] = oracle.cycle(e, k)
    return mb.make_descs(src_off, src_off, sizes, keys), src


# ---- the search cases of tests/kernel_model.py ----------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def cases_by_cell():
    return {c.cell: c for c in km.find_cases()}


def decipher_entries(descs, image):
    """The deciphered bytes of a model case's (src_off, len, key) descriptors."""
    return [oracle.cycle(image[so:so + ln], key) for so, ln, key in descs]


def model_descs(descs):
    """A model case's (src_off, len, key) descriptors as mod_desc records, in place (dst_off == src_off)."""
    so, ln, key = zip(*descs)
    return mb.make_descs(list(so), list(so), list(ln), [k & 0xFFFFFFFF for k in key])


def shm_dir(tmp_path):
    """A fresh directory in /dev/shm when it is writable (large archives), else under tmp_path."""
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else str(tmp_path)
    return tempfile.mkdtemp(prefix="modfind", dir=base)
