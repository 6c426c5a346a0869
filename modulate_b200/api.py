"""Host-side mirror of the reference's interface for the hot path, over the C ABI."""
from __future__ import annotations

import ctypes
from typing import Any, Optional, Tuple

import numpy as np

from . import _abi
from ._abi import ModError

# numpy view of ``mod_desc``
DESC_DTYPE = np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("len", "<u4"), ("key", "<i4")])
assert DESC_DTYPE.itemsize == 24


def _i32(key: int) -> int:
    """Reinterpret any 32-bit pattern as the ``int`` the reference's Cycle takes (CArk.cpp:339
    passes the ``unsigned int`` platform key to an ``int`` parameter)."""
    key = int(key) & 0xFFFFFFFF
    return key - (1 << 32) if key & 0x80000000 else key


def _buffer_info(buf: Any) -> Tuple[int, int, bool]:
    """-> (address, nbytes, is_cuda) for bytearray / memoryview / numpy / torch / raw int address."""
    if isinstance(buf, int):
        return buf, -1, False
    if hasattr(buf, "data_ptr") and hasattr(buf, "is_cuda"):  # torch.Tensor, without importing torch
        if not buf.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return buf.data_ptr(), buf.numel() * buf.element_size(), bool(buf.is_cuda)
    if isinstance(buf, np.ndarray):
        if not buf.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        if not buf.flags["WRITEABLE"]:
            raise ValueError("array must be writeable (Cycle works in place)")
        return buf.ctypes.data, buf.nbytes, False
    if isinstance(buf, (bytearray, memoryview)):
        mv = memoryview(buf)
        if mv.readonly:
            raise ValueError("buffer must be writeable (Cycle works in place)")
        c = (ctypes.c_char * mv.nbytes).from_buffer(mv)
        return ctypes.addressof(c), mv.nbytes, False
    raise TypeError(f"unsupported buffer type {type(buf)!r}")


def init(device: int = -1) -> None:
    _abi.check(_abi.load().mod_init(device))


def device_count() -> int:
    return _abi.check(_abi.load().mod_device_count())


def launch_count() -> int:
    return int(_abi.load().mod_launch_count())


def key_jump(key: int, pos: int) -> int:
    """Key whose stream equals `key`'s stream from byte `pos` on (O(log pos) jump-ahead)."""
    return int(_abi.load().mod_key_jump(_i32(key), int(pos)))


def cycle(buf: Any, size: Optional[int], key: int) -> None:
    """``CEncryptionCycler::Cycle`` in place on a host or device buffer (synchronous)."""
    addr, nbytes, _ = _buffer_info(buf)
    if size is None:
        size = nbytes
    if nbytes >= 0 and size > nbytes:
        raise ValueError(f"liDataSize {size} exceeds the {nbytes}-byte buffer")
    _abi.check(_abi.load().mod_cycle(addr, int(size), _i32(key)))


def cycle_sharded(buf: Any, size: Optional[int], key: int, dev_mask: int = 0) -> None:
    """``Cycle`` on a HOST buffer split by offset range over the GPUs ``dev_mask`` selects (0 = all
    visible), one host thread + stream set per device inside this process (synchronous)."""
    addr, nbytes, is_cuda = _buffer_info(buf)
    if is_cuda:
        raise ValueError("cycle_sharded takes a host buffer")
    if size is None:
        size = nbytes
    if nbytes >= 0 and size > nbytes:
        raise ValueError(f"liDataSize {size} exceeds the {nbytes}-byte buffer")
    _abi.check(_abi.load().mod_cycle_sharded(addr, int(size), _i32(key), int(dev_mask)))


def cycle_device(src: Any, dst: Any, size: int, key: int, stream: int = 0) -> None:
    """Asynchronous device-resident Cycle (src may equal dst)."""
    s_addr, s_n, _ = _buffer_info(src)
    d_addr, d_n, _ = _buffer_info(dst)
    if (s_n >= 0 and size > s_n) or (d_n >= 0 and size > d_n):
        raise ValueError("size exceeds a buffer")
    _abi.check(_abi.load().mod_cycle_device(s_addr, d_addr, int(size), _i32(key), stream or None))


class CEncryptionCycler:
    """Same surface as the reference class (``CEncryptionCycler.h:3-10``): stateless, one method."""

    def Cycle(self, lpData: Any, liDataSize: Optional[int], liInitialKey: int) -> None:
        cycle(lpData, liDataSize, liInitialKey)


def make_descs(src_off, dst_off, length, key) -> np.ndarray:
    n = len(src_off)
    d = np.zeros(n, dtype=DESC_DTYPE)
    d["src_off"] = src_off
    d["dst_off"] = dst_off
    d["len"] = length
    d["key"] = np.asarray(key, dtype=np.int64).astype(np.uint32).view(np.int32) \
        if not isinstance(key, np.ndarray) or key.dtype != np.int32 else key
    return d


# numpy view of ``mod_match``: where a pattern starts inside a descriptor's deciphered bytes
MATCH_DTYPE = np.dtype([("desc", "<u4"), ("pos", "<u4")])
MAX_PATTERN = 64


def _pattern(pattern: Any) -> bytes:
    p = bytes(pattern.encode() if isinstance(pattern, str) else pattern)
    if not 1 <= len(p) <= MAX_PATTERN:
        raise ValueError(f"the pattern must be 1 to {MAX_PATTERN} bytes, not {len(p)}")
    return p


def _mask(mask: Any, n: int) -> bytes:
    m = bytes(mask)
    if len(m) != n:
        raise ValueError(f"the mask must have one byte per pattern byte ({n}), not {len(m)}")
    return m


def _fold(p: bytes) -> bytes:
    """ASCII upper case: b'a'..b'z' -> b'A'..b'Z', every other byte itself."""
    return bytes(b - 0x20 if 0x61 <= b <= 0x7A else b for b in p)


def wildcard_pattern(hex_text: str) -> Tuple[bytes, bytes]:
    """(pattern, mask) of hex digit pairs in which any digit may be ``?`` (any nibble; ``??`` any byte), whitespace
    ignored -- the ``-findwild`` syntax.  ``wildcard_pattern("0a ?? 4?")`` -> (b"\x0a\x00\x40", b"\xff\x00\xf0")."""
    digits = "".join(hex_text.split()).lower()
    if len(digits) % 2 or any(c not in "0123456789abcdef?" for c in digits):
        raise ValueError(f"not pairs of hex digits or ?: {hex_text!r}")
    if not 1 <= len(digits) // 2 <= MAX_PATTERN:
        raise ValueError(f"the pattern must be 1 to {MAX_PATTERN} bytes, not {len(digits) // 2}")
    if set(digits) == {"?"}:
        raise ValueError("the pattern has no hex digit that is not ?")
    value = bytes(int(digits[i:i + 2].replace("?", "0"), 16) for i in range(0, len(digits), 2))
    mask = bytes((0 if digits[i] == "?" else 0xF0) | (0 if digits[i + 1] == "?" else 0x0F) for i in range(0, len(digits), 2))
    return value, mask


def ignore_case_pattern(text: Any) -> Tuple[bytes, bytes]:
    """(pattern, mask) that matches `text` with every ASCII letter in either case: letters upper-cased with mask 0xDF,
    every other byte exact (0xFF)."""
    p = _fold(_pattern(text))
    return p, bytes(0xDF if 0x41 <= b <= 0x5A else 0xFF for b in p)


# numpy view of ``mod_set_match``: pattern `pattern` of a set starts at `pos` inside descriptor `desc`
SET_MATCH_DTYPE = np.dtype([("desc", "<u4"), ("pos", "<u4"), ("pattern", "<u4")])
MAX_SET_PATTERNS = 256


def _pattern_list(patterns: Any, ignore_case: bool = False) -> Tuple[np.ndarray, np.ndarray]:
    """-> (concatenated bytes, uint32 lengths) of 1 to 256 distinct patterns of 1 to 64 bytes (distinct ignoring ASCII
    case with `ignore_case`)."""
    ps = [_pattern(p) for p in patterns]
    if not 1 <= len(ps) <= MAX_SET_PATTERNS:
        raise ValueError(f"a set holds 1 to {MAX_SET_PATTERNS} patterns, not {len(ps)}")
    if len(set(_fold(p) if ignore_case else p for p in ps)) != len(ps):
        raise ValueError("the set holds the same pattern twice" + (" ignoring case" if ignore_case else ""))
    return np.frombuffer(b"".join(ps), np.uint8).copy(), np.array([len(p) for p in ps], np.uint32)


class PatternSet:
    """A set of 1 to 256 distinct byte patterns (1 to 64 bytes each, lengths mixed) resident on the current
    device, for ``Plan.find_set``: its filter and index are the library's business.  With `ignore_case` ASCII letters
    match either case (``mod_pattern_set_create_nocase``), and the patterns must differ ignoring case."""

    def __init__(self, patterns: Any, ignore_case: bool = False):
        data, lens = _pattern_list(patterns, ignore_case)
        self._lib = _abi.load()
        self._handle = ctypes.c_void_p()
        create = self._lib.mod_pattern_set_create_nocase if ignore_case else self._lib.mod_pattern_set_create
        _abi.check(create(data.ctypes.data, lens.ctypes.data, len(lens), ctypes.byref(self._handle)))
        self.n = len(lens)
        self.lengths = lens
        self.ignore_case = bool(ignore_case)

    def close(self) -> None:
        if self._handle:
            self._lib.mod_pattern_set_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _descs(descs: np.ndarray) -> np.ndarray:
    d = np.ascontiguousarray(descs, dtype=DESC_DTYPE)
    return d


class Plan:
    """Descriptors + tile map resident in HBM; ``run`` is one launch of the batched kernel."""

    def __init__(self, descs: np.ndarray, src_bytes: int, dst_bytes: int, dst_align: int = 0):
        d = _descs(descs)
        self._handle = ctypes.c_void_p()
        self._lib = _abi.load()
        _abi.check(self._lib.mod_plan_create(d.ctypes.data if len(d) else None, len(d), int(src_bytes),
                                             int(dst_bytes), int(dst_align), ctypes.byref(self._handle)))
        self.n = len(d)

    @property
    def payload_bytes(self) -> int:
        return int(self._lib.mod_plan_payload_bytes(self._handle))

    @property
    def num_tiles(self) -> int:
        return int(self._lib.mod_plan_num_tiles(self._handle))

    def run(self, src: Any, dst: Any, stream: int = 0) -> None:
        s_addr, _, _ = _buffer_info(src)
        d_addr, _, _ = _buffer_info(dst)
        _abi.check(self._lib.mod_plan_run(self._handle, s_addr, d_addr, stream or None))

    def tile_range(self, entry_begin: int, entry_end: int) -> Tuple[int, int]:
        """Tiles that belong to descriptors [entry_begin, entry_end)."""
        t0, t1 = ctypes.c_uint64(), ctypes.c_uint64()
        _abi.check(self._lib.mod_plan_tile_range(self._handle, int(entry_begin), int(entry_end),
                                                 ctypes.byref(t0), ctypes.byref(t1)))
        return int(t0.value), int(t1.value)

    def run_window(self, tile_begin: int, tile_end: int, src_win: Any, src_win_off: int, src_win_bytes: int,
                   dst_win: Any, dst_win_off: int, dst_win_bytes: int, stream: int = 0) -> None:
        """Run a tile sub-range with only a window of each buffer resident (slot-ring streaming)."""
        s_addr, _, _ = _buffer_info(src_win)
        d_addr, _, _ = _buffer_info(dst_win)
        _abi.check(self._lib.mod_plan_run_window(self._handle, int(tile_begin), int(tile_end), s_addr,
                                                 int(src_win_off), int(src_win_bytes), d_addr, int(dst_win_off),
                                                 int(dst_win_bytes), stream or None))

    def find(self, src: Any, pattern: Any, counts: Any, matches: Any, cap: int, total: Any, stream: int = 0,
             mask: Any = None) -> None:
        """Asynchronous search (``mod_plan_find``) of every descriptor for `pattern`: `counts` (uint32 per
        descriptor), `matches` (``MATCH_DTYPE`` slots, `cap` of them) and `total` (one uint64) are device buffers
        the results ACCUMULATE into.  The plan must have dst_off == src_off and dst_align == src & 15.  `mask` (one
        byte per pattern byte; ``mod_plan_find_masked``): byte t matches pattern byte k when
        ``(t ^ pattern[k]) & mask[k] == 0`` -- see ``wildcard_pattern`` and ``ignore_case_pattern``."""
        p = _pattern(pattern)
        args = (_buffer_info(counts)[0], _buffer_info(matches)[0] if cap else None, int(cap), _buffer_info(total)[0], stream or None)
        if mask is None:
            _abi.check(self._lib.mod_plan_find(self._handle, _buffer_info(src)[0], p, len(p), *args))
        else:
            _abi.check(self._lib.mod_plan_find_masked(self._handle, _buffer_info(src)[0], p, _mask(mask, len(p)), len(p), *args))

    def find_window(self, tile_begin: int, tile_end: int, src_win: Any, src_win_off: int, src_win_bytes: int,
                    pattern: Any, counts: Any, matches: Any, cap: int, total: Any, stream: int = 0, mask: Any = None) -> None:
        """``find`` over a tile sub-range with only a window of the source resident (slot-ring streaming)."""
        p = _pattern(pattern)
        win = (self._handle, int(tile_begin), int(tile_end), _buffer_info(src_win)[0], int(src_win_off), int(src_win_bytes))
        args = (_buffer_info(counts)[0], _buffer_info(matches)[0] if cap else None, int(cap), _buffer_info(total)[0], stream or None)
        if mask is None:
            _abi.check(self._lib.mod_plan_find_window(*win, p, len(p), *args))
        else:
            _abi.check(self._lib.mod_plan_find_masked_window(*win, p, _mask(mask, len(p)), len(p), *args))

    def find_set(self, src: Any, pattern_set: PatternSet, counts: Any, pattern_counts: Any, matches: Any, cap: int, total: Any,
                 owned: Any = None, stream: int = 0) -> None:
        """Asynchronous search (``mod_plan_find_set``) of every descriptor for every pattern of `pattern_set` in one
        pass: `counts` (uint32 per descriptor), `pattern_counts` (uint64 per pattern), `matches` (``SET_MATCH_DTYPE``
        slots, `cap` of them) and `total` (one uint64) are device buffers the results ACCUMULATE into; `owned`
        (device, uint32 per descriptor, or None) bounds the starts reported per descriptor."""
        _abi.check(self._lib.mod_plan_find_set(self._handle, _buffer_info(src)[0], pattern_set._handle,
                                               _buffer_info(owned)[0] if owned is not None else None, _buffer_info(counts)[0],
                                               _buffer_info(pattern_counts)[0], _buffer_info(matches)[0] if cap else None,
                                               int(cap), _buffer_info(total)[0], stream or None))

    def find_set_window(self, tile_begin: int, tile_end: int, src_win: Any, src_win_off: int, src_win_bytes: int,
                        pattern_set: PatternSet, counts: Any, pattern_counts: Any, matches: Any, cap: int, total: Any,
                        owned: Any = None, stream: int = 0) -> None:
        """``find_set`` over a tile sub-range with only a window of the source resident (slot-ring streaming)."""
        _abi.check(self._lib.mod_plan_find_set_window(self._handle, int(tile_begin), int(tile_end), _buffer_info(src_win)[0],
                                                      int(src_win_off), int(src_win_bytes), pattern_set._handle,
                                                      _buffer_info(owned)[0] if owned is not None else None,
                                                      _buffer_info(counts)[0], _buffer_info(pattern_counts)[0],
                                                      _buffer_info(matches)[0] if cap else None, int(cap),
                                                      _buffer_info(total)[0], stream or None))

    def close(self) -> None:
        if self._handle:
            self._lib.mod_plan_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def cycle_batch(descs: np.ndarray, src: Any, dst: Any, src_bytes: Optional[int] = None,
                dst_bytes: Optional[int] = None) -> None:
    """Gather/scatter + per-entry Cycle for every descriptor (synchronous; host or device buffers)."""
    d = _descs(descs)
    s_addr, s_n, _ = _buffer_info(src)
    d_addr, d_n, _ = _buffer_info(dst)
    src_bytes = s_n if src_bytes is None else src_bytes
    dst_bytes = d_n if dst_bytes is None else dst_bytes
    if src_bytes < 0 or dst_bytes < 0:
        raise ValueError("buffer sizes are required with raw addresses")
    _abi.check(_abi.load().mod_cycle_batch(d.ctypes.data if len(d) else None, len(d), s_addr, int(src_bytes),
                                           d_addr, int(dst_bytes)))


def find_batch(descs: np.ndarray, src: Any, pattern: Any, src_bytes: Optional[int] = None,
               max_matches: int = 1 << 20, mask: Any = None) -> Tuple[np.ndarray, np.ndarray, int]:
    """Search each descriptor's deciphered bytes (``src`` on the device: a raw address or a CUDA tensor) for
    `pattern` (synchronous).  -> (counts uint32[n], matches ``MATCH_DTYPE`` sorted by (desc, pos), at most
    `max_matches` of them, exact total).  `mask`: as for ``Plan.find`` (``mod_find_masked_batch``)."""
    d = _descs(descs)
    p = _pattern(pattern)
    s_addr, s_n, _ = _buffer_info(src)
    src_bytes = s_n if src_bytes is None else src_bytes
    if src_bytes < 0:
        raise ValueError("src_bytes is required with a raw address")
    counts = np.zeros(len(d), dtype=np.uint32)
    matches = np.zeros(max(0, int(max_matches)), dtype=MATCH_DTYPE)
    total = ctypes.c_uint64()
    out = (counts.ctypes.data if len(d) else None, matches.ctypes.data if len(matches) else None, len(matches), ctypes.byref(total))
    if mask is None:
        _abi.check(_abi.load().mod_find_batch(d.ctypes.data if len(d) else None, len(d), s_addr, int(src_bytes), p, len(p), *out))
    else:
        _abi.check(_abi.load().mod_find_masked_batch(d.ctypes.data if len(d) else None, len(d), s_addr, int(src_bytes), p,
                                                     _mask(mask, len(p)), len(p), *out))
    return counts, matches[:min(total.value, len(matches))].copy(), int(total.value)


def find_set_batch(descs: np.ndarray, src: Any, patterns: Any, src_bytes: Optional[int] = None,
                   max_matches: int = 1 << 20) -> Tuple[np.ndarray, np.ndarray, np.ndarray, int]:
    """``find_batch`` for a list of 1 to 256 distinct patterns in one pass (synchronous).  -> (counts uint32[n],
    pattern counts uint64[len(patterns)], matches ``SET_MATCH_DTYPE`` sorted by (desc, pos, pattern), at most
    `max_matches` of them, exact total)."""
    d = _descs(descs)
    data, lens = _pattern_list(patterns)
    s_addr, s_n, _ = _buffer_info(src)
    src_bytes = s_n if src_bytes is None else src_bytes
    if src_bytes < 0:
        raise ValueError("src_bytes is required with a raw address")
    counts = np.zeros(len(d), dtype=np.uint32)
    pattern_counts = np.zeros(len(lens), dtype=np.uint64)
    matches = np.zeros(max(0, int(max_matches)), dtype=SET_MATCH_DTYPE)
    total = ctypes.c_uint64()
    _abi.check(_abi.load().mod_find_set_batch(d.ctypes.data if len(d) else None, len(d), s_addr, int(src_bytes), data.ctypes.data,
                                              lens.ctypes.data, len(lens), counts.ctypes.data if len(d) else None,
                                              pattern_counts.ctypes.data, matches.ctypes.data if len(matches) else None,
                                              len(matches), ctypes.byref(total)))
    return counts, pattern_counts, matches[:min(total.value, len(matches))].copy(), int(total.value)


def cycle_batch_sharded(descs: np.ndarray, src: Any, dst: Any, src_bytes: Optional[int] = None,
                        dst_bytes: Optional[int] = None, dev_mask: int = 0) -> None:
    """``cycle_batch`` on HOST buffers with the descriptor list cut into equal-payload shards, one per
    selected GPU (``dev_mask`` bit d = CUDA device d, 0 = all), inside this process (synchronous)."""
    d = _descs(descs)
    s_addr, s_n, _ = _buffer_info(src)
    d_addr, d_n, _ = _buffer_info(dst)
    src_bytes = s_n if src_bytes is None else src_bytes
    dst_bytes = d_n if dst_bytes is None else dst_bytes
    if src_bytes < 0 or dst_bytes < 0:
        raise ValueError("buffer sizes are required with raw addresses")
    _abi.check(_abi.load().mod_cycle_batch_sharded(d.ctypes.data if len(d) else None, len(d), s_addr, int(src_bytes),
                                                   d_addr, int(dst_bytes), int(dev_mask)))


def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    b, e = ctypes.c_uint64(), ctypes.c_uint64()
    _abi.check(_abi.load().mod_shard_range(int(total), rank, world, ctypes.byref(b), ctypes.byref(e)))
    return int(b.value), int(e.value)


def shard_descs(descs: np.ndarray, rank: int, world: int) -> np.ndarray:
    """Rank's share of a descriptor list, balanced by payload bytes (large entries are cut and
    the tail piece gets the jumped key)."""
    d = _descs(descs)
    L = _abi.load()
    ptr = d.ctypes.data if len(d) else None
    n = _abi.check(L.mod_shard_descs(ptr, len(d), rank, world, None, 0))
    out = np.zeros(n, dtype=DESC_DTYPE)
    if n:
        _abi.check(L.mod_shard_descs(ptr, len(d), rank, world, out.ctypes.data, n))
    return out


def group_descs(descs: np.ndarray, group_bytes: int, dst_phase: int = 0, modulus: int = 128):
    """The pieces the host-pointer batch path cuts a descriptor list into and, per piece, whether a pipeline
    group ends after it (mod_group_descs; host logic)."""
    d = _descs(descs)
    L = _abi.load()
    ptr = d.ctypes.data if len(d) else None
    n = _abi.check(L.mod_group_descs(ptr, len(d), group_bytes, dst_phase, modulus, None, None, 0))
    out = np.zeros(n, dtype=DESC_DTYPE)
    closes = np.zeros(n, dtype=np.uint8)
    if n:
        _abi.check(L.mod_group_descs(ptr, len(d), group_bytes, dst_phase, modulus, out.ctypes.data, closes.ctypes.data, n))
    return out, closes


# ---- archive-level facade (include/modulate_ark.h): the reference's Unpack / Pack command bodies ----------

class ArkError(RuntimeError):
    """Carries the reference's eError code (Error.h:5-20)."""

    def __init__(self, code: int, what: str):
        super().__init__(f"{what} failed with eError {code}")
        self.code = code


def _slash(path: str) -> bytes:
    return (path if path.endswith("/") else path + "/").encode()


def ark_unpack(header_path: str, part_dir: str, target_dir: str, body_key: int = 0) -> None:
    """``CArk::Load`` + ``CArk::ExtractFiles`` (reference Modulate.cpp:291-317)."""
    rc = _abi.load().mod_ark_unpack(header_path.encode(), _slash(part_dir) if part_dir else b"", _slash(target_dir),
                                    _i32(body_key))
    if rc:
        raise ArkError(rc, "mod_ark_unpack")


def ark_pack(reference_header_path: str, input_dir: str, output_dir: str, header_name: str, *, ps4: bool = True,
             pack_all: bool = False, ignore_new_files: bool = True, body_key: int = 0) -> None:
    """The reference's Pack (Modulate.cpp:380-450): ``ConstructFromDirectory`` + ``BuildArk`` + ``SaveArk``."""
    rc = _abi.load().mod_ark_pack(reference_header_path.encode(), _slash(input_dir), _slash(output_dir),
                                  header_name.encode(), int(ps4), int(pack_all), int(ignore_new_files), _i32(body_key))
    if rc:
        raise ArkError(rc, "mod_ark_pack")


def ark_find(header_path: str, part_dir: str, pattern: Any, body_key: int = 0,
             max_matches: int = 1 << 20, mask: Any = None) -> Tuple[list, int]:
    """``CArk::Load`` + ``CArk::FindInFiles``: -> ([(file_index, offset), ...] sorted, exact total).  `mask`: as for
    ``Plan.find`` (``CArk::FindMaskedInFiles``)."""
    p = _pattern(pattern)
    files = np.zeros(max(0, int(max_matches)), dtype=np.uint32)
    offsets = np.zeros_like(files)
    total = ctypes.c_uint64()
    lib, where = _abi.load(), (header_path.encode(), _slash(part_dir) if part_dir else b"")
    out = (_i32(body_key), len(files), files.ctypes.data if len(files) else None, offsets.ctypes.data if len(files) else None,
           ctypes.byref(total))
    if mask is None:
        rc, name = lib.mod_ark_find(*where, p, len(p), *out), "mod_ark_find"
    else:
        rc, name = lib.mod_ark_find_masked(*where, p, _mask(mask, len(p)), len(p), *out), "mod_ark_find_masked"
    if rc:
        raise ArkError(rc, name)
    k = min(total.value, len(files))
    return [(int(f), int(o)) for f, o in zip(files[:k], offsets[:k])], int(total.value)


def ark_find_set(header_path: str, part_dir: str, patterns: Any, body_key: int = 0,
                 max_matches: int = 1 << 20, ignore_case: bool = False) -> Tuple[list, np.ndarray, int]:
    """``CArk::Load`` + ``CArk::FindSetInFiles``: -> ([(file_index, offset, pattern), ...] sorted, pattern counts, exact
    total).  `ignore_case`: ASCII letters match either case (``mod_ark_find_set_nocase``)."""
    data, lens = _pattern_list(patterns, ignore_case)
    name = "mod_ark_find_set_nocase" if ignore_case else "mod_ark_find_set"
    files = np.zeros(max(0, int(max_matches)), dtype=np.uint32)
    offsets, which = np.zeros_like(files), np.zeros_like(files)
    pattern_counts = np.zeros(len(lens), dtype=np.uint64)
    total = ctypes.c_uint64()
    rc = getattr(_abi.load(), name)(header_path.encode(), _slash(part_dir) if part_dir else b"", data.ctypes.data,
                                      lens.ctypes.data, len(lens), _i32(body_key), len(files),
                                      files.ctypes.data if len(files) else None, offsets.ctypes.data if len(files) else None,
                                      which.ctypes.data if len(files) else None, ctypes.byref(total), pattern_counts.ctypes.data)
    if rc:
        raise ArkError(rc, name)
    k = min(total.value, len(files))
    return [(int(f), int(o), int(w)) for f, o, w in zip(files[:k], offsets[:k], which[:k])], pattern_counts, int(total.value)


def dta_set_int(dta_path: str, key: str, value: int) -> None:
    rc = _abi.load().mod_dta_set_int(dta_path.encode(), key.encode(), int(value))
    if rc:
        raise ArkError(rc, "mod_dta_set_int")
