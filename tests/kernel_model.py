"""Host model of the cipher kernels' dispatch -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The batched kernel (modulate_b200/csrc/cycle_kernels.cu) speculates: it packs keystream bytes straight
from lazily reduced LCG states and redoes a thread's chunks exactly only when one of their states had
bit 31 set.  That branch runs for about one thread in 3 600, so which seeds happen to reach it is a
lottery.  This module restates, in plain numpy, which path every tile and chunk of a launch takes:

* the geometry (tiles_for_entry, make_tile_rec, tile_start_state) and the flavour and source bounds that
  each host entry point (mod_cycle_batch / mod_plan_run, mod_cycle_device, mod_plan_run_window) gives the
  kernel;
* the branch run_tile takes per tile, and per chunk whether its 16 lazy states trigger the redo;
* a key search that makes a chosen chunk byte trigger it.

It models the dispatch, not the output: the bytes are the oracle's job.  tests/test_kernel_model.py
ties the model to the oracle on the CPU; tests/test_gpu_kernel_paths.py runs one case per cell on the GPU.
"""
from __future__ import annotations

import dataclasses
import functools
import os
import re
import zlib
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Set, Tuple

import numpy as np

M = 0x7FFFFFFF
A = 16807
_MASK32 = np.uint64(0xFFFFFFFF)
_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "modulate_b200", "csrc")


def _parse(fname: str, pattern: str) -> int:
    with open(os.path.join(_CSRC, fname)) as f:
        m = re.search(pattern, f.read(), re.M)
    if m is None:
        raise RuntimeError(f"{pattern!r} not found in {fname}: the kernel model no longer matches the kernel")
    return int(m.group(1))


def _define(fname: str, name: str) -> int:
    """Default value of a `#define NAME <int>` knob in a kernel source file."""
    return _parse(fname, r"^#define\s+%s\s+(\d+)\b" % name)


THREADS = _define("cycle_kernels.cuh", "MODK_THREADS")
UNROLL = _define("cycle_kernels.cuh", "MODK_UNROLL")
EDGE_ROUNDS = _define("cycle_kernels.cu", "MODK_EDGE_ROUNDS")
GENERAL_FULL = _define("cycle_kernels.cu", "MODK_GENERAL_FULL")
CHUNKS = THREADS * UNROLL          # kChunksPerTile
TILE_BYTES = 16 * CHUNKS           # kTileBytes
TW0 = 1024                         # kTw0Size
TW1 = (1 << 32) // TILE_BYTES // TW0 + 2  # kTw1Size
MAX_PIECE = 1 << _parse("mod_abi.cu", r"kMaxPiece = 1ull << (\d+);")  # a contiguous call is cut into pieces
MAX_INLINE_DESCS = _parse("cycle_kernels.cuh", r"kMaxInlineDescs = (\d+);")  # pieces per launch


def pow_a(e: int) -> int:
    return pow(A, e % (M - 1), M)


def pow_a_inv(e: int) -> int:
    return pow_a((M - 1) - e % (M - 1))


CHUNK_POW2 = np.array([2 * pow_a(16 * j) for j in range(CHUNKS)], dtype=np.uint64)  # g_chunk_pow2


def i32(key: int) -> int:
    key = int(key) & 0xFFFFFFFF
    return key - (1 << 32) if key & 0x80000000 else key


def key_residue(key: int) -> int:
    return i32(key) % M


def key_to_neg_state(key: int) -> int:
    r = key_residue(key)
    return 0 if r == 0 else M - r


def tiles_for_entry(h0: int, length: int) -> int:
    if length == 0:
        return 0
    return ((h0 + length + 15) // 16 + CHUNKS - 1) // CHUNKS


def tile_start_state(n0: int, h0: int, tin: int) -> int:
    """(Negated, canonical) state just before byte TILE_BYTES * tin - h0 of the entry; the jump factor is
    split into the kernel's two tables."""
    assert tin // TW0 < TW1, "tile index beyond c_tw1"
    st = n0 * pow_a_inv(h0) % M
    return st * (pow_a(TILE_BYTES * (tin % TW0)) * pow_a(TILE_BYTES * TW0 * (tin // TW0)) % M) % M


@dataclass(frozen=True)
class TileRec:
    entry: int
    tin: int
    length: int    # the entry's length
    h0: int
    n_valid: int
    head: int
    tail: int
    src_rel: int
    dst_rel: int
    state: int
    pos0: int = 0  # stream byte of the entry's byte 0 (a piece of a contiguous call starts `done` bytes in)

    @property
    def full(self) -> bool:
        return self.n_valid == CHUNKS and self.head == 0 and self.tail == 16

    def stored(self, idx: int) -> Tuple[int, int]:
        """Bytes [lo, hi) of tile chunk `idx` that belong to the entry (lo == hi: none)."""
        if idx >= self.n_valid:
            return 0, 0
        return (self.head if idx == 0 else 0), (self.tail if idx + 1 == self.n_valid else 16)

    def entry_byte(self, idx: int, b: int) -> int:
        return TILE_BYTES * self.tin + 16 * idx + b - self.h0


def make_tile_rec(src_off: int, dst_off: int, length: int, n0: Optional[int], tin: int, dst_align: int, entry: int,
                  pos0: int = 0) -> TileRec:
    h0 = (dst_align + dst_off) & 15
    span = h0 + length
    nchunks = (span + 15) >> 4
    c_begin = tin * CHUNKS
    n_valid = min(CHUNKS, nchunks - c_begin)
    last = c_begin + n_valid == nchunks
    return TileRec(entry, tin, length, h0, n_valid, h0 if tin == 0 else 0, ((span - 1) & 15) + 1 if last else 16,
                   src_off - h0 + 16 * c_begin, dst_off - h0 + 16 * c_begin,
                   0 if n0 is None else tile_start_state(n0, h0, tin), pos0)


# ---- launches ---------------------------------------------------------------------------------------
# Addresses are offsets from 16-byte aligned allocation bases: only residues mod 16 and distances inside
# one buffer matter to the kernel.

@dataclass
class Launch:
    src: int           # BatchArgs::src (a virtual base for a window)
    dst: int
    lo16: int
    hi16: int
    coaligned: bool
    tiles: List[TileRec]


def uniform_delta_of(descs) -> int:
    delta = -1
    for so, do, ln, _ in descs:
        if ln == 0:
            continue
        d = (so - do) & 15
        if delta < 0:
            delta = d
        elif delta != d:
            return -1
    return delta


def _coaligned(src: int, dst: int, delta: int, force_general: bool) -> bool:
    return delta >= 0 and not force_general and ((src - dst + delta) & 15) == 0


def plan_tiles(descs, dst_align: int) -> List[TileRec]:
    """mod_plan_create: every tile record of the plan, in launch order."""
    out = []
    for e, (so, do, ln, key) in enumerate(descs):
        n0 = None if key is None else key_to_neg_state(key)  # no key: geometry only
        for tin in range(tiles_for_entry((dst_align + do) & 15, ln)):
            out.append(make_tile_rec(so, do, ln, n0, tin, dst_align, e))
    return out


def plan_first_tiles(descs, dst_align: int) -> List[int]:
    """first_tile of every descriptor plus the total (mod_plan_tile_range's table)."""
    ft, t = [], 0
    for so, do, ln, key in descs:
        ft.append(t)
        t += tiles_for_entry((dst_align + do) & 15, ln)
    return ft + [t]


def batch_launch(descs, src: int, dst: int, src_bytes: int, dst_align: Optional[int] = None,
                 force_general: bool = False) -> Launch:
    """mod_plan_run (and mod_cycle_batch on device pointers, which plans with dst_align = dst & 15)."""
    dst_align = dst & 15 if dst_align is None else dst_align
    assert dst & 15 == dst_align
    return Launch(src, dst, (src + 15) & ~15, (src + src_bytes) & ~15,
                  _coaligned(src, dst, uniform_delta_of(descs), force_general), plan_tiles(descs, dst_align))


def window_launch(descs, dst_align: int, tile_begin: int, tile_end: int, src_win: int, src_win_off: int,
                  src_win_bytes: int, dst_win: int, dst_win_off: int, force_general: bool = False) -> Launch:
    """mod_plan_run_window: virtual bases, and source bounds from the window."""
    src, dst = src_win - src_win_off, dst_win - dst_win_off
    assert dst & 15 == dst_align
    return Launch(src, dst, (src_win + 15) & ~15, (src_win + src_win_bytes) & ~15,
                  _coaligned(src, dst, uniform_delta_of(descs), force_general),
                  plan_tiles(descs, dst_align)[tile_begin:tile_end])


def inline_launches(src: int, dst: int, length: int, key: int, force_general: bool = False,
                    edges_only: bool = False) -> List[Launch]:
    """mod_cycle_device (launch_contiguous): 1 GiB pieces, up to 64 per launch, bounds from the call's extent.
    The bounds are not the pieces': the tiles either side of a piece boundary have a partial chunk and still
    read whole granules.  edges_only keeps tiles 0, 1, n-2 and n-1 of each piece: tiles 1 .. n-2 are all
    whole interior tiles that read nothing near the call's ends, so they take tile 1's path."""
    h0 = dst & 15
    lo16, hi16 = (src + 15) & ~15, (src + length) & ~15
    k0 = 0 if key is None else key_residue(key)
    out, done = [], 0
    while done < length:
        base, tiles, n = done, [], 0
        while done < length and n < MAX_INLINE_DESCS:
            this = min(MAX_PIECE, length - done)
            n0 = None if key is None else key_to_neg_state(k0 * pow_a(done) % M)
            off = done - base
            nt = tiles_for_entry(h0, this)
            keep = sorted({t for t in (0, 1, nt - 2, nt - 1) if 0 <= t < nt}) if edges_only else range(nt)
            tiles += [make_tile_rec(off, off, this, n0, t, (dst + base) & 15, n, done) for t in keep]
            done += this
            n += 1
        out.append(Launch(src + base, dst + base, lo16, hi16, _coaligned(src + base, dst + base, 0, force_general), tiles))
    return out


# ---- run_tile's branch -----------------------------------------------------------------------------

def tile_path(launch: Launch, r: TileRec) -> Tuple[str, int]:
    """-> (path, rounds that generate keystream states).  Paths: coal/fast, coal/slow, coal/U1..U3 (edge
    rounds), coal/U4-partial, gen/slow, gen/full/ws<k>, gen/partial/ws<k> with k = -1 (co-aligned tile in
    the general kernel) or the word shift 0..3."""
    sv = launch.src + r.src_rel
    shift = sv & 15
    src_tile = sv - shift
    if launch.coaligned and r.full and shift == 0 and src_tile >= launch.lo16 and src_tile + TILE_BYTES <= launch.hi16:
        return "coal/fast", UNROLL
    src_end = src_tile + 16 * (r.n_valid + (1 if shift else 0))
    if src_tile < launch.lo16 or src_end > launch.hi16 or (launch.coaligned and shift != 0):
        return ("coal/slow" if launch.coaligned else "gen/slow"), 0
    if launch.coaligned:
        if EDGE_ROUNDS and UNROLL == 4 and r.n_valid <= 3 * THREADS:
            u = (r.n_valid + THREADS - 1) // THREADS
            return f"coal/U{u}", u
        return f"coal/U{UNROLL}-partial", UNROLL
    ws = -1 if shift == 0 else shift >> 2
    return (f"gen/full/ws{ws}" if GENERAL_FULL and r.full else f"gen/partial/ws{ws}"), UNROLL


# ---- the speculative keystream -----------------------------------------------------------------------

def _lazy(p: np.ndarray) -> np.ndarray:
    return ((p >> np.uint64(32)) + ((p & _MASK32) >> np.uint64(1))) & _MASK32


def chunk_states(states, chunks) -> np.ndarray:
    """Lazy states after steps 1..16 of each chunk chain: jump_lazy(st, 2 a^(16 j)) then step_lazy.
    `states` and `chunks` broadcast; the result has one more axis of 16."""
    st = np.asarray(states, dtype=np.uint64)
    s = _lazy(st * CHUNK_POW2[np.asarray(chunks)])
    out = np.empty(s.shape + (16,), dtype=np.uint64)
    a2 = np.uint64(2 * A)
    for b in range(16):
        s = _lazy(s * a2)
        out[..., b] = s
    return out


def canonical_bytes(s: np.ndarray) -> np.ndarray:
    """What cycle_chunk_exact stores: low8 of the canonical residue."""
    return ((s + (s >> np.uint64(31))) & np.uint64(0xFF)).astype(np.uint8)


def speculative_bytes(s: np.ndarray) -> np.ndarray:
    """What the hot loop packs: the lazy states' low bytes, no fix-up."""
    return (s & np.uint64(0xFF)).astype(np.uint8)


def triggers(s: np.ndarray) -> np.ndarray:
    return (s >> np.uint64(31)).astype(bool)


TRIGGERS = ("none", "head", "tail", "interior", "last-round", "ghost", "double")


@dataclass
class TileModel:
    """One tile as the kernel runs it."""
    rec: TileRec
    path: str
    rounds: int
    trig: np.ndarray = field(repr=False)   # [rounds, THREADS, 16]: state of chunk t + THREADS*u, byte b had bit 31
    redo: np.ndarray = field(repr=False)   # [THREADS]: the thread takes the redo branch

    def trigger_bytes(self) -> List[Tuple[int, int, int]]:
        """(chunk, byte, entry byte) of every triggering state the tile generates."""
        u, t, b = np.nonzero(self.trig)
        return [(int(uu) * THREADS + int(tt), int(bb), self.rec.entry_byte(int(uu) * THREADS + int(tt), int(bb)))
                for uu, tt, bb in zip(u, t, b)]

    def cells(self) -> Set[str]:
        """The trigger cells this tile hits (see TRIGGERS)."""
        r = self.rec
        if not self.redo.any():
            return {"none"}
        out = set()
        stored_threads = set()
        for idx, b, eb in self.trigger_bytes():
            lo, hi = r.stored(idx)
            t, u = idx % THREADS, idx // THREADS
            if lo <= b < hi:
                assert 0 <= eb < r.length
                stored_threads.add(t)
                if idx == 0 and r.head:
                    out.add("head")
                if idx + 1 == r.n_valid and r.tail < 16:
                    out.add("tail")
                if lo == 0 and hi == 16:
                    out.add("interior")
                if u == self.rounds - 1:
                    out.add("last-round")
            elif idx >= r.n_valid and t < r.n_valid:
                out.add("ghost")
        if len(stored_threads) >= 2:
            out.add("double")
        return out


def model_tile(launch: Launch, r: TileRec) -> TileModel:
    path, rounds = tile_path(launch, r)
    if rounds == 0:  # the byte-granular path is exact: nothing speculative
        return TileModel(r, path, 0, np.zeros((0, THREADS, 16), bool), np.zeros(THREADS, bool))
    idx = np.arange(rounds * THREADS).reshape(rounds, THREADS)
    trig = triggers(chunk_states(r.state, idx))
    return TileModel(r, path, rounds, trig, trig.any(axis=(0, 2)))


def geometric_cells(launch: Launch, r: TileRec) -> Tuple[str, Set[str]]:
    """(path, trigger cells some key could reach) of a tile: the geometry alone decides which exist."""
    path, rounds = tile_path(launch, r)
    if rounds == 0:
        return path, {"none"}
    n = r.n_valid
    out = {"none", "last-round"}
    if r.head:
        out.add("head")
    if r.tail < 16:
        out.add("tail")
    if any(r.stored(i) == (0, 16) for i in (0, 1, 2) if i < n):
        out.add("interior")
    if any(c % THREADS < n for c in range(n, rounds * THREADS)):
        out.add("ghost")
    if n >= 2:
        out.add("double")
    if n <= THREADS * (rounds - 1):  # last round holds no valid chunk (general kernel, short tile)
        out.discard("last-round")
    return path, out


# ---- key search ------------------------------------------------------------------------------------

def find_tile_state(chunk: int, byte_lo: int, byte_hi: int, rng: np.random.Generator, count: int = 256) -> np.ndarray:
    """Tile states whose chain for `chunk` has bit 31 set at a byte in [byte_lo, byte_hi).

    A lazy state has bit 31 set only when its canonical residue is below 2 * 16807, so the search runs
    backwards: draw a small canonical residue c and a byte b, rewind c by a^(16 chunk + b + 1) to a tile
    state, and keep the states whose forward chain really triggers at b (about half of them)."""
    c = rng.integers(1, 12000, size=count, dtype=np.uint64)
    b = rng.integers(byte_lo, byte_hi, size=count)
    rew = np.array([pow_a_inv(16 * chunk + int(x) + 1) for x in b], dtype=np.uint64)
    st = (c * rew) % np.uint64(M)
    s = chunk_states(st, chunk)
    return st[triggers(s)[np.arange(count), b]]


def key_for_state(st: int, h0: int, tin: int, pos0: int = 0) -> int:
    """The (positive) key whose stream has state `st` at tile `tin` (chunk-grid offset h0) of the entry or
    piece that starts at stream byte pos0."""
    n0 = st * pow_a(h0) % M * pow_a_inv(TILE_BYTES * tin + pos0) % M
    assert n0 != 0
    k = M - n0
    assert tile_start_state(key_to_neg_state(k) * pow_a(pos0) % M, h0, tin) == st
    return k


# ---- the cell matrix -----------------------------------------------------------------------------------

KINDS = ("batch", "window", "inline", "inline-inplace")
PATHS = (["coal/fast", "coal/slow", "coal/U1", "coal/U2", "coal/U3", f"coal/U{UNROLL}-partial", "gen/slow"]
         + [f"gen/{f}/ws{w}" for f in ("full", "partial") for w in (-1, 0, 1, 2, 3)])


def all_cells() -> List[Tuple[str, str, str]]:
    return [(k, p, t) for k in KINDS for p in PATHS for t in TRIGGERS if not (p.endswith("/slow") and t != "none")]


def unreachable_reason(kind: str, path: str, trig: str) -> Optional[str]:
    """Why a cell cannot occur, or None.  test_kernel_model checks every reason against an enumeration."""
    inline = kind.startswith("inline")
    shifted = path.startswith("gen/") and path != "gen/slow" and not path.endswith("ws-1")
    if kind == "inline-inplace" and shifted:
        return "in place: source and destination agree mod 16, so there is no word shift"
    if (path.endswith("/fast") or "/full/" in path) and trig in ("head", "tail", "ghost"):
        return "a full tile has no partial chunk and no chunk beyond n_valid"
    if path == "coal/U1" and trig == "ghost":
        return "one round: a chunk beyond n_valid belongs to a thread with no valid chunk"
    if inline and trig == "tail" and path != "coal/U1" and not path.startswith("gen/partial/"):
        return ("inline: the call's own last chunk takes the slow path (the bounds are the call's extent); the only "
                "other partial last chunk is the one a 1 GiB piece ends with, alone in its tile")
    return None


def reachable_cells() -> Set[Tuple[str, str, str]]:
    return {c for c in all_cells() if unreachable_reason(*c) is None}


# ---- cases: one launch per cell --------------------------------------------------------------------------

@dataclass
class Case:
    """One GPU launch.  `descs` are relative to the src / dst pointers, which sit `src_ptr` / `dst_ptr` bytes
    into 16-byte aligned buffers of src_alloc / dst_alloc bytes.  A window case runs tiles [t0, t1) of the
    plan over a source and a destination window, each held `ptr` bytes into a buffer of its own (`win`)."""
    cell: Tuple[str, str, str]
    kind: str
    descs: List[Tuple[int, int, int, int]]
    target: int
    src_ptr: int
    src_bytes: int
    dst_ptr: int
    dst_bytes: int
    force_general: bool = False
    win: Optional[Tuple[int, int, int, int, int, int, int, int]] = None  # t0, t1, src_ptr, src_off, src_bytes, dst_ptr, dst_off, dst_bytes

    @property
    def src_alloc(self) -> int:
        return self.src_ptr + self.src_bytes

    @property
    def dst_alloc(self) -> int:
        return self.dst_ptr + self.dst_bytes

    @property
    def dst_align(self) -> int:
        return self.dst_ptr & 15

    def launches(self) -> List[Launch]:
        if self.kind in ("inline", "inline-inplace"):
            (so, do, ln, key), = self.descs
            return inline_launches(self.src_ptr + so, self.dst_ptr + do, ln, key, self.force_general,
                                   edges_only=ln > MAX_PIECE)
        if self.kind == "window":
            t0, t1, sp, soff, sb, dp, doff, db = self.win
            return [window_launch(self.descs, self.dst_align, t0, t1, sp, soff, sb, dp, doff, self.force_general)]
        return [batch_launch(self.descs, self.src_ptr, self.dst_ptr, self.src_bytes, force_general=self.force_general)]

    def tiles(self) -> List[Tuple[Launch, TileRec]]:
        return [(la, r) for la in self.launches() for r in la.tiles]

    def modelled_ranges(self) -> List[Tuple[int, int]]:
        """[lo, hi) byte ranges of a contiguous call covered by the tiles the model keeps."""
        out = []
        for _, r in self.tiles():
            lo = max(0, TILE_BYTES * r.tin - r.h0)
            hi = min(r.length, TILE_BYTES * (r.tin + 1) - r.h0)
            out.append((r.pos0 + lo, r.pos0 + hi))
        return out

    def is_target(self, r: TileRec) -> bool:
        """The tile belongs to the entry the case was built for (every piece of a contiguous call does)."""
        return self.kind.startswith("inline") or r.entry == self.target

    def cells(self) -> Set[Tuple[str, str, str]]:
        """Cells the launch reaches (a call of several pieces: in the tiles inline_launches keeps)."""
        out = set()
        for la, r in self.tiles():
            tm = model_tile(la, r)
            out |= {(self.kind, tm.path, t) for t in tm.cells()}
        return out


_DECOY = (37, 23)  # lengths of the entries around the target in batch and window cases


def _layout(kind: str, ps: int, pd: int, length: int, place: str, general: bool, dst_ptr: int, key: int) -> Case:
    """A launch whose target entry starts at source residue ps and destination residue pd.  place: 'start' /
    'end' puts the entry against the start / end of the source buffer (or window), 'mid' leaves room."""
    if kind.startswith("inline"):
        inplace = kind == "inline-inplace"
        src_ptr = ps
        d_ptr = ps if inplace else 16 + pd
        return Case((kind, "", ""), kind, [(0, 0, length, key)], 0, src_ptr, length + 16 + 32,
                    d_ptr, length + 16 + 32, force_general=general and ps == pd)
    shift = (ps - pd) & 15
    mixed = general and shift == 0  # a co-aligned tile in the general kernel: one decoy gets another delta
    d0, d1 = _DECOY
    # destination: [guard | decoy0 | hole | target | hole | decoy1 | guard], target at residue pd
    dst0 = 16
    tgt_dst = dst0 + d0 + 5
    tgt_dst += (pd - dst_ptr - tgt_dst) & 15
    dst1 = tgt_dst + length + 7
    dst_bytes = dst1 + d1 + 16
    # source: the target at residue ps, decoys elsewhere
    if place == "start":
        src_ptr, tgt_src = ps, 0
        s0 = length + 16
        s1 = s0 + d0 + 3
        src_bytes = s1 + d1 + 16
    else:
        src_ptr = 0
        s0 = 0
        tgt_src = d0 + 16 + ((ps - d0 - 16) & 15)
        s1 = tgt_src + length + 32
        src_bytes = s1 + d1 + 1 if place == "mid" else None
        if place == "end":  # decoy1 moves before the target, the buffer ends with the target's last byte
            s1 = d0 + 2
            tgt_src = s1 + d1 + 16
            tgt_src += (ps - tgt_src) & 15
            src_bytes = tgt_src + length
    # decoys keep the target's delta (so the launch flavour is the target's) unless `mixed`
    delta = (tgt_src + src_ptr - tgt_dst - dst_ptr) & 15
    def fit(s, d):
        return s + ((d + dst_ptr + delta - s - src_ptr) & 15)
    s0 = fit(s0, dst0)
    s1 = fit(s1, dst1) if not mixed else fit(s1, dst1) + 1
    if place == "start":
        src_bytes = max(src_bytes, s1 + d1 + 16)
    elif place == "mid":
        src_bytes = s1 + d1 + 1
    keys = [None, None] if key is None else \
        [int(k) for k in np.random.default_rng(length * 256 + ps * 16 + pd).integers(1, 1 << 32, size=2)]
    descs = [(s0, dst0, d0, keys[0]), (tgt_src, tgt_dst, length, key), (s1, dst1, d1, keys[1])]
    assert all(s + ln <= src_bytes for s, _, ln, _ in descs), (place, descs, src_bytes)
    case = Case((kind, "", ""), kind, descs, 1, src_ptr, src_bytes, dst_ptr, dst_bytes)
    if kind == "window":
        ft = plan_first_tiles(descs, dst_ptr & 15)
        lo = tgt_src if place == "start" else tgt_src - 16 - (ps & 3)
        hi = tgt_src + length if place == "end" else tgt_src + length + 16
        d_lo, d_hi = tgt_dst - 3, tgt_dst + length + 3
        win_src_ptr = (ps - (tgt_src - lo)) & 15
        win_dst_ptr = 16 + ((dst_ptr + d_lo - 16) & 15)
        case.win = (ft[1], ft[2], win_src_ptr, lo, hi - lo, win_dst_ptr, d_lo, d_hi - d_lo)
    return case


def _shifts(general: bool) -> List[Tuple[int, int]]:
    """(ps, pd) pairs: co-aligned pairs for the co-aligned flavour, every pair for the general one."""
    return [(ps, pd) for ps in range(16) for pd in range(16) if general or ps == pd]


_LENGTHS = sorted(set(range(1, 36)) | {b + d for b in (2048, 4096, 6144, 8192, 16384, 24576)
                                        for d in (-17, -16, -15, -1, 0, 1, 15, 16, 17)} | {3000, 5000, 7000, 20000})


# contiguous calls of two pieces: the second piece's first tile in every edge-round class
_PIECE_LENGTHS = [MAX_PIECE + d for d in (1, 17, 2047, 2049, 4000, 5000, 7000, 8100, 8192, 8300, 20000)]


def _geometries(kind: str):
    inline = kind.startswith("inline")
    places = ("mid",) if inline else ("mid", "start", "end")
    for general in (False, True):
        pairs = [(p, p) for p in range(16)] if kind == "inline-inplace" else _shifts(general)
        for ps, pd in pairs:
            for length in _LENGTHS + (_PIECE_LENGTHS if inline else []):
                for place in places:
                    yield ps, pd, length, place, general, (5 * ps + 3 * pd + length) & 15


@functools.lru_cache(maxsize=None)
def _sweep(kind: str):
    """Geometries of `kind` (see _geometries) and, per reachable cell, the ones whose target entry has a tile
    that makes it possible: (geometries, {cell: [(geometry index, (entry, tile index), sensitive)]})."""
    geoms = list(_geometries(kind))
    hits: Dict[Tuple[str, str, str], list] = {}
    for gi, (ps, pd, length, place, general, dst_ptr) in enumerate(geoms):
        case = _layout(kind, ps, pd, length, place, general, dst_ptr, key=None)
        for la, r in case.tiles():
            if not case.is_target(r):
                continue
            path, trig = geometric_cells(la, r)
            rounds = tile_path(la, r)[1]
            for t in trig:
                hits.setdefault((kind, path, t), []).append((gi, (r.entry, r.tin), _sensitive(t, r, rounds)))
    return geoms, hits


def enumerate_reachable(kind: str) -> Set[Tuple[str, str, str]]:
    """Every (kind, path, trigger) cell that some geometry of `kind` makes possible for some key: all 16 x 16
    source / destination residues, lengths around every round and tile boundary, entries against either end
    of their buffer or with room, and contiguous calls that cross a piece boundary."""
    return set(_sweep(kind)[1])


def _target_chunks(trig: str, r: TileRec, rounds: int) -> List[Tuple[int, int, int]]:
    """Candidate (chunk, byte_lo, byte_hi) to make trigger, best first: the redone thread should own a valid
    chunk in a round > 0, so that a redo that restarts every chunk from round 0's state changes a byte."""
    n = r.n_valid
    T = THREADS

    def span(i):
        lo, hi = r.stored(i)
        return (i, lo, hi) if hi > lo else None

    def valid_later(i):  # the thread owning chunk i has a valid chunk in a round > 0
        return i % T + T < n

    cand = []
    if trig in ("interior", "double", "none"):
        cand = [i for i in range(n) if r.stored(i) == (0, 16)]
        cand.sort(key=lambda i: (not valid_later(i), i // T != 1))
    elif trig == "last-round":
        cand = [i for i in range((rounds - 1) * T, min(n, rounds * T))]
        cand.sort(key=lambda i: r.stored(i) != (0, 16))
    elif trig == "head":
        cand = [0] if r.head else []
    elif trig == "tail":
        cand = [n - 1] if r.tail < 16 else []
    elif trig == "ghost":
        cand = [c for c in range(n, rounds * T) if c % T < n]
        cand.sort(key=lambda c: not valid_later(c))
        return [(c, 0, 16) for c in cand[:1]]
    return [s for s in (span(i) for i in cand[:1]) if s]


def _sensitive(trig: str, r: TileRec, rounds: int) -> bool:
    """The cell's trigger can sit in a thread that owns a valid chunk in a round > 0 (see _target_chunks)."""
    n, T = r.n_valid, THREADS
    if trig == "none":
        return True
    if trig == "last-round":
        return rounds >= 2 and n > (rounds - 1) * T
    if trig == "ghost":
        t_max = min(T - 1, n - T - 1)
        return t_max >= 0 and t_max + (rounds - 1) * T >= n
    return n > T + 1


def _tile_chunks(geom, tile) -> int:
    ps, pd, length, place, general, dst_ptr = geom  # pd: the target's destination residue, its chunk-grid offset h0
    entry, tin = tile  # the entry is a piece index only in a contiguous call longer than one piece
    piece_len = min(MAX_PIECE, length - entry * MAX_PIECE) if length > MAX_PIECE else length
    return min(CHUNKS, (pd + piece_len + 15) // 16 - tin * CHUNKS)


def make_case(cell: Tuple[str, str, str]) -> Case:
    """A launch that hits `cell` with its target entry: a geometry from the sweep behind enumerate_reachable
    (picked by a hash of the cell, so dst_align, shifts and lengths vary from cell to cell), preferring one
    where the redone thread owns a valid chunk in a round > 0, then a key that makes the chosen chunk trigger."""
    kind, path, trig = cell
    geoms, hits = _sweep(kind)
    # entries of at most 64 KiB where they reach the cell; a contiguous call across a 1 GiB piece boundary otherwise
    usable = [h for h in hits[cell] if geoms[h[0]][2] <= 64 << 10] or hits[cell]
    if trig == "double":  # two triggering threads in one tile: give the second one room to happen
        usable = [h for h in usable if _tile_chunks(geoms[h[0]], h[1]) >= THREADS // 2] or usable
    cand = [h for h in usable if h[2]] or usable
    seed = zlib.crc32(repr(cell).encode())
    gi, tile, _ = cand[seed % len(cand)]
    ps, pd, length, place, general, dst_ptr = geoms[gi]
    case = _layout(kind, ps, pd, length, place, general, dst_ptr, key=0)  # the target's key is chosen below
    la, r = next((la, r) for la, r in case.tiles() if case.is_target(r) and (r.entry, r.tin) == tile)
    return _with_key(case, la, r, trig, tile_path(la, r)[1], np.random.default_rng(seed))


def _with_key(case: Case, la: Launch, r: TileRec, trig: str, rounds: int, rng) -> Case:
    kind = case.kind
    cell = (kind, tile_path(la, r)[0], trig)

    def rekey(key):
        so, do, ln, _ = case.descs[case.target]
        c = Case(cell, kind, list(case.descs), case.target, case.src_ptr, case.src_bytes, case.dst_ptr,
                 case.dst_bytes, case.force_general, case.win)
        c.descs[case.target] = (so, do, ln, key)
        return c

    def target_tile(c):
        for la2, r2 in c.tiles():
            if c.is_target(r2) and (r2.entry, r2.tin) == (r.entry, r.tin):
                return model_tile(la2, r2)

    if rounds == 0 or trig == "none":
        for _ in range(1000):
            c = rekey(int(rng.integers(1, M)))
            if rounds == 0 or not target_tile(c).redo.any():
                return c
        raise AssertionError("no quiet key")
    for chunk, lo, hi in _target_chunks(trig, r, rounds):
        for _ in range(64):
            for st in find_tile_state(chunk, lo, hi, rng):
                if trig in model_tile(la, dataclasses.replace(r, state=int(st))).cells():
                    c = rekey(key_for_state(int(st), r.h0, r.tin, r.pos0))
                    assert trig in target_tile(c).cells()
                    return c
    raise AssertionError(f"no key found for {cell}")


def cases() -> List[Case]:
    return [make_case(c) for c in sorted(reachable_cells())]


# ---- whole batches --------------------------------------------------------------------------------------

def entries_with_trigger_bytes(descs, dst_align: int = 0, tiles_per_pass: int = 2048) -> np.ndarray:
    """Indices of the entries of which some stored byte comes from a state with bit 31 set, i.e. would be
    wrong if the kernel skipped its redo.  Tiles are modelled `tiles_per_pass` at a time."""
    recs = plan_tiles(descs, dst_align)
    hit = np.zeros(len(descs), bool)
    idx = np.arange(CHUNKS)
    for t0 in range(0, len(recs), tiles_per_pass):
        part = recs[t0:t0 + tiles_per_pass]
        trig = triggers(chunk_states(np.array([r.state for r in part], np.uint64)[:, None], idx[None, :]))
        for k in np.nonzero(trig.any(axis=(1, 2)))[0]:
            r = part[k]
            for c, b in zip(*np.nonzero(trig[k])):
                lo, hi = r.stored(int(c))
                if lo <= b < hi:
                    hit[r.entry] = True
                    break
    return np.nonzero(hit)[0]
