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


MAX_PATTERN = _parse("cycle_kernels.cuh", r"kMaxPattern = (\d+);")  # the search's longest pattern
if not re.search(r"kHaloChunks = \(int\)\(\(kMaxPattern - 1 \+ 15\) / 16\);",
                 open(os.path.join(_CSRC, "cycle_kernels.cuh")).read()):
    raise RuntimeError("kHaloChunks changed in cycle_kernels.cuh: the kernel model no longer matches the kernel")
HALO_CHUNKS = (MAX_PATTERN - 1 + 15) // 16  # kHaloChunks: chunks past a tile a match may reach into

# g_chunk_pow2, then c_halo_pow2: halo chunk k of a tile is stream chunk CHUNKS + k of the tile state
CHUNK_POW2 = np.array([2 * pow_a(16 * j) for j in range(CHUNKS + HALO_CHUNKS)], dtype=np.uint64)


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


# ==== search: find_batch_kernel ===========================================================================
# One CTA per tile of a plan whose chunk grid lies on the source (dst_off == src_off, dst_align == source
# address & 15).  The CTA loads its chunks (whole granules when the tile lies inside the source bounds, else byte
# loads that zero-fill every byte that is not the entry's), deciphers them with the speculative keystream (exact
# for a thread that takes the redo: any of its 4 rounds' states had bit 31 set), deciphers the halo -- the next
# min(rest, L - 1) bytes of the entry -- exactly with byte loads, and tests the starts [head, p_end).  The model
# restates that per tile; emulate_find_tile replays the shared-memory tile in numpy, with switches that drop
# one guard at a time.  tests/test_gpu_find_paths.py runs one case per (kind, load path, cell) on the GPU.

def tile_rest(r: TileRec) -> int:
    """make_tile_rec's `rest`: bytes of the entry after the tile (0 for its last tile)."""
    span = r.h0 + r.length
    c_end = r.tin * CHUNKS + r.n_valid
    return 0 if c_end == (span + 15) >> 4 else span - 16 * c_end


@dataclass
class FindLaunch:
    src: int    # FindArgs::src, the virtual base: a window's address minus its offset
    lo16: int
    hi16: int
    tiles: List[TileRec]


def _grid_descs(descs):
    return [(so, so, ln, key) for so, ln, key in descs]


def find_batch_launch(descs, src: int, src_bytes: int) -> FindLaunch:
    """mod_find_batch on (src_off, len, key) descriptors: dst_off = src_off, dst_align = src & 15, and the
    whole source buffer bounds the whole-granule loads."""
    return FindLaunch(src, (src + 15) & ~15, (src + src_bytes) & ~15, plan_tiles(_grid_descs(descs), src & 15))


def find_window_launch(descs, dst_align: int, t0: int, t1: int, win: int, win_off: int, win_bytes: int) -> FindLaunch:
    """mod_plan_find_window: tiles [t0, t1) of the plan, the window bounds the loads."""
    return FindLaunch(win - win_off, (win + 15) & ~15, (win + win_bytes) & ~15,
                      plan_tiles(_grid_descs(descs), dst_align)[t0:t1])


def find_window_ok(descs, dst_align: int, t0: int, t1: int, win_off: int, win_bytes: int, L: int) -> bool:
    """mod_plan_find_window's host check: every entry byte the tiles read, halos included, lies in the window."""
    ft = plan_first_tiles(_grid_descs(descs), dst_align)
    for e, (so, ln, _) in enumerate(descs):
        if ft[e + 1] == ft[e] or ft[e + 1] <= t0 or ft[e] >= t1:
            continue
        h0 = (dst_align + so) & 15
        ta, tb = max(t0, ft[e]) - ft[e], min(t1, ft[e + 1]) - ft[e]
        b0 = 0 if ta == 0 else ta * TILE_BYTES - h0
        b1 = min(ln, tb * TILE_BYTES - h0 + L - 1)
        if so + b0 < win_off or so + b1 > win_off + win_bytes:
            return False
    return True


GUARDS = ("head", "reach", "halo", "tile")


def scan_bounds(r: TileRec, L: int, guards=GUARDS) -> Tuple[int, int, int]:
    """(halo, first start, p_end) of the kernel, with the guards not in `guards` dropped:
    head  -- `p < head`: without it the scan starts at the word that holds `head`;
    reach -- p_end <= end + halo - L + 1: without it p_end = end;
    halo  -- halo = min(rest, L - 1): without it the halo is L - 1 bytes whether or not the entry has them;
    tile  -- p_end <= end, with the halo at most L - 1: without it the halo holds what it can of the entry
             (up to HALO_CHUNKS chunks) and the tile also takes the starts that fit in it."""
    rest = tile_rest(r)
    end = 16 * (r.n_valid - 1) + r.tail
    if "tile" not in guards:
        halo = min(rest, 16 * HALO_CHUNKS)
    else:
        halo = min(rest, L - 1) if "halo" in guards else L - 1
    reach = end + halo - L + 1
    if "reach" not in guards:
        p_end = end
    elif "tile" not in guards:
        p_end = max(0, reach)
    else:
        p_end = max(0, min(end, reach))
    return halo, (r.head if "head" in guards else r.head & ~3), p_end


@dataclass
class FindTile:
    """One tile of a search launch as the kernel runs it, for a pattern of L bytes."""
    rec: TileRec
    L: int
    whole: bool            # CTA-uniform: the chunks are loaded as whole granules
    rest: int
    halo: int
    end: int               # tile-local end of the entry's bytes
    p_end: int
    trig: np.ndarray = field(repr=False)       # [UNROLL, THREADS, 16]: bit 31 set (all four rounds count)
    redo: np.ndarray = field(repr=False)       # [THREADS]
    halo_trig: np.ndarray = field(repr=False)  # [HALO_CHUNKS, 16]

    @property
    def path(self) -> str:
        return "whole" if self.whole else "bytes"

    def halo_loaded(self) -> List[Tuple[int, int]]:
        """(halo chunk, bytes loaded from the source; the rest of the chunk is zero-filled) of every written
        halo chunk.  Chunks past the halo are never written: they hold stale shared memory."""
        return [(k, min(16, self.halo - 16 * k)) for k in range(HALO_CHUNKS) if 16 * k < self.halo]

    def compared(self, idx: int) -> Tuple[int, int]:
        """Bytes [lo, hi) of tile chunk `idx` that some start's window covers (lo == hi: none)."""
        a = self.rec.head
        b = min(self.end, self.p_end + self.L - 1) if self.p_end > a else a
        lo, hi = max(a, 16 * idx) - 16 * idx, min(b, 16 * idx + 16) - 16 * idx
        return (lo, hi) if hi > lo else (0, 0)

    def cells(self) -> Set[str]:
        """The redo and halo cells this tile hits with its key (see FIND_CELLS)."""
        out = set() if self.redo.any() else {"none"}
        n, T = self.rec.n_valid, THREADS
        compared_threads = set()
        for u, t, b in zip(*np.nonzero(self.trig)):
            u, t, b = int(u), int(t), int(b)
            idx = u * T + t
            lo, hi = self.compared(idx)
            if lo <= b < hi:
                compared_threads.add(t)
                if idx == 0 and self.rec.head:
                    out.add("head")
                if idx + 1 == n and self.rec.tail < 16:
                    out.add("tail")
                if (lo, hi) == (0, 16):
                    out.add("interior")
                if u == UNROLL - 1:
                    out.add("last-round")
            elif idx >= n and t < n:
                out.add("ghost")
        if len(compared_threads) >= 2:
            out.add("double")
        for k, nb in self.halo_loaded():
            if self.halo_trig[k, :nb].any():
                out.add(f"halo{k}")
        return out


def model_find_tile(launch: FindLaunch, r: TileRec, L: int, keyed: bool = True) -> FindTile:
    """keyed=False: geometry only (no trigger is computed)."""
    src_tile = launch.src + r.src_rel
    assert src_tile % 16 == 0, "the plan's chunk grid is not on the source"
    whole = src_tile >= launch.lo16 and src_tile + 16 * r.n_valid <= launch.hi16
    halo, _, p_end = scan_bounds(r, L)
    if keyed:
        trig = triggers(chunk_states(np.uint64(r.state), np.arange(CHUNKS + HALO_CHUNKS)))
    else:
        trig = np.zeros((CHUNKS + HALO_CHUNKS, 16), bool)
    main = trig[:CHUNKS].reshape(UNROLL, THREADS, 16)
    return FindTile(r, L, whole, tile_rest(r), halo, 16 * (r.n_valid - 1) + r.tail, p_end, main,
                    main.any(axis=(0, 2)), trig[CHUNKS:])


def find_keystream(r: TileRec) -> Tuple[np.ndarray, np.ndarray]:
    """(speculative, exact) keystream bytes [CHUNKS + HALO_CHUNKS, 16] of every chunk the CTA may decipher, the
    chunk-0 bytes before `head`, the last chunk's bytes after `tail` and the halo chunks included."""
    s = chunk_states(np.uint64(r.state), np.arange(CHUNKS + HALO_CHUNKS))
    return speculative_bytes(s), canonical_bytes(s)


def _read(mem: np.ndarray, a: int, n: int) -> np.ndarray:
    out = np.zeros(n, np.uint8)
    lo, hi = max(a, 0), min(a + n, mem.size)
    if hi > lo:
        out[lo - a:hi - a] = mem[lo:hi]
    return out


def find_tile_bytes(launch: FindLaunch, r: TileRec, mem: np.ndarray, L: int, guards=GUARDS,
                    redo: str = "exact") -> np.ndarray:
    """The CTA's shared-memory tile (int16, -1 where never written) for source bytes `mem` (launch addresses
    index it; bytes outside it read as zero, which only a dropped halo guard can load).  redo: "exact" (the
    kernel), "off" (never redo) or "round0" (a redone chunk starts from round 0's state: g_chunk_pow2[tid])."""
    ft = model_find_tile(launch, r, L)
    halo = scan_bounds(r, L, guards)[0]
    spec, exact = find_keystream(r)
    tile = np.full(16 * (CHUNKS + HALO_CHUNKS) + 16, -1, np.int16)
    src_tile = launch.src + r.src_rel
    for idx in range(r.n_valid):
        if ft.whole:
            data = _read(mem, src_tile + 16 * idx, 16)
        else:
            lo, hi = r.stored(idx)
            data = np.zeros(16, np.uint8)
            data[lo:hi] = _read(mem, src_tile + 16 * idx + lo, hi - lo)
        t = idx % THREADS
        ks = spec[idx] if not ft.redo[t] or redo == "off" else exact[t if redo == "round0" else idx]
        tile[16 * idx:16 * idx + 16] = data ^ ks
    for k in range(HALO_CHUNKS):
        if 16 * k < halo:
            data = np.zeros(16, np.uint8)
            nb = min(16, halo - 16 * k)
            data[:nb] = _read(mem, src_tile + 16 * (r.n_valid + k), nb)
            tile[16 * (r.n_valid + k):16 * (r.n_valid + k + 1)] = data ^ exact[CHUNKS + k]
    return tile


def emulate_find_tile(launch: FindLaunch, r: TileRec, mem: np.ndarray, pattern: bytes, guards=GUARDS,
                      redo: str = "exact") -> List[int]:
    """Tile-local starts the CTA reports.  With every guard on, no compared byte is stale (asserted)."""
    L = len(pattern)
    tile = find_tile_bytes(launch, r, mem, L, guards, redo)
    _, lo, p_end = scan_bounds(r, L, guards)
    if p_end <= lo:
        return []
    win = np.lib.stride_tricks.sliding_window_view(tile[lo:p_end + L - 1], L)
    if set(guards) == set(GUARDS):
        assert (win >= 0).all(), "a compared byte was never written"
    return [lo + int(p) for p in np.nonzero((win == np.frombuffer(pattern, np.uint8)).all(axis=1))[0]]


# ---- the search's cell matrix ------------------------------------------------------------------------------

FIND_KINDS = ("batch", "window")
FIND_PATHS = ("whole", "bytes")
HALO_CELLS = tuple(f"halo{k}" for k in range(HALO_CHUNKS))
GUARD_CELLS = ("before-head", "after-end", "past-rest", "across-tile")
FIND_CELLS = TRIGGERS + HALO_CELLS + GUARD_CELLS
GUARD_OF = {"before-head": "head", "after-end": "reach", "past-rest": "halo", "across-tile": "tile"}
FIND_LENGTHS = (1, 2, 17, 64)


def all_find_cells() -> List[Tuple[str, str, str]]:
    return [(k, p, c) for k in FIND_KINDS for p in FIND_PATHS for c in FIND_CELLS]


def find_unreachable_reason(kind: str, path: str, cell: str) -> Optional[str]:
    """Why a search cell cannot occur, or None.  test_kernel_model checks every reason against the sweep."""
    if cell.startswith("halo") and 16 * int(cell[4:]) >= MAX_PATTERN - 1:
        return "the halo is at most kMaxPattern - 1 bytes"
    return None


def reachable_find_cells() -> Set[Tuple[str, str, str]]:
    return {c for c in all_find_cells() if find_unreachable_reason(*c) is None}


def _decoy_start(ft: FindTile, cell: str) -> Optional[int]:
    """Tile-local start of the decoy a guard cell plants, or None if the geometry has no room for one."""
    r, L = ft.rec, ft.L
    if cell == "before-head":
        p = r.head & ~3
        return p if r.head & 3 and p < ft.p_end else None
    if cell == "after-end":
        p = max(r.head, ft.end - L + 1)
        return p if ft.rest == 0 and L >= 2 and p < ft.end and p + L <= 16 * r.n_valid else None
    if cell == "past-rest":
        p = ft.end + ft.rest + 1 - L
        return p if 0 < ft.rest < L - 1 and ft.rest % 16 and p >= r.head else None
    if cell == "across-tile":  # the match [end - L + 1, end] ends in halo chunk 0; the decoy follows it
        return ft.end + 1 if L >= 2 and ft.rest >= L + 1 and L + 1 <= 16 * HALO_CHUNKS else None
    raise ValueError(cell)


def find_geometric_cells(ft: FindTile) -> Set[str]:
    """Cells some key (redo, halo) or decoy (guards) could reach in this tile: the geometry alone decides."""
    r, n, T = ft.rec, ft.rec.n_valid, THREADS
    out = {"none"}
    lo = r.head
    hi = min(ft.end, ft.p_end + ft.L - 1) if ft.p_end > lo else lo  # compared bytes [lo, hi), as FindTile.compared
    if hi > lo:
        c0, c1 = lo // 16, (hi - 1) // 16  # compared chunks c0..c1
        if r.head and c0 == 0:
            out.add("head")
        if r.tail < 16 and c1 == n - 1:
            out.add("tail")
        if any(ft.compared(i) == (0, 16) for i in (c0, c0 + 1, c1 - 1, c1) if c0 <= i <= c1):
            out.add("interior")
        if c1 >= (UNROLL - 1) * T:
            out.add("last-round")
        if c1 > c0 and (c1 - c0 >= T or c0 % T != c1 % T):
            out.add("double")
        if n < CHUNKS and bool((np.arange(n, CHUNKS) % T < n).any()):
            out.add("ghost")
    out |= {f"halo{k}" for k, _ in ft.halo_loaded()}
    out |= {c for c in GUARD_CELLS if _decoy_start(ft, c) is not None}
    return out


@dataclass
class FindCase:
    """One search launch over three entries (src_off, len, key) of a source image.  batch: the image sits
    `src_ptr` bytes into a 16-byte aligned buffer.  window: tiles [t0, t1) of a plan with `dst_align` run over
    image bytes [win_off, win_off + win_bytes), held `win_ptr` bytes into a buffer of their own."""
    cell: Tuple[str, str, str]
    kind: str
    descs: List[Tuple[int, int, int]]
    target: int
    tin: int            # the target's tile the cell is built in
    L: int
    src_ptr: int
    image_bytes: int
    win: Optional[Tuple[int, int, int, int, int]] = None  # t0, t1, win_ptr, win_off, win_bytes
    pattern: bytes = b""
    image: Optional[np.ndarray] = field(default=None, repr=False)  # cipher bytes, built by make_find_case
    decoys: List[int] = field(default_factory=list)               # tile-local starts of guard decoys

    @property
    def dst_align(self) -> int:
        return (self.win[2] - self.win[3]) & 15 if self.win else self.src_ptr & 15

    def launch(self) -> FindLaunch:
        if self.win:
            t0, t1, wp, wo, wb = self.win
            return find_window_launch(self.descs, self.dst_align, t0, t1, wp, wo, wb)
        return find_batch_launch(self.descs, self.src_ptr, self.image_bytes)

    def memory(self) -> np.ndarray:
        """The source allocation the kernel reads."""
        if self.win:
            _, _, wp, wo, wb = self.win
            return np.concatenate([np.zeros(wp, np.uint8), self.image[wo:wo + wb]])
        return np.concatenate([np.zeros(self.src_ptr, np.uint8), self.image])

    def target_tile(self) -> Tuple[FindLaunch, TileRec]:
        la = self.launch()
        return la, next(r for r in la.tiles if r.entry == self.target and r.tin == self.tin)

    def cells(self) -> Set[Tuple[str, str, str]]:
        """Cells the case reaches in its target tile: the key's redo and halo cells, and each guard cell whose
        decoy the case planted."""
        la, r = self.target_tile()
        ft = model_find_tile(la, r, self.L)
        got = ft.cells()
        if self.decoys:
            got.add(self.cell[2])
        return {(self.kind, ft.path, c) for c in got}

    def entry_starts(self) -> Tuple[int, int]:
        """Entry positions [lo, hi) of the starts the launch's tiles of the target own."""
        la = self.launch()
        so, ln, _ = self.descs[self.target]
        tins = [r.tin for r in la.tiles if r.entry == self.target]
        h0 = (self.dst_align + so) & 15
        return max(0, TILE_BYTES * min(tins) - h0), min(ln - self.L + 1, TILE_BYTES * (max(tins) + 1) - h0)


_FIND_NEIGHBOURS = (37, 23)


def _find_layout(kind: str, h0: int, length: int, place: str, L: int, sub: str) -> Optional[FindCase]:
    """Entries [n0, target, n1] in a source image, the target at chunk-grid offset h0.  batch: place 'start' /
    'end' puts the target against the start / end of the source buffer, 'mid' leaves room.  window: the image
    always has room; `sub` picks the tile range ('all', or the target's 'first', 'last' or 'mid' tile) and
    `place` puts the window's start ('start') or end ('end') exactly on the bytes the range reads."""
    d0, d1 = _FIND_NEIGHBOURS
    if kind == "batch" and place == "start":
        src_ptr, tgt = h0, 0
        s1 = length + 5
        s0 = s1 + d1 + 3
        image_bytes = s0 + d0 + 11
    else:
        src_ptr = (5 * h0 + length + 3 * L) & 15
        s0 = 0
        tgt = d0 + 4 + ((h0 - src_ptr - d0 - 4) & 15)
        s1 = tgt + length
        image_bytes = s1 + d1 + 29
        if kind == "batch" and place == "end":
            s1 = d0 + 2
            tgt = s1 + d1 + ((h0 - src_ptr - s1 - d1) & 15)
            image_bytes = tgt + length
    descs = [(s0, d0, None), (tgt, length, None), (s1, d1, None)]
    case = FindCase((kind, "", ""), kind, descs, 1, 0, L, src_ptr, image_bytes)
    if kind == "batch":
        return case
    dst_align = (h0 - tgt) & 15
    ft = plan_first_tiles(_grid_descs(descs), dst_align)
    nt = ft[2] - ft[1]
    ta, tb = {"all": (0, nt), "first": (0, 1), "last": (nt - 1, nt), "mid": (1, nt - 1)}[sub]
    if tb <= ta or (sub != "all" and nt < 2) or (sub == "mid" and nt < 3):
        return None
    b0 = tgt + (0 if ta == 0 else ta * TILE_BYTES - h0)
    b1 = tgt + min(length, tb * TILE_BYTES - h0 + L - 1)
    lo = b0 if place == "start" else max(0, b0 - 19)
    hi = b1 if place == "end" else min(image_bytes, b1 + 21)
    case.win = (ft[1] + ta, ft[1] + tb, (lo + dst_align) & 15, lo, hi - lo)
    case.src_ptr = 0
    assert find_window_ok(descs, dst_align, ft[1] + ta, ft[1] + tb, lo, hi - lo, L)
    return case


def _find_lengths(h0: int, L: int) -> List[int]:
    out = set(range(1, 40)) | {3000, 5000, 7000}
    for b in (TILE_BYTES, 2 * TILE_BYTES):
        for d in (-L, 1 - L, 2 - L, -17, -16, -15, -2, -1, 0, 1, 2, 15, 16, 17, L - 2, L - 1, L, L + 1, 200):
            out.add(b - h0 + d)
    return sorted(x for x in out if x > 0)


def _find_geometries(kind: str):
    subs = ("all", "first", "last", "mid") if kind == "window" else ("all",)
    for L in FIND_LENGTHS:
        for h0 in range(16):
            for length in _find_lengths(h0, L):
                for place in ("mid", "start", "end"):
                    for sub in subs:
                        yield h0, length, place, L, sub


@functools.lru_cache(maxsize=None)
def _find_sweep(kind: str):
    """(geometries, {cell: [(geometry index, target tile index)]}) of every geometry of `kind`."""
    geoms, hits = [], {}
    for g in _find_geometries(kind):
        case = _find_layout(kind, *g)
        if case is None:
            continue
        gi = len(geoms)
        geoms.append(g)
        la = case.launch()
        for r in la.tiles:
            if r.entry != case.target:
                continue
            ft = model_find_tile(la, r, g[3], keyed=False)
            for c in find_geometric_cells(ft):
                hits.setdefault((kind, ft.path, c), []).append((gi, r.tin))
    return geoms, hits


def enumerate_reachable_find(kind: str) -> Set[Tuple[str, str, str]]:
    """Every search cell some geometry of `kind` makes possible: h0 0..15, lengths around every tile boundary
    +- (L - 1), the entry against the start or end of its buffer (or window) or with room, L in FIND_LENGTHS, and
    window ranges that start and end inside the entry."""
    return set(_find_sweep(kind)[1])


def _find_target_chunks(cell: str, ft: FindTile) -> List[Tuple[int, int, int]]:
    """(chunk, byte_lo, byte_hi) to make trigger for a redo or halo cell: the redone thread should own a valid
    chunk in a round > 0, so that a redo from round 0's state changes a compared byte."""
    n, T = ft.rec.n_valid, THREADS
    if cell.startswith("halo"):
        k = int(cell[4:])
        return [(CHUNKS + k, 0, dict(ft.halo_loaded())[k])]

    def later(i):
        return i % T + T < n

    comp = [i for i in range(n) if ft.compared(i) != (0, 0)]
    if cell == "ghost":
        cand = sorted((c for c in range(n, CHUNKS) if c % T < n), key=lambda c: not later(c))
        return [(c, 0, 16) for c in cand[:1]]
    if cell in ("interior", "double", "none"):
        cand = sorted((i for i in comp if ft.compared(i) == (0, 16)), key=lambda i: (not later(i), i // T != 1))
    elif cell == "last-round":
        cand = sorted((i for i in comp if i >= (UNROLL - 1) * T), key=lambda i: ft.compared(i) != (0, 16))
    elif cell == "head":
        cand = [0]
    else:  # tail
        cand = [n - 1]
    return [(i, *ft.compared(i)) for i in cand[:1] if ft.compared(i) != (0, 0)]


def _find_key(case: FindCase, rng) -> int:
    kind, path, cell = case.cell
    la, r = case.target_tile()
    if cell in GUARD_CELLS or cell == "none":  # a quiet key: no redo, no halo trigger
        for _ in range(1000):
            key = int(rng.integers(1, M))
            ft = model_find_tile(la, dataclasses.replace(r, state=tile_start_state(key_to_neg_state(key), r.h0, r.tin)), case.L)
            if ft.cells() == {"none"}:
                return key
        raise AssertionError("no quiet key")
    ft0 = model_find_tile(la, r, case.L, keyed=False)
    for chunk, lo, hi in _find_target_chunks(cell, ft0):
        for _ in range(64):
            for st in find_tile_state(chunk, lo, hi, rng):
                if cell in model_find_tile(la, dataclasses.replace(r, state=int(st)), case.L).cells():
                    return key_for_state(int(st), r.h0, r.tin)
    raise AssertionError(f"no key found for {case.cell}")


def _fill_find_case(case: FindCase, rng) -> None:
    """Pattern, plaintext plants, decoys and the enciphered image of a case whose keys are set."""
    import oracle
    L, cell = case.L, case.cell[2]
    la, r = case.target_tile()
    ft = model_find_tile(la, r, L)
    spec, exact = (a.reshape(-1) for a in find_keystream(r))
    used = np.where(np.repeat(ft.redo[np.arange(CHUNKS + HALO_CHUNKS) % THREADS], 16)
                    & (np.arange(16 * (CHUNKS + HALO_CHUNKS)) < 16 * CHUNKS), exact, spec)
    used[16 * CHUNKS:] = exact[16 * CHUNKS:]  # tile byte x -> keystream byte x (the halo follows a full tile)
    pat = rng.integers(1, 256, size=L, dtype=np.uint8)
    so_t, ln_t, _ = case.descs[case.target]

    def epos(x):  # entry position of tile-local byte x
        return TILE_BYTES * r.tin + x - r.h0

    plants: Dict[int, int] = {}  # target entry position -> plain byte
    image_sets: Dict[int, int] = {}  # image position -> cipher byte
    taken: List[Tuple[int, int]] = []

    def free(p):
        return all(p + L <= a or b <= p for a, b in taken)

    def plant(p, override=None):
        taken.append((p, p + L))
        for j in range(L):
            plants[epos(p + j)] = int(pat[j]) if override is None or j != override[0] else override[1]

    case.decoys = []
    if cell in GUARD_CELLS:
        p = _decoy_start(ft, cell)
        if cell == "across-tile":
            plant(ft.end - L + 1)  # a true match that ends in halo chunk 0
        for j in range(L):
            x, e = p + j, epos(p + j)
            if 0 <= e < ln_t:
                continue
            if cell == "past-rest":  # zero-filled halo bytes: the tile holds the exact keystream
                pat[j] = exact[x]
                image_sets[so_t + e] = 0
            elif ft.whole:
                image_sets[so_t + e] = int(pat[j] ^ used[x])
            else:  # zero-filled by the byte loads: the tile holds the keystream itself
                pat[j] = used[x]
        for j in range(L):
            if 0 <= epos(p + j) < ln_t:
                plants[epos(p + j)] = int(pat[j])
        case.decoys = [p]
    elif cell != "none":
        trig = [16 * (u * THREADS + t) + b for u, t, b in zip(*np.nonzero(ft.trig))
                if ft.compared(u * THREADS + t)[0] <= b < ft.compared(u * THREADS + t)[1]]
        trig += [16 * (r.n_valid + k) + int(b) for k, nb in ft.halo_loaded() for b in np.nonzero(ft.halo_trig[k, :nb])[0]]
        lo_p, hi_p = r.head, ft.p_end - 1

        def start_over(x):
            for p in range(max(lo_p, x - L + 1), min(hi_p, x) + 1):
                if free(p):
                    return p
            return None

        if trig:  # a match over a triggering byte: a skipped redo (or a speculative halo) misses it
            p = start_over(trig[0])
            if p is not None:
                plant(p)
        for x in trig[1:2]:  # a false match: plain byte = pattern ^ exact ^ speculative there
            q = start_over(x)
            if q is not None:
                plant(q, (x - q, int(pat[x - q] ^ exact[x] ^ spec[x])))
        for t in np.nonzero(ft.redo)[0]:  # a match in each redone thread's last valid round
            idx = max(i for i in range(int(t), r.n_valid, THREADS)) if t < r.n_valid else None
            if idx is not None and ft.compared(idx) != (0, 0):
                p = start_over(16 * idx + ft.compared(idx)[0])
                if p is not None:
                    plant(p)
    case.pattern = pat.tobytes()
    image = rng.integers(0, 256, size=case.image_bytes, dtype=np.uint8)
    for e, (so, ln, key) in enumerate(case.descs):
        plain = rng.integers(0, 256, size=ln, dtype=np.uint8)
        if e == case.target:
            for pos, v in plants.items():
                plain[pos] = v
        image[so:so + ln] = oracle.cycle(plain, key)
    for pos, v in image_sets.items():
        if 0 <= pos < image.size:
            image[pos] = v
    case.image = image


def make_find_case(cell: Tuple[str, str, str]) -> FindCase:
    """A launch that reaches `cell` in its target's tile: a geometry from the sweep (picked by a hash of the cell,
    preferring a redone thread with a valid chunk in a round > 0), a key, then plants and decoys."""
    kind, path, c = cell
    geoms, hits = _find_sweep(kind)
    seed = zlib.crc32(repr(cell).encode())
    rng = np.random.default_rng(seed)
    cand = list(hits[cell])
    order = rng.permutation(len(cand))
    pick = None
    for i in order[:200]:
        gi, tin = cand[int(i)]
        case = _find_layout(kind, *geoms[gi])
        r = next(r for r in case.launch().tiles if r.entry == case.target and r.tin == tin)
        if pick is None:
            pick = (gi, tin)
        n = r.n_valid
        if c in ("interior", "double", "head", "tail", "last-round") and n <= THREADS + 1:
            continue
        if c == "ghost" and not THREADS < n < CHUNKS:
            continue
        pick = (gi, tin)
        break
    gi, tin = pick
    case = _find_layout(kind, *geoms[gi])
    case.cell, case.tin = cell, tin
    keys = [int(k) for k in rng.integers(1, M, size=len(case.descs))]
    case.descs = [(so, ln, k) for (so, ln, _), k in zip(case.descs, keys)]
    so, ln, _ = case.descs[case.target]
    case.descs[case.target] = (so, ln, 0)
    case.descs[case.target] = (so, ln, _find_key(case, rng))
    _fill_find_case(case, rng)
    return case


def find_cases() -> List[FindCase]:
    return [make_find_case(c) for c in sorted(reachable_find_cells())]
