"""The masked search (find_batch_kernel<true>) and the case-folded pattern sets (find_set_kernel<true>), restated in
plain numpy on top of tests/kernel_model.py: the anchor choice, the masked filter on 32-bit words, an emulation of the
CTA's shared-memory tile with stale bytes, the filter's farthest read, and the folded set's bitmap."""
from __future__ import annotations

from typing import List

import numpy as np

from kernel_model import HALO_CHUNKS, TILE_BYTES, FindLaunch, TileRec, _parse, find_tile_bytes, scan_bounds

# ---- the masked search (find_batch_kernel<true>) -------------------------------------------------------------
#
# Pattern byte k is (value[k], mask[k]) with value[k] & mask[k] == value[k]: entry byte t matches when
# ((t ^ value[k]) & mask[k]) == 0.  The filter tests the anchor pair (a, a + 1) of every start with the exact kernel's
# SWAR zero-byte test on (bytes ^ rep) & mrep; a start that passes is compared under the mask.

FIND_SLACK_WORDS = _parse("cycle_kernels.cu", r"kFindSlackWords = (\d+)u;")
S_W_BYTES = TILE_BYTES + 16 * HALO_CHUNKS + 4 * FIND_SLACK_WORDS  # find_batch_kernel's s_w


def find_anchor(mask: bytes) -> int:
    """mod_abi.cu's find_anchor: the adjacent pair (a, a + 1) with the most mask bits, the first of equals."""
    if len(mask) == 1:
        return 0
    bits = [bin(mask[k]).count("1") + bin(mask[k + 1]).count("1") for k in range(len(mask) - 1)]
    return bits.index(max(bits))


def _swar_zero(v: int) -> int:
    return ((v - 0x01010101) & ~v & 0x80808080) & 0xFFFFFFFF


def masked_filter_word(sw: np.ndarray, w: int, value: bytes, mask: bytes) -> int:
    """The filter of word w over the uint8 shared array `sw`: bit 8 o + 7 set for every start 4 w + o whose anchor
    pair matches (and possibly above such a byte).  The clamped funnel shift of a & 3 == 3 takes all of the second word."""
    L, a = len(value), find_anchor(mask)
    wa, sh = w + (a >> 2), 8 * (a & 3)
    xa = int(sw[4 * wa:4 * wa + 4].view("<u4")[0])
    ya = int(sw[4 * wa + 4:4 * wa + 8].view("<u4")[0])
    pair = ya << 32 | xa
    m = _swar_zero(((pair >> sh) & 0xFFFFFFFF ^ 0x01010101 * value[a]) & 0x01010101 * mask[a])
    if L > 1:
        m &= _swar_zero(((pair >> min(sh + 8, 32)) & 0xFFFFFFFF ^ 0x01010101 * value[a + 1]) & 0x01010101 * mask[a + 1])
    return m


def masked_filter_reach(L: int, a: int, end: int, halo: int) -> int:
    """The farthest s_w byte the masked filter reads in a tile whose entry bytes end at `end` (tile-local) with
    `halo` bytes past it, or -1 when no word is tested."""
    p_end = max(0, min(end, end + halo - L + 1))
    if p_end == 0:
        return -1
    w = (p_end - 1) // 4
    return 4 * (w + (a >> 2) + 1) + 3


def emulate_masked_find_tile(launch: FindLaunch, r: TileRec, mem: np.ndarray, value: bytes, mask: bytes,
                             stale: int = 0xA5) -> List[int]:
    """Tile-local starts find_batch_kernel<true> reports.  Never-written shared bytes read as `stale`; the filter
    may read them, and it is asserted that the compare never does and that the filter stays inside s_w."""
    L = len(value)
    value = bytes(v & m for v, m in zip(value, mask))
    tile = find_tile_bytes(launch, r, mem, L)
    sw = np.full(S_W_BYTES, stale, np.uint8)
    sw[:tile.size] = np.where(tile >= 0, tile, stale).astype(np.uint8)
    _, head, p_end = scan_bounds(r, L)
    a = find_anchor(mask)
    vm, mm = np.frombuffer(value, np.uint8), np.frombuffer(mask, np.uint8)
    out = []
    for w in range(head >> 2, (p_end + 3) // 4):
        assert 4 * (w + (a >> 2) + 1) + 3 < S_W_BYTES, "the masked filter reads past s_w"
        if masked_filter_word(sw, w, value, mask) == 0:
            continue
        for o in range(4):
            p = 4 * w + o
            if p < head or p >= p_end:
                continue
            win = tile[p:p + L]
            assert (win >= 0).all(), "a compared byte was never written"
            if not ((win.astype(np.uint8) ^ vm) & mm).any():
                out.append(p)
    return out


def masked_positions(data: np.ndarray, value: bytes, mask: bytes) -> List[int]:
    """numpy: every start of `data` whose bytes match (value, mask)."""
    L = len(value)
    if data.size < L:
        return []
    win = np.lib.stride_tricks.sliding_window_view(data, L)
    mm = np.frombuffer(mask, np.uint8)
    hit = ((win & mm) == (np.frombuffer(value, np.uint8) & mm)).all(axis=1)
    return [int(i) for i in np.nonzero(hit)[0]]


# ---- case-folded pattern sets (find_set_kernel<true>) --------------------------------------------------------

def fold(b: int) -> int:
    """modk::fold_ascii: a..z -> A..Z, every other byte itself."""
    return b - 0x20 if 0x61 <= b <= 0x7A else b


def fold_set_bitmap(patterns: List[bytes]) -> np.ndarray:
    """The filter bitmap of mod_pattern_set_create_nocase, as 65536 bools indexed by b0 | b1 << 8: every case
    variant of each folded pattern's first two bytes (both (b0, *) rows of a length-1 letter)."""
    bm = np.zeros(65536, bool)
    for p in patterns:
        b0 = fold(p[0])
        v0 = {b0, b0 | 0x20} if 0x41 <= b0 <= 0x5A else {b0}
        for c0 in v0:
            if len(p) == 1:
                bm[c0 | np.arange(256) << 8] = True
                continue
            b1 = fold(p[1])
            for c1 in ({b1, b1 | 0x20} if 0x41 <= b1 <= 0x5A else {b1}):
                bm[c0 | c1 << 8] = True
    return bm
