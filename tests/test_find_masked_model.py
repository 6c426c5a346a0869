"""CPU: the masked search (find_batch_kernel<true>) and the case-folded set filter restated in tests/kernel_model.py.
The anchor choice, the masked filter over an emulated shared-memory tile against numpy over the oracle-deciphered
entries for every search cell, the bound on the filter's farthest read, and the folded set's bitmap."""
import functools

import numpy as np
import pytest

import kernel_model as km
import kernel_model_masked as kmm
import oracle


@functools.lru_cache(maxsize=None)
def _find_cases():
    return km.find_cases()


def test_anchor_takes_the_pair_with_the_most_mask_bits_first_of_equals():
    assert kmm.find_anchor(b"\xff") == 0
    assert kmm.find_anchor(b"\x00\x00\xff\xff\x00") == 2       # leading wildcards are skipped
    assert kmm.find_anchor(b"\xff\xff\x00\xff\xff") == 0       # ties go to the smallest a
    assert kmm.find_anchor(b"\xf0\x0f\xff\xdf") == 2
    assert kmm.find_anchor(b"\x00\x0f") == 0
    assert kmm.find_anchor(bytes(63) + b"\x01") == 62


def test_the_filter_read_stays_inside_shared_memory():
    """For every L, anchor, tile end near the tile's size and halo the farthest filter read lies in s_w."""
    assert kmm.S_W_BYTES == km.TILE_BYTES + 16 * km.HALO_CHUNKS + 16
    worst = 0
    for L in range(1, km.MAX_PATTERN + 1):
        for a in range(max(1, L - 1)):
            for end in list(range(1, 9)) + list(range(km.TILE_BYTES - 8, km.TILE_BYTES + 1)):
                for halo in range(0, L):
                    worst = max(worst, kmm.masked_filter_reach(L, a, end, halo))
    assert worst < kmm.S_W_BYTES
    assert worst <= km.TILE_BYTES + km.MAX_PATTERN + 4  # the bound the kernel's comment states


def _masks(L, rng):
    """(name, mask): random bytes and nibbles, leading wildcards, trailing wildcards, both."""
    out = []
    m = rng.choice(np.array([0xFF, 0xFF, 0x00, 0xF0, 0x0F, 0xDF], np.uint8), size=L)
    if not m.any():
        m[L // 2] = 0xFF
    out.append(("random", bytes(m)))
    if L >= 3:
        k = min(L - 2, 1 + L // 4)
        out.append(("lead", bytes(k) + b"\xff" * (L - k)))
        out.append(("trail", b"\xff" * (L - k) + bytes(k)))
        out.append(("both", b"\x00" + b"\xff" * (L - 2) + b"\x00"))
    return out


def test_masked_emulation_equals_numpy_for_every_search_cell():
    """Every kernel-model search case run through the emulated masked kernel: the target tile reports exactly the
    masked matches numpy finds over the oracle-deciphered entry in the starts the tile owns."""
    rng = np.random.default_rng(14)
    checked = 0
    for case in _find_cases():
        la, r = case.target_tile()
        so, ln, key = case.descs[case.target]
        plain = oracle.cycle(case.image[so:so + ln], key)
        mem = case.memory()
        L = len(case.pattern)
        base = km.TILE_BYTES * r.tin - r.h0
        _, head, p_end = km.scan_bounds(r, L)
        for name, mask in _masks(L, rng):
            value = bytes(v & m for v, m in zip(case.pattern, mask))
            want = [p - base for p in kmm.masked_positions(plain, value, mask) if base + head <= p < base + p_end]
            got = kmm.emulate_masked_find_tile(la, r, mem, value, mask)
            assert got == want, (case.cell, name)
            # stale bytes are only read by the filter: the result does not depend on them
            assert kmm.emulate_masked_find_tile(la, r, mem, value, mask, stale=0x00) == want
            checked += 1
    assert checked > 3 * len(_find_cases())


def test_masked_filter_has_no_false_negative():
    """A start whose anchor pair matches under the mask is always flagged, whatever the other bytes hold."""
    rng = np.random.default_rng(3)
    for _ in range(2000):
        L = int(rng.integers(1, 65))
        mask = bytes(rng.choice(np.array([0, 0xF0, 0x0F, 0xDF, 0xFF], np.uint8), size=L))
        if not any(mask):
            continue
        value = bytes(int(v) & m for v, m in zip(rng.integers(0, 256, L), mask))
        a = kmm.find_anchor(mask)
        sw = rng.integers(0, 256, size=64 + 16, dtype=np.uint8)
        o = int(rng.integers(0, 4))
        for k in (a, a + 1) if L > 1 else (a,):
            sw[o + k] = (value[k] & mask[k]) | (int(sw[o + k]) & ~mask[k] & 0xFF)
        assert kmm.masked_filter_word(sw, 0, value, mask) & (0x80 << (8 * o)), (L, mask.hex(), o)


@pytest.mark.parametrize("byte", [0x40, 0x60, 0x5B, 0x7B, 0xC1, 0xE1, 0xDF, 0xFF, 0x5F, 0x7F])
def test_fold_leaves_non_letters_alone(byte):
    assert kmm.fold(byte) == byte


def test_folded_set_bitmap_flags_exactly_the_case_variants():
    pats = [b"Ab", b"zz", b"@`", b"q", b"[x", b"\xe1a"]
    bm = kmm.fold_set_bitmap(pats)
    keys = np.arange(65536)
    b0, b1 = keys & 0xFF, keys >> 8
    f0 = np.array([kmm.fold(int(x)) for x in range(256)])[b0]
    f1 = np.array([kmm.fold(int(x)) for x in range(256)])[b1]
    want = np.zeros(65536, bool)
    for p in pats:
        q = bytes(kmm.fold(c) for c in p)
        want |= (f0 == q[0]) & ((f1 == q[1]) if len(q) > 1 else True)
    assert (bm == want).all()
    assert bm[0x40 | 0x60 << 8] and not bm[0x60 | 0x60 << 8]  # '@' and '`' do not fold
