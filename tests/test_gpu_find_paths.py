"""GPU: the search kernel (find_batch_kernel) over its path matrix, its compare and filter, its result buffers, its
window and alignment checks and its largest entry, against numpy over the oracle-deciphered entries.

One launch per (kind, load path, cell) that tests/kernel_model.py finds reachable: redo triggers and halo
triggers come from keys the model's backward search picks, with a match planted over the triggering byte (and,
where the tile has a second trigger, a false match that only a skipped redo reports).  Guard cells plant a
decoy in the bytes the CTA deciphers but does not own -- chunk 0 before the entry, the last chunk after it, the
zero-filled end of the halo, the next tile -- written in cipher space so that the tile holds the pattern there:
the kernel must not count it."""
import numpy as np
import pytest

import kernel_model as km
import oracle
import modulate_b200 as mb
from gpuutil import DeviceBuffer, Results, aligned_buffer, cases_by_cell, decipher_entries, model_descs, sync
from searchutil import MOD_ERR_ALIGN, MOD_ERR_ARG, search_one

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("cell", sorted(km.reachable_find_cells()), ids=lambda c: "-".join(c))
def test_find_path_cell(mb, cell):
    case = cases_by_cell()[cell]
    assert cell in case.cells()
    pat = case.pattern
    want, want_counts = search_one(decipher_entries(case.descs, case.image), pat)
    mem = case.memory()
    buf = aligned_buffer(mem)
    try:
        if case.kind == "batch":
            counts, matches, total = mb.find_batch(model_descs(case.descs), buf.ptr + case.src_ptr, pat,
                                                   src_bytes=case.image_bytes, max_matches=1 << 16)
            matches = [(int(a), int(b)) for a, b in zip(matches["desc"], matches["pos"])]
        else:
            t0, t1, wp, wo, wb = case.win
            lo, hi = case.entry_starts()
            want = [(d, p) for d, p in want if d == case.target and lo <= p < hi]
            want_counts = np.zeros(len(case.descs), np.uint32)
            want_counts[case.target] = len(want)
            plan = mb.Plan(model_descs(case.descs), case.image_bytes, case.image_bytes, case.dst_align)
            res = Results(len(case.descs), 1 << 12)
            plan.find_window(t0, t1, buf.ptr + wp, wo, wb, pat, res.counts, res.matches, res.cap, res.total)
            sync()
            total, counts, matches = res.read()
            matches.sort()
            plan.close()
    finally:
        buf.free()
    assert total == len(want) and counts.tolist() == want_counts.tolist() and matches == want, cell
    la, r = case.target_tile()
    base = km.TILE_BYTES * r.tin - r.h0
    own = [p for d, p in want if d == case.target and base + r.head <= p < base + km.scan_bounds(r, case.L)[2]]
    assert own == [base + p for p in km.emulate_find_tile(la, r, mem, pat)]


# ---- compare and filter -----------------------------------------------------------------------------------

SPECIAL = (0x00, 0x01, 0x7F, 0x80, 0xFE, 0xFF)
MATRIX_LENGTHS = [1, 2, 3, 4, 5, 8, 15, 16, 17, 32, 33, 48, 63, 64]
ENTRY = 5 * km.TILE_BYTES - 900


def _matrix_pattern(kind, L, rng):
    if kind == "random":
        return rng.integers(0, 256, size=L, dtype=np.uint8)
    if kind == "special":
        return np.array([SPECIAL[(i * 5 + L) % len(SPECIAL)] if i % 3 != 2 else rng.integers(0, 256) for i in range(L)],
                        np.uint8)
    if kind == "one-byte":
        return np.full(L, 0x80 if L % 2 else 0x01, np.uint8)
    return np.array([(0xFE, 0x7F)[i % 2] for i in range(L)], np.uint8)  # period 2


def _matrix_entry(pat, h0, e, rng):
    """Plain bytes of one entry at chunk-grid offset h0: random, with the pattern at the first and last start,
    straddling tile ends into halo chunk (e + k) % n_halo, near misses, and a long run of pattern[0]."""
    L = pat.size
    plain = rng.integers(0, 256, size=ENTRY, dtype=np.uint8)
    plain[0:L] = pat
    plain[ENTRY - L:] = pat
    n_halo = max(1, (L - 2) // 16 + 1)
    for k in (1, 2, 3):
        j = (e + k) % n_halo
        last = k * km.TILE_BYTES - h0 + 16 * j + min(15, max(0, L - 2 - 16 * j))
        plain[last - L + 1:last + 1] = pat
    # near misses: every proper prefix then a wrong byte, every single-byte substitution (^0x01, ^0x80)
    at = 3 * km.TILE_BYTES + 700
    misses = []
    for j in range(L):
        w = pat.copy()
        w[j] ^= 0x01 if j % 2 else 0x80
        misses.append(w[:j + 1])
        for x in (0x01, 0x80):
            w = pat.copy()
            w[j] ^= x
            misses.append(w)
    for w in misses:
        plain[at:at + w.size] = w
        at += w.size + 1 + (at & 3)
        assert at < ENTRY - 200
    plain[200:200 + 70] = pat[0]  # every start of these words passes the filter
    plain[300:300 + 2 * L] = np.tile(pat, 2)  # back to back
    return plain


@pytest.mark.parametrize("kind", ["random", "special", "one-byte", "period2"])
@pytest.mark.parametrize("L", MATRIX_LENGTHS)
def test_compare_and_filter_matrix(mb, L, kind):
    """Every pattern length the filter and the exact compare treat differently, at all 16 chunk-grid offsets:
    planted matches at the first and last start and across tile ends into every halo chunk, near misses that
    differ in one byte (the SWAR borrow and high-bit cases included), and runs that flag every start of a word."""
    rng = np.random.default_rng(1000 * L + len(kind))
    pat = _matrix_pattern(kind, L, rng)
    src_ptr = L % 16
    plains, descs, off = [], [], 40
    for h0 in range(16):
        off += (h0 - src_ptr - off) & 15
        plains.append(_matrix_entry(pat, h0, h0, rng))
        descs.append((off, ENTRY, int(rng.integers(1, 1 << 32)) - (1 << 31)))
        off += ENTRY + 3
    image = rng.integers(0, 256, size=off + 40, dtype=np.uint8)
    for (so, ln, key), p in zip(descs, plains):
        image[so:so + ln] = oracle.cycle(p, key)
    want, want_counts = search_one(plains, pat.tobytes())
    buf = aligned_buffer(np.concatenate([np.zeros(src_ptr, np.uint8), image]))
    counts, matches, total = mb.find_batch(model_descs(descs), buf.ptr + src_ptr, pat.tobytes(), src_bytes=image.size,
                                           max_matches=1 << 20)
    buf.free()
    got = [(int(a), int(b)) for a, b in zip(matches["desc"], matches["pos"])]
    assert total == len(want) and counts.tolist() == want_counts.tolist(), (L, kind)
    assert got == want, (L, kind, sorted(set(got) ^ set(want))[:10])


# ---- result buffers -----------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def many_matches():
    rng = np.random.default_rng(8)
    sizes = [int(s) for s in rng.integers(1, 30000, size=25)]
    plains = [rng.integers(0, 4, size=s, dtype=np.uint8) for s in sizes]
    descs, off = [], 0
    for s in sizes:
        descs.append((off, s, int(rng.integers(1, 1 << 31))))
        off += s
    image = np.zeros(off, np.uint8)
    for (so, ln, key), p in zip(descs, plains):
        image[so:so + ln] = oracle.cycle(p, key)
    return descs, image, plains


@pytest.mark.parametrize("which", ["0", "1", "n-1", "n", "n+1"])
def test_cap_keeps_exact_counts_and_lists_true_matches(mb, many_matches, which):
    descs, image, plains = many_matches
    pat = b"\x01\x02\x03"
    want, want_counts = search_one(plains, pat)
    n = len(want)
    cap = {"0": 0, "1": 1, "n-1": n - 1, "n": n, "n+1": n + 1}[which]
    buf = aligned_buffer(image)
    plan = mb.Plan(model_descs(descs), image.size, image.size, 0)
    res = Results(len(descs), cap)
    plan.find(buf.ptr, pat, res.counts, res.matches if cap else 0, cap, res.total)
    sync()
    total, counts, matches = res.read()
    assert total == n and counts.tolist() == want_counts.tolist()
    assert len(matches) == min(cap, n) and len(set(matches)) == len(matches) and set(matches) <= set(want)
    plan.find(buf.ptr, pat, res.counts, res.matches if cap else 0, cap, res.total)  # results accumulate
    sync()
    total, counts, _ = res.read()
    assert total == 2 * n and counts.tolist() == (2 * want_counts).tolist()
    plan.close()
    buf.free()


# ---- window bounds and the chunk grid -------------------------------------------------------------------------

@pytest.mark.parametrize("L", [1, 64])
def test_window_bounds_inside_an_entry(mb, L):
    """A tile range that starts and ends inside an entry: the minimal window (the tile's bytes plus L - 1) is
    accepted and gives exactly the starts the model assigns the tile; a window one byte short at either end is
    refused with MOD_ERR_ARG before anything runs."""
    rng = np.random.default_rng(L)
    h0, so, ln = 7, 1000, 4 * km.TILE_BYTES + 333
    pat = np.full(L, 0xA7, np.uint8)  # one byte value: plants may overlap and stay matches
    plain = rng.integers(0, 256, size=ln, dtype=np.uint8)
    for s in list(range(km.TILE_BYTES - h0 - L - 2, km.TILE_BYTES - h0 + 3)) + [2 * km.TILE_BYTES - h0 - L,
                                                                                  2 * km.TILE_BYTES - h0 - L + 1]:
        plain[s:s + L] = pat  # the last starts of tile 0, the first of tile 1, the last of tile 1
    key = 0x31415926
    descs = [(so, ln, key)]
    dst_align = (h0 - so) & 15
    image = rng.integers(0, 256, size=so + ln + 500, dtype=np.uint8)
    image[so:so + ln] = oracle.cycle(plain, key)
    plan = mb.Plan(model_descs(descs), image.size, image.size, dst_align)
    t0, t1 = 1, 3
    b0 = so + km.TILE_BYTES - h0
    b1 = so + 3 * km.TILE_BYTES - h0 + L - 1
    assert km.find_window_ok(descs, dst_align, t0, t1, b0, b1 - b0, L)
    la = km.find_window_launch(descs, dst_align, t0, t1, 0, b0, b1 - b0)
    lo = km.TILE_BYTES - h0
    starts = set()
    for r in la.tiles:
        _, a, p_end = km.scan_bounds(r, L)
        starts |= {km.TILE_BYTES * r.tin - h0 + p for p in range(a, p_end)}
    assert starts == set(range(lo, 3 * km.TILE_BYTES - h0))
    want = sorted((0, q) for _, q in search_one([plain], pat.tobytes())[0] if q in starts)
    for w_lo, w_hi, ok in ((b0, b1, True), (b0 + 1, b1, False), (b0, b1 - 1, False)):
        win_ptr = (w_lo + dst_align) & 15
        buf = aligned_buffer(np.concatenate([np.zeros(win_ptr, np.uint8), image[w_lo:w_hi]]))
        res = Results(1, 1 << 10)
        assert km.find_window_ok(descs, dst_align, t0, t1, w_lo, w_hi - w_lo, L) == ok
        if ok:
            plan.find_window(t0, t1, buf.ptr + win_ptr, w_lo, w_hi - w_lo, pat.tobytes(), res.counts, res.matches,
                             res.cap, res.total)
        else:
            with pytest.raises(mb.ModError) as err:
                plan.find_window(t0, t1, buf.ptr + win_ptr, w_lo, w_hi - w_lo, pat.tobytes(), res.counts, res.matches,
                                 res.cap, res.total)
            assert err.value.code == MOD_ERR_ARG
        sync()
        total, counts, matches = res.read()
        if ok:
            assert sorted(matches) == want and total == len(want) and len(want) >= 4
        else:
            assert total == 0 and not counts.any()
        buf.free()
    plan.close()


def test_plans_off_the_source_grid_are_refused(mb):
    """mod_plan_find needs the chunk grid on the source: a plan built for another dst_align, or one whose
    descriptors disagree on (src_off - dst_off) mod 16, is refused with MOD_ERR_ALIGN; a delta that is a
    multiple of 16 keeps the grid on the source and gives the same matches."""
    rng = np.random.default_rng(4)
    plains = [rng.integers(0, 4, size=s, dtype=np.uint8) for s in (9000, 300, 20000)]
    descs, off = [], 5
    for p in plains:
        descs.append((off, p.size, int(rng.integers(1, 1 << 31))))
        off += p.size + 1
    image = np.zeros(off, np.uint8)
    for (so, ln, key), p in zip(descs, plains):
        image[so:so + ln] = oracle.cycle(p, key)
    pat = b"\x02\x03"
    want, want_counts = search_one(plains, pat)
    src_ptr = 3
    buf = aligned_buffer(np.concatenate([np.zeros(src_ptr, np.uint8), image]))
    so, ln, key = zip(*descs)
    key = [k & 0xFFFFFFFF for k in key]

    def run(dst_off, dst_align):
        plan = mb.Plan(mb.make_descs(list(so), dst_off, list(ln), key), image.size, image.size + 64, dst_align)
        res = Results(len(descs), 1 << 14)
        try:
            plan.find(buf.ptr + src_ptr, pat, res.counts, res.matches, res.cap, res.total)
            sync()
            total, counts, matches = res.read()
            return total, counts.tolist(), sorted(matches)
        finally:
            plan.close()

    ok = (len(want), want_counts.tolist(), want)
    assert run(list(so), src_ptr) == ok
    assert run([s + 16 for s in so], src_ptr) == ok            # delta 16 for every entry
    assert run([s + 32 * (i % 2) for i, s in enumerate(so)], src_ptr) == ok  # deltas 0 and 32: still on the grid
    for dst_off, dst_align in ((list(so), (src_ptr + 1) & 15),   # dst_align is not the source's
                               ([s + 1 for s in so], src_ptr),   # delta 1 moves the grid off the source
                               ([s + (i == 1) for i, s in enumerate(so)], src_ptr)):  # descriptors disagree
        with pytest.raises(mb.ModError) as err:
            run(dst_off, dst_align)
        assert err.value.code == MOD_ERR_ALIGN
    buf.free()


# ---- the largest entry ------------------------------------------------------------------------------------------

def test_largest_entry(mb):
    """One entry of 2^32 - 1 bytes at h0 = 15, enciphered on the GPU: the search returns exactly the planted
    positions -- near 0, around 2^31 (where a signed 32-bit position would turn negative), across the last two
    tile ends, and at len - L.  Match positions are 32-bit, computed from 64-bit tile offsets."""
    n = (1 << 32) - 1
    h0 = 15
    L = 17
    key = 0x0BADF00D
    rng = np.random.default_rng(17)
    pat = rng.integers(1, 256, size=L, dtype=np.uint8)
    last_tile = (h0 + n + 15) // 16 // km.CHUNKS * km.TILE_BYTES - h0  # entry byte where the last tile starts
    # n - L starts in the second-to-last tile and ends in the last one (a single chunk)
    plants = sorted({3, 100, (1 << 31) - 20, (1 << 31) - 1, (1 << 31) + 16, last_tile - km.TILE_BYTES - 9, n - L})
    assert n - L < last_tile < n
    assert all(b - a >= L for a, b in zip(plants, plants[1:]))
    buf = DeviceBuffer(h0 + n + 1)
    try:
        zero = np.zeros(256 << 20, np.uint8)
        for o in range(0, buf.nbytes, zero.size):
            buf.upload(zero[:min(zero.size, buf.nbytes - o)], o)
        for p in plants:
            buf.upload(pat, h0 + p)
        mb.cycle_device(buf.ptr + h0, buf.ptr + h0, n, key)
        sync()
        for p in plants + [0, 1 << 31, n - 4096]:
            lo = max(0, p - 40)
            hi = min(n, p + 4096)
            plain = np.zeros(hi - lo, np.uint8)
            for q in plants:
                a, b = max(q, lo), min(q + L, hi)
                if a < b:
                    plain[a - lo:b - lo] = pat[a - q:b - q]
            assert (buf.download(h0 + lo, hi - lo) == oracle.cycle_at(plain, key, lo)).all(), p
        descs = mb.make_descs([0], [0], [n], [key])
        counts, matches, total = mb.find_batch(descs, buf.ptr + h0, pat.tobytes(), src_bytes=n, max_matches=64)
        assert total == len(plants) and counts.tolist() == [len(plants)]
        assert [int(p) for p in matches["pos"]] == plants and set(matches["desc"].tolist()) == {0}
    finally:
        buf.free()
