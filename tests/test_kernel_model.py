"""CPU checks of tests/kernel_model.py, the host model of the cipher kernels' dispatch: its keystream
math against the oracle, its redo predicate against the bytes it would spoil, and the cell matrix that
tests/test_gpu_kernel_paths.py runs on the GPU."""
import functools

import numpy as np
import pytest

import kernel_model as km
import oracle
import synth


def test_geometry_is_parsed_from_the_kernel_header():
    assert km.THREADS > 0 and km.THREADS % 32 == 0
    assert km.UNROLL > 0 and km.CHUNKS <= 2048  # TileRec::geom holds the chunk count in 12 bits
    assert km.TILE_BYTES == 16 * km.THREADS * km.UNROLL
    assert km.EDGE_ROUNDS in (0, 1) and km.GENERAL_FULL in (0, 1)
    assert km.tiles_for_entry(0, km.TILE_BYTES) == 1 and km.tiles_for_entry(1, km.TILE_BYTES) == 2
    assert km.tiles_for_entry(15, (1 << 32) - 1) - 1 < km.TW0 * km.TW1  # the last tile of the longest entry


@pytest.mark.parametrize("key", synth.EDGE_KEYS + [0x12345678, 0x2468ACE1, 0x9E3779B9, 0x00000002])
def test_canonical_keystream_equals_oracle(key):
    """Tile state (c_ainv, c_tw0, c_tw1), chunk jump (g_chunk_pow2) and exact steps give the reference's
    keystream for every chunk of the tile, at every chunk-grid offset h0, up to the top of c_tw1."""
    n0 = km.key_to_neg_state(key)
    chunks = np.arange(km.CHUNKS)
    for tin in (0, 1, 1023, 1024, 1 << 19):
        states = np.array([km.tile_start_state(n0, h0, tin) for h0 in range(16)], np.uint64)
        got = km.canonical_bytes(km.chunk_states(states[:, None], chunks[None, :])).reshape(16, -1)
        for h0 in range(16):
            pos = km.TILE_BYTES * tin - h0
            skip = max(0, -pos)  # bytes before the entry's first byte
            want = oracle.cycle_at(np.zeros(km.TILE_BYTES - skip, np.uint8), key, pos + skip)
            assert (got[h0, skip:] == want).all(), (hex(key), tin, h0)


def test_speculative_bytes_differ_from_oracle_exactly_where_bit31_is_set():
    """The hot loop's bytes are the lazy low bytes; they are wrong exactly where a state has bit 31 set,
    so the redo predicate is "some byte would be wrong".  Also pins the trigger rates the kernel's
    comments quote."""
    rng = np.random.default_rng(11)
    n_tiles = 3000
    keys = [int(k) for k in rng.integers(1, km.M, size=n_tiles)]
    tins = rng.integers(0, 1 << 19, size=n_tiles)
    states = np.array([km.tile_start_state(km.key_to_neg_state(k), 0, int(t)) for k, t in zip(keys, tins)], np.uint64)
    # plus tiles made to trigger in a chosen chunk, so the comparison sees many triggers
    forced = km.find_tile_state(300, 0, 16, rng)[:40]
    s = km.chunk_states(states[:, None], np.arange(km.CHUNKS)[None, :])
    trig = km.triggers(s)
    spec = km.speculative_bytes(s).reshape(n_tiles, -1)
    flat = trig.reshape(n_tiles, -1)
    for i in list(np.nonzero(flat.any(axis=1))[0]) + list(range(20)):
        want = oracle.cycle_at(np.zeros(km.TILE_BYTES, np.uint8), keys[i], km.TILE_BYTES * int(tins[i]))
        assert ((spec[i] != want) == flat[i]).all(), i
    for st in forced:
        key = km.key_for_state(int(st), 0, 5)
        sf = km.chunk_states(np.uint64(st), np.arange(km.CHUNKS))
        want = oracle.cycle_at(np.zeros(km.TILE_BYTES, np.uint8), key, km.TILE_BYTES * 5)
        assert ((km.speculative_bytes(sf).reshape(-1) != want) == km.triggers(sf).reshape(-1)).all()
        assert km.triggers(sf)[300].any()
    chunk_rate = trig.any(axis=2).mean()
    thread_rate = trig.any(axis=2).reshape(n_tiles, km.UNROLL, km.THREADS).any(axis=1).mean()
    tile_rate = trig.any(axis=(1, 2)).mean()
    print(f"\nredo trigger rates: 1 chunk in {1 / chunk_rate:.0f}, 1 thread in {1 / thread_rate:.0f}, "
          f"1 tile in {1 / tile_rate:.1f}")
    assert 10_000 < 1 / chunk_rate < 20_000  # the kernel's comments: ~1 chunk in 14 000
    assert 2_500 < 1 / thread_rate < 5_000   # ~1 thread in 3 600


def test_cell_matrix_matches_enumeration():
    """Every cell the model declares unreachable is unreachable for every source / destination residue over
    a sweep of lengths and placements, and every other cell is reached by some geometry."""
    declared = km.reachable_cells()
    for kind in km.KINDS:
        got = km.enumerate_reachable(kind)
        assert got == {c for c in declared if c[0] == kind}, (kind, sorted(got ^ {c for c in declared if c[0] == kind}))
    # a contiguous call's bounds are its own extent: its partial chunks that read whole granules are the ones
    # either side of a 1 GiB piece boundary, and the chunk that ends a piece is alone in its tile
    assert ("inline", "coal/U4-partial", "head") in declared and ("inline", "gen/partial/ws3", "tail") in declared
    assert ("inline", "coal/U1", "tail") in declared and ("inline", "coal/U2", "tail") not in declared
    assert ("inline-inplace", "gen/partial/ws0", "none") not in declared
    assert ("batch", "gen/partial/ws3", "head") in declared and ("window", "coal/U2", "tail") in declared


def test_gpu_cases_cover_every_reachable_cell():
    """The launches of tests/test_gpu_kernel_paths.py, classified by the model: each reaches its cell, and a
    redo cell puts a trigger byte inside its entry (so a skipped or wrong redo changes a stored byte).
    Entries stay within 64 KiB, but for contiguous calls that must cross a 1 GiB piece boundary."""
    cases = km.cases()
    covered = set()
    for case in cases:
        kind, path, trig = case.cell
        one_piece = max(d[2] for d in case.descs) <= 64 << 10
        assert one_piece or kind.startswith("inline") and case.descs[0][2] <= km.MAX_PIECE + (64 << 10)
        models = [km.model_tile(la, r) for la, r in case.tiles()]
        covered |= {(kind, m.path, t) for m in models for t in m.cells()}
        hits = [m for m in models if case.is_target(m.rec) and m.path == path and trig in m.cells()]
        assert hits, case.cell
        if trig in ("none", "ghost") or path.endswith("/slow"):
            continue
        m = hits[0]
        inside = [eb for idx, b, eb in m.trigger_bytes() if 0 <= eb < m.rec.length]
        assert inside, case.cell
    assert covered >= km.reachable_cells()
    assert {c.dst_align for c in cases if c.kind == "batch"} >= {0, 1, 7, 8, 15}

    rows = sorted({(k, p) for k, p, _ in km.all_cells()})
    print("\ncell matrix (x: GPU case, -: unreachable)")
    print(f"{'':34}" + " ".join(f"{t:>10}" for t in km.TRIGGERS))
    for k, p in rows:
        marks = ["x" if (k, p, t) in covered else "-" for t in km.TRIGGERS]
        print(f"{k + ' ' + p:34}" + " ".join(f"{m:>10}" for m in marks))


def test_entries_with_trigger_bytes_equals_byte_compare():
    """entries_with_trigger_bytes flags exactly the entries whose speculative bytes differ from the oracle."""
    rng = np.random.default_rng(3)
    n = 300
    sizes = rng.integers(1, 20_000, size=n)
    off = synth.packed_offsets(sizes)
    keys = synth.entry_keys(n, seed=9)
    descs = [(int(o), int(o), int(s), int(k)) for o, s, k in zip(off, sizes, keys)]
    flagged = set(km.entries_with_trigger_bytes(descs, tiles_per_pass=7).tolist())
    want = set()
    for e, (so, do, ln, key) in enumerate(descs):
        spec = []
        for r in km.plan_tiles([descs[e]], 0):
            s = km.chunk_states(np.uint64(r.state), np.arange(r.n_valid))
            spec.append(km.speculative_bytes(s).reshape(-1))
        h0 = do & 15
        spec = np.concatenate(spec)[h0:h0 + ln]
        if (spec != oracle.keystream(key, ln)).any():
            want.add(e)
    assert flagged == want and len(want) > 0


# ---- the search kernel (find_batch_kernel) ---------------------------------------------------------------

def test_search_geometry_is_parsed_from_the_kernel_header():
    assert km.MAX_PATTERN == 64 and km.HALO_CHUNKS == (km.MAX_PATTERN - 1 + 15) // 16
    assert km.CHUNK_POW2.size == km.CHUNKS + km.HALO_CHUNKS  # g_chunk_pow2, then c_halo_pow2


@pytest.mark.parametrize("L", [1, 2, 3, 4, 5, 16, 17, 63, 64])
def test_tile_start_ranges_partition_the_entry(L):
    """The tiles' start ranges [head, p_end), in entry positions, are exactly [0, len - L + 1): no start is lost
    at a tile end or the entry end, none is taken by two tiles."""
    for h0 in range(16):
        lengths = set(range(1, 3 * L + 3))
        for b in (km.TILE_BYTES, 2 * km.TILE_BYTES, 3 * km.TILE_BYTES):
            lengths |= {b - h0 + d for d in range(-L - 1, L + 2)}
        for length in sorted(x for x in lengths if x > 0):
            seen = np.zeros(length, np.int8)
            for r in km.plan_tiles([(h0, h0, length, None)], 0):
                _, lo, p_end = km.scan_bounds(r, L)
                base = km.TILE_BYTES * r.tin - h0
                if p_end > lo:
                    seen[base + lo:base + p_end] += 1
            assert (seen[:max(0, length - L + 1)] == 1).all() and not seen[max(0, length - L + 1):].any(), (L, h0, length)


@pytest.mark.parametrize("key", synth.EDGE_KEYS + [0x12345678, 0x9E3779B9])
def test_halo_keystream_equals_oracle(key):
    """c_halo_pow2: halo chunk k of tile t is the stream's chunk 512 k later, exactly as the oracle has it."""
    n0 = km.key_to_neg_state(key)
    halo = np.arange(km.CHUNKS, km.CHUNKS + km.HALO_CHUNKS)
    for tin in (0, 1, 1023, (1 << 19) - 1):
        for h0 in range(16):
            st = km.tile_start_state(n0, h0, tin)
            got = km.canonical_bytes(km.chunk_states(np.uint64(st), halo)).reshape(-1)
            want = oracle.cycle_at(np.zeros(got.size, np.uint8), key, km.TILE_BYTES * (tin + 1) - h0)
            assert (got == want).all(), (hex(key), tin, h0)


@functools.lru_cache(maxsize=None)
def _find_cases():
    return km.find_cases()


def _tile_oracle(case):
    """Entry positions of the target's true matches whose start the target tile owns."""
    la, r = case.target_tile()
    so, ln, key = case.descs[case.target]
    plain = oracle.cycle(case.image[so:so + ln], key)
    L = len(case.pattern)
    lo, hi = max(0, km.TILE_BYTES * r.tin - r.h0), min(ln - L + 1, km.TILE_BYTES * (r.tin + 1) - r.h0)
    if hi <= lo:
        return []
    win = np.lib.stride_tricks.sliding_window_view(plain[lo:hi + L - 1], L)
    return [lo + int(p) for p in np.nonzero((win == np.frombuffer(case.pattern, np.uint8)).all(axis=1))[0]]


def test_find_emulation_equals_oracle_and_every_guard_and_redo_matters():
    """For every GPU case: the emulated tile with every guard on finds exactly the oracle's matches; with the
    case's guard dropped its decoy is counted as well; without the redo (or with the redo from round 0's state,
    for a ghost cell) the count changes."""
    for case in _find_cases():
        la, r = case.target_tile()
        mem = case.memory()
        base = km.TILE_BYTES * r.tin - r.h0
        got = [base + p for p in km.emulate_find_tile(la, r, mem, case.pattern)]
        assert got == _tile_oracle(case), case.cell
        kind, path, cell = case.cell
        if cell in km.GUARD_CELLS:
            off = tuple(g for g in km.GUARDS if g != km.GUARD_OF[cell])
            bad = km.emulate_find_tile(la, r, mem, case.pattern, guards=off)
            assert set(case.decoys) <= set(bad) - {p - base for p in got}, case.cell
        elif cell.startswith("halo"):
            continue  # the halo is always exact; the GPU cases plant a match over its triggering byte
        elif cell != "none":
            mode = "round0" if cell == "ghost" else "off"
            assert km.emulate_find_tile(la, r, mem, case.pattern, redo=mode) != [p - base for p in got], case.cell


def test_find_cells_match_the_sweep_and_the_cases_cover_them():
    declared = km.reachable_find_cells()
    for kind in km.FIND_KINDS:
        got = km.enumerate_reachable_find(kind)
        assert got == {c for c in declared if c[0] == kind}, (kind, sorted(got ^ {c for c in declared if c[0] == kind}))
    covered = set()
    for case in _find_cases():
        cells = case.cells()
        assert case.cell in cells, case.cell
        covered |= cells
    assert covered >= declared
    print("\nsearch cell matrix (x: GPU case, -: unreachable)")
    print(f"{'':16}" + " ".join(f"{c:>11}" for c in km.FIND_CELLS))
    for k in km.FIND_KINDS:
        for p in km.FIND_PATHS:
            print(f"{k + ' ' + p:16}" + " ".join(f"{'x' if (k, p, c) in covered else '-':>11}" for c in km.FIND_CELLS))
