"""GPU: the masked search (find_batch_kernel<true>: wildcard bytes and nibbles, ASCII case folding) and the
case-folded pattern sets (find_set_kernel<true>) against numpy over the oracle-deciphered entries: every kernel-model
search cell, a length / anchor / phase matrix with planted near misses, the fold's edge bytes, the result buffers and
windows, the refusals, the 1 GiB set, and the CLI on the CUDA library."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import arkfixture
import kernel_model as km
import kernel_model_masked as kmm
import oracle
import synth
import modulate_b200 as mb
from modulate_b200 import _abi
from gpuutil import DeviceBuffer, sync
from test_find_masked_host import check_nocase, check_nocase_set, check_wild
from test_find_host import piece_cut_archive
from test_gpu_find import CLI, build_source, shm_dir
from test_gpu_find_paths import Results, _buffer, _cases, _mdescs, _plain
from test_gpu_find_set import as_list

pytestmark = pytest.mark.gpu

MOD_ERR_ARG = -2
FOLD = np.array([kmm.fold(b) for b in range(256)], np.uint8)


def masked_find(plain_entries, value, mask):
    """numpy: matches (desc, pos) and counts per entry."""
    out = []
    for i, e in enumerate(plain_entries):
        out += [(i, p) for p in kmm.masked_positions(e, value, mask)]
    return out, np.bincount([d for d, _ in out], minlength=len(plain_entries)).astype(np.uint32)


def fold_mask(value: bytes) -> bytes:
    return bytes(0xDF if 0x41 <= b <= 0x5A else 0xFF for b in value)


def cell_masks(L):
    """(away, lead): one wildcard away from the anchor; leading wildcards that put the anchor pair at the pattern's
    end, so that for the starts near a tile's end it lies in the halo chunks."""
    if L == 1:
        return b"\x0f", b"\xf0"
    if L == 2:
        return b"\xff\xf0", b"\x00\xff"
    return b"\xff\xff" + b"\xff" * (L - 3) + b"\x00", bytes(L - 2) + b"\xff\xff"


@pytest.mark.parametrize("cell", sorted(km.reachable_find_cells()), ids=lambda c: "-".join(c))
def test_model_cases_through_the_masked_kernel(mb, cell):
    case = _cases()[cell]
    plain = _plain(case.descs, case.image)
    mem = case.memory()
    buf = _buffer(mem)
    la, r = case.target_tile()
    base = km.TILE_BYTES * r.tin - r.h0
    try:
        for mask in cell_masks(case.L):
            value = bytes(v & m for v, m in zip(case.pattern, mask))
            want, want_counts = masked_find(plain, value, mask)
            if case.kind == "batch":
                counts, matches, total = mb.find_batch(_mdescs(case.descs), buf.ptr + case.src_ptr, value,
                                                       src_bytes=case.image_bytes, max_matches=1 << 16, mask=mask)
                matches = [(int(a), int(b)) for a, b in zip(matches["desc"], matches["pos"])]
            else:
                t0, t1, wp, wo, wb = case.win
                lo, hi = case.entry_starts()
                want = [(d, p) for d, p in want if d == case.target and lo <= p < hi]
                want_counts = np.zeros(len(case.descs), np.uint32)
                want_counts[case.target] = len(want)
                plan = mb.Plan(_mdescs(case.descs), case.image_bytes, case.image_bytes, case.dst_align)
                res = Results(len(case.descs), 1 << 12)
                plan.find_window(t0, t1, buf.ptr + wp, wo, wb, value, res.counts, res.matches, res.cap, res.total, mask=mask)
                sync()
                total, counts, matches = res.read()
                matches.sort()
                plan.close()
            assert total == len(want) and counts.tolist() == want_counts.tolist() and matches == want, (cell, mask.hex())
            own = [p for d, p in want if d == case.target and base + r.head <= p < base + km.scan_bounds(r, case.L)[2]]
            assert own == [base + p for p in kmm.emulate_masked_find_tile(la, r, mem, value, mask)], (cell, mask.hex())
    finally:
        buf.free()


MATRIX_LENGTHS = [1, 2, 3, 5, 17, 63, 64]


def _anchored_mask(L, a, kind, rng):
    """A mask whose anchor is a: the pair (a, a + 1) exact, every other byte weaker (nibble, fold or wildcard)."""
    if kind == "fold":
        weak = np.array([0xDF, 0x00], np.uint8)
    else:
        weak = np.array([0xF0, 0x0F, 0x00], np.uint8)
    m = rng.choice(weak, size=L)
    m[a] = 0xFF
    if L > 1:
        m[a + 1] = 0xFF
    return bytes(m)


def _matrix_entries(value, mask, phase, rng, fold):
    """Entries holding matches with random masked-out bits (must match) and near misses that differ in one masked-in
    bit (must not), across chunk and tile boundaries."""
    L = len(value)
    sizes = [L, L - 1, 100, 8192 + 70, 3 * 8192 + 5, 20000, 16, 0]
    ents = [rng.integers(0, 256, size=s, dtype=np.uint8) for s in sizes]
    V, M = np.frombuffer(value, np.uint8), np.frombuffer(mask, np.uint8)
    for i, e in enumerate(ents):
        h0 = (phase + sum(sizes[:i])) & 15
        starts = {0, e.size - L}
        for b in list(range(16, e.size, 16 * 41)) + list(range(8192, e.size, 8192)):
            for j in (1, L // 2, L - 1):
                starts.add(b - h0 - j)
        for n, s in enumerate(sorted(starts)):
            if not (0 <= s and s + L <= e.size):
                continue
            free = rng.integers(0, 256, size=L, dtype=np.uint8)
            if fold:  # a letter in either case
                free = np.where(M == 0xDF, rng.choice(np.array([0, 0x20], np.uint8), size=L), free)
            w = (V & M) | (free & ~M)
            if n % 3 == 2:  # near miss: one masked-in bit flipped
                k = int(rng.choice(np.nonzero(M)[0]))
                bits = [b for b in range(8) if (M[k] >> b) & 1]
                w[k] ^= np.uint8(1 << int(rng.choice(bits)))
            e[s:s + L] = w
    return ents


@pytest.mark.parametrize("kind", ["nibble", "fold"])
@pytest.mark.parametrize("L", MATRIX_LENGTHS)
def test_length_anchor_phase_matrix(mb, L, kind):
    """Every anchor position of every length, all 16 source phases: planted matches with random masked-out bits are
    found, near misses in a masked-in bit are not, exactly as numpy says."""
    rng = np.random.default_rng(L * 7 + (kind == "fold"))
    anchors = range(max(1, L - 1))
    runs = [(a, (5 * a + L) % 16) for a in anchors] + [(a, ph) for a in {0, max(0, L - 2)} for ph in range(16)]
    for a, phase in runs:
        mask = _anchored_mask(L, a, kind, rng)
        assert kmm.find_anchor(mask) == a or L == 1
        if kind == "fold":
            value = bytes(int(x) for x in rng.integers(0x41, 0x5B, size=L))
        else:
            value = bytes(int(x) for x in rng.integers(0, 256, size=L))
        value = bytes(v & m for v, m in zip(value, mask))
        ents = _matrix_entries(value, mask, phase, rng, kind == "fold")
        keys = [int(k) for k in rng.integers(-(1 << 31), 1 << 31, size=len(ents))]
        descs, src = build_source(ents, keys, phase)
        buf = DeviceBuffer.from_numpy(src)
        try:
            counts, matches, total = mb.find_batch(descs, buf.ptr, value, src_bytes=src.size, max_matches=1 << 16, mask=mask)
        finally:
            buf.free()
        want, want_counts = masked_find(ents, value, mask)
        got = [(int(d), int(p)) for d, p in zip(matches["desc"], matches["pos"])]
        assert total == len(want) and got == want and counts.tolist() == want_counts.tolist(), (L, a, phase, mask.hex())
        assert total >= 4


@pytest.mark.parametrize("pair", [(0x40, 0x60), (0x5B, 0x7B), (0xC1, 0xE1), (0xDF, 0xFF), (0x5F, 0x7F)])
def test_fold_edge_bytes_do_not_fold(mb, pair):
    """Only A-Z / a-z fold: each byte of these pairs finds itself, never the other, through a fold-mask search and a
    folded set."""
    lo, hi = pair
    body = bytes([lo, 0x41, hi, 0x61, lo, hi]) * 40
    ents = [np.frombuffer(body, np.uint8).copy()]
    for b in (lo, hi):
        value, mask = mb.ignore_case_pattern(bytes([b, 0x61]))
        assert mask[0] == 0xFF
        want, _ = masked_find(ents, value, mask)
        descs, src = build_source(ents, [0x1234], 3)
        buf = DeviceBuffer.from_numpy(src)
        _, matches, total = mb.find_batch(descs, buf.ptr, value, src_bytes=src.size, mask=mask)
        assert total == len(want) == 40 and [(int(d), int(p)) for d, p in zip(matches["desc"], matches["pos"])] == want
        pset = mb.PatternSet([bytes([b, 0x61]), bytes([b])], ignore_case=True)
        plan = mb.Plan(descs, src.size, src.size, buf.ptr & 15)
        res = Results(1, 1 << 10)
        pc = DeviceBuffer.from_numpy(np.zeros(2, np.uint64))
        m = DeviceBuffer(12 << 10)
        plan.find_set(buf.ptr, pset, res.counts, pc.ptr, m.ptr, 1 << 10, res.total)
        sync()
        assert pc.download().view(np.uint64).tolist() == [40, int((ents[0] == b).sum())]
        for x in (plan, pset):
            x.close()
        for x in (buf, pc, m):
            x.free()


def _one_entry_plan(rng):
    ent = rng.integers(0, 256, size=3 * 8192 + 77, dtype=np.uint8)
    value, mask = b"\x13\x00\x37\x40\x05", b"\xff\x00\xff\xf0\xff"
    for s in range(100, ent.size - 5, 311):
        ent[s:s + 5] = (np.frombuffer(value, np.uint8) | (rng.integers(0, 256, 5, dtype=np.uint8) & ~np.frombuffer(mask, np.uint8)))
    descs, src = build_source([ent], [0x2468], 0)
    return ent, descs, src, value, mask


def test_cap_accumulation_and_windows(mb):
    rng = np.random.default_rng(9)
    ent, descs, src, value, mask = _one_entry_plan(rng)
    want, _ = masked_find([ent], value, mask)
    n = len(want)
    buf = DeviceBuffer.from_numpy(src)
    plan = mb.Plan(descs, src.size, src.size, buf.ptr & 15)
    for cap in (0, 1, n - 1, n, n + 1):
        res = Results(1, cap)
        plan.find(buf.ptr, value, res.counts, res.matches, cap, res.total, mask=mask)
        plan.find(buf.ptr, value, res.counts, res.matches, cap, res.total, mask=mask)  # accumulates
        sync()
        total, counts, matches = res.read()
        assert total == 2 * n and counts.tolist() == [2 * n]
        assert len(matches) == min(cap, 2 * n) and set(matches) <= set(want)
    # a window over tile 1 only: its bytes plus L - 1 halo bytes are needed
    L = len(value)
    h0 = buf.ptr & 15
    lo, hi = 8192 - h0, 2 * 8192 - h0 + L - 1
    res = Results(1, 1 << 10)
    plan.find_window(1, 2, buf.ptr + lo, lo, hi - lo, value, res.counts, res.matches, res.cap, res.total, mask=mask)
    sync()
    total, _, matches = res.read()
    assert sorted(matches) == [(0, p) for _, p in want if lo <= p < 2 * 8192 - h0]
    for wlo, whi in ((lo + 1, hi), (lo, hi - 1)):
        with pytest.raises(mb.ModError, match="reads outside the source window"):
            plan.find_window(1, 2, buf.ptr + wlo, wlo, whi - wlo, value, res.counts, res.matches, res.cap, res.total, mask=mask)
    plan.close()
    buf.free()


def test_refusals(mb):
    rng = np.random.default_rng(2)
    ent, descs, src, value, mask = _one_entry_plan(rng)
    buf = DeviceBuffer.from_numpy(src)
    plan = mb.Plan(descs, src.size, src.size, buf.ptr & 15)
    res = Results(1, 4)
    lib = _abi.load()
    assert lib.mod_plan_find_masked(plan._handle, buf.ptr, value, None, 5, res.counts, res.matches, 4, res.total, None) == MOD_ERR_ARG
    assert lib.mod_plan_find_masked(plan._handle, buf.ptr, value, bytes(5), 5, res.counts, res.matches, 4, res.total,
                                    None) == MOD_ERR_ARG
    for L in (0, 65):
        assert lib.mod_plan_find_masked(plan._handle, buf.ptr, b"\x01" * 65, b"\xff" * 65, L, res.counts, res.matches, 4,
                                        res.total, None) == MOD_ERR_ARG
    assert lib.mod_plan_find_masked_window(plan._handle, 0, 1, buf.ptr, 0, src.size, value, None, 5, res.counts, res.matches, 4,
                                           res.total, None) == MOD_ERR_ARG
    counts = np.zeros(1, np.uint32)
    total = ctypes.c_uint64()
    assert lib.mod_find_masked_batch(descs.ctypes.data, 1, buf.ptr, src.size, value, bytes(5), 5, counts.ctypes.data, None, 0,
                                     ctypes.byref(total)) == MOD_ERR_ARG
    assert lib.mod_find_masked_batch(descs.ctypes.data, 1, buf.ptr, src.size, value, None, 5, counts.ctypes.data, None, 0,
                                     ctypes.byref(total)) == MOD_ERR_ARG
    # an all-0xFF mask is the exact search
    assert mb.find_batch(descs, buf.ptr, value, src_bytes=src.size, mask=b"\xff" * 5)[2] == \
        mb.find_batch(descs, buf.ptr, value, src_bytes=src.size)[2]
    with pytest.raises(ValueError):
        mb.find_batch(descs, buf.ptr, value, src_bytes=src.size, mask=b"\xff" * 4)
    sync()
    assert res.read()[0] == 0
    plan.close()
    buf.free()


def _mixed_case(p, rng):
    return bytes(b ^ 0x20 if (0x41 <= (b & 0xDF) <= 0x5A and rng.integers(2)) else b for b in p)


def plain_find_set_nocase(ents, pats):
    out = []
    for i, e in enumerate(ents):
        fe = FOLD[e]
        for j, p in enumerate(pats):
            out += [(i, q, j) for q in kmm.masked_positions(fe, bytes(FOLD[np.frombuffer(p, np.uint8)]), b"\xff" * len(p))]
    out.sort()
    return out


@pytest.mark.parametrize("K", [1, 17, 256])
def test_folded_sets_against_numpy(mb, K):
    rng = np.random.default_rng(K)
    letters = np.frombuffer(b"AbCdEfGhIjKlMnOpQrStUvWxYz@[`{\xc1\xe1", np.uint8)
    pats, seen = [], set()
    while len(pats) < K:
        L = int(rng.choice([1, 2, 3, 4, 7, 17, 64])) if K > 1 else 5
        p = bytes(rng.choice(letters, size=L))
        if bytes(FOLD[np.frombuffer(p, np.uint8)]) not in seen:
            seen.add(bytes(FOLD[np.frombuffer(p, np.uint8)]))
            pats.append(p)
    ents = [rng.choice(letters, size=s).astype(np.uint8) for s in (1, 63, 64, 5000, 8192 + 100, 3 * 8192 + 9)]
    for e in ents:
        for s in range(0, e.size - 64, 997):
            p = pats[int(rng.integers(len(pats)))]
            e[s:s + len(p)] = np.frombuffer(_mixed_case(p, rng), np.uint8)
    keys = [int(k) for k in rng.integers(-(1 << 31), 1 << 31, size=len(ents))]
    for phase in (0, 7):
        descs, src = build_source(ents, keys, phase)
        buf = DeviceBuffer.from_numpy(src)
        try:
            pset = mb.PatternSet(pats, ignore_case=True)
            plan = mb.Plan(descs, src.size, src.size, buf.ptr & 15)
            cap = 1 << 18
            res = Results(len(ents), 1)
            pc = DeviceBuffer.from_numpy(np.zeros(K, np.uint64))
            m = DeviceBuffer(12 * cap)
            plan.find_set(buf.ptr, pset, res.counts, pc.ptr, m.ptr, cap, res.total)
            sync()
            total = res.read()[0]
            got = sorted(as_list(m.download().view(mb.SET_MATCH_DTYPE)[:total]))
            want = plain_find_set_nocase(ents, pats)
            assert total == len(want) and got == want, (K, phase)
            assert pc.download().view(np.uint64).tolist() == np.bincount([w[2] for w in want], minlength=K).tolist()
            for x in (plan, pset):
                x.close()
            for x in (pc, m):
                x.free()
        finally:
            buf.free()


def test_folded_set_prefixes_letters_and_refusals(mb):
    rng = np.random.default_rng(5)
    ents = [np.frombuffer(b"aB1 Ab2 AB1 ab2 x X y ~ @ ` " * 50, np.uint8).copy(),
            rng.integers(0, 256, size=9000, dtype=np.uint8)]
    keys = [11, -5]
    # prefixes that differ only in case are one key; length-1 letters take both rows
    pats = [b"ab1", b"AB2", b"x", b"@"]
    descs, src = build_source(ents, keys, 2)
    buf = DeviceBuffer.from_numpy(src)
    pset = mb.PatternSet(pats, ignore_case=True)
    plan = mb.Plan(descs, src.size, src.size, buf.ptr & 15)
    res = Results(2, 1)
    pc = DeviceBuffer.from_numpy(np.zeros(4, np.uint64))
    m = DeviceBuffer(12 << 14)
    plan.find_set(buf.ptr, pset, res.counts, pc.ptr, m.ptr, 1 << 14, res.total)
    sync()
    total = res.read()[0]
    want = plain_find_set_nocase(ents, pats)
    assert sorted(as_list(m.download().view(mb.SET_MATCH_DTYPE)[:total])) == want
    assert pc.download().view(np.uint64).tolist() == np.bincount([w[2] for w in want], minlength=4).tolist()
    assert sum(1 for w in want if w[0] == 0 and w[2] < 2) == 200  # aB1 AB1 / Ab2 ab2
    for x in (plan, pset):
        x.close()
    for x in (pc, m):
        x.free()
    # a one-pattern folded set equals the masked search with the fold mask
    for p in (b"Ab1", b"x", b"AB2 "):
        value, mask = mb.ignore_case_pattern(p)
        c1, m1, t1 = mb.find_batch(descs, buf.ptr, value, src_bytes=src.size, mask=mask)
        s = mb.PatternSet([p], ignore_case=True)
        plan = mb.Plan(descs, src.size, src.size, buf.ptr & 15)
        r2 = Results(2, 1)
        pc = DeviceBuffer.from_numpy(np.zeros(1, np.uint64))
        m2 = DeviceBuffer(12 << 12)
        plan.find_set(buf.ptr, s, r2.counts, pc.ptr, m2.ptr, 1 << 12, r2.total)
        sync()
        t2, c2, _ = r2.read()
        got = sorted((d, q) for d, q, _ in as_list(m2.download().view(mb.SET_MATCH_DTYPE)[:t2]))
        assert t2 == t1 and c2.tolist() == c1.tolist() and got == [(int(d), int(q)) for d, q in zip(m1["desc"], m1["pos"])]
        plan.close()
        s.close()
        pc.free()
        m2.free()
    buf.free()
    # duplicates after folding are refused, by the library and by the Python check
    lib = _abi.load()
    h = ctypes.c_void_p()
    data = np.frombuffer(b"AbaB", np.uint8)
    assert lib.mod_pattern_set_create_nocase(data.ctypes.data, np.array([2, 2], np.uint32).ctypes.data, 2,
                                             ctypes.byref(h)) == MOD_ERR_ARG
    assert lib.mod_pattern_set_create(data.ctypes.data, np.array([2, 2], np.uint32).ctypes.data, 2, ctypes.byref(h)) == 0
    lib.mod_pattern_set_destroy(h)
    with pytest.raises(ValueError):
        mb.PatternSet([b"Ab", b"aB"], ignore_case=True)


def test_one_gib_ten_thousand_entries_fold_and_wildcard_against_numpy(mb):
    sizes = synth.entry_sizes_loguniform(10000, 1 << 30, seed=7)
    src_off = synth.packed_offsets(sizes)
    keys = synth.entry_keys(len(sizes))
    descs = mb.make_descs(src_off, src_off, sizes, keys)
    n = int(src_off[-1] + sizes[-1])
    src = synth.payload(0, n)
    plain = np.empty_like(src)
    for o, s, k in zip(src_off, sizes, keys):
        plain[o:o + s] = oracle.cycle(src[o:o + s], int(k))
    text = b"aMpLiTuDe"
    for i in range(0, 10000, 499):
        o, s = int(src_off[i]), int(sizes[i])
        if s < 64:
            continue
        p = o + s // 2
        plain[p:p + 9] = np.frombuffer(_mixed_case(text, np.random.default_rng(i)), np.uint8)
        plain[p + 20:p + 24] = np.frombuffer(bytes([0x13, i & 0xFF, 0x37, 0x40 | (i & 15)]), np.uint8)
        src[o:o + s] = oracle.cycle(plain[o:o + s], int(keys[i]))
    buf = DeviceBuffer.from_numpy(src)
    ends = src_off + sizes
    try:
        for value, mask in (mb.ignore_case_pattern(text), mb.wildcard_pattern("13 ?? 37 4?")):
            L = len(value)
            hit = np.ones(n - L + 1, bool)
            for j in range(L):
                hit &= (plain[j:n - L + 1 + j] & mask[j]) == value[j]
            pos = np.nonzero(hit)[0]
            d = np.searchsorted(src_off, pos, side="right") - 1
            keep = pos + L <= ends[d]
            want = sorted(zip(d[keep].tolist(), (pos[keep] - src_off[d[keep]]).tolist()))
            counts, matches, total = mb.find_batch(descs, buf.ptr, value, src_bytes=n, max_matches=1 << 20, mask=mask)
            assert total == len(want) >= 15 and [(int(a), int(b)) for a, b in zip(matches["desc"], matches["pos"])] == want
            assert (np.bincount(d[keep], minlength=len(sizes)) == counts).all()
    finally:
        buf.free()


@pytest.mark.parametrize("L", [1, 2, 17, 64])
def test_cli_over_pieces_on_every_gpu(tmp_path, L):
    """-findwild, -findi and -findilist through the CLI on the CUDA library, with 1 MiB groups (pieces overlapping by
    L - 1 bytes) and with every GPU."""
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    pat, key = piece_cut_archive(tmp_path, L)
    mask = b"\x0f" if L == 1 else b"\x00\xff" if L == 2 else b"\x00" + b"\xff" * (L - 2) + b"\x00"
    all_gpus = hex((1 << mb.device_count()) - 1)
    for env in (dict(os.environ, MOD_IO_GROUP_MIB="1"), dict(os.environ, MOD_IO_GROUP_MIB="1", MOD_DEVICES=all_gpus)):
        assert check_wild(CLI, tmp_path, "ps4", pat, mask, key=key, env=env)[1] >= 8
    assert check_wild(CLI, tmp_path, "ps4", pat, mask, key=key)[1] >= 8


def test_cli_text_commands_on_the_cuda_library(tmp_path):
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    contents = {0: b"Amplitude AMPLITUDE amplitude aMpLiTuDe", 1: b"@`[{\xc1\xe1\xdf\xff_\x7f" * 3, 2: b"symbol SYMBOL"}
    arkfixture.write_archive(str(tmp_path), n_files=40, n_parts=2, seed=7, sizes=[len(contents[0]), 30, 13] + [5000] * 37,
                             contents=contents)
    assert check_nocase(CLI, tmp_path, "ps4", b"amplitude")[1] >= 4
    for b in (b"@", b"`", b"\xc1", b"\xdf"):
        check_nocase(CLI, tmp_path, "ps4", b)
    assert check_nocase_set(CLI, tmp_path, "ps4", [b"AMPLITUDE", b"sym", b"s", b"@`", b"\xc1", b"q"]) >= 8


def test_large_archive_cli_on_every_gpu(tmp_path):
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    root = shm_dir(tmp_path)
    try:
        key = 0x5EED1234
        sizes = [int(x) for x in synth.entry_sizes_loguniform(2000, 300 << 20, seed=5)]
        arkfixture.write_archive(root, n_files=len(sizes), n_parts=3, seed=37, body_key=key, sizes=sizes)
        all_gpus = hex((1 << mb.device_count()) - 1)
        from pathlib import Path
        for extra in ({}, {"MOD_DEVICES": all_gpus}):
            env = dict(os.environ, MOD_TRACE="1", **extra)
            check_wild(CLI, Path(root), "ps4", b"\x5a\x00\x0f", b"\xff\x00\x0f", key=key, env=env)
    finally:
        shutil.rmtree(root, ignore_errors=True)
