"""GPU: the pattern-set search (find_set_kernel behind mod_find_set_batch / mod_plan_find_set / mod_plan_find_set_window)
and -findlist on the real library, against numpy over the oracle-deciphered entries: every start compared with every
pattern of the set, so overlapping matches and several patterns at one start all count."""
import ctypes
import os
import shutil
import subprocess
import zlib

import numpy as np
import pytest

import arkfixture
import kernel_model as km
import oracle
import synth
import modulate_b200 as mb
from gpuutil import (CLI, EDGE_KEYS, DeviceBuffer, Results, aligned_buffer, as_list, build_source, cases_by_cell,
                     decipher_entries, model_descs, shm_dir, sync)
from searchutil import MOD_ERR_ALIGN, MOD_ERR_ARG, check_set, expected_output, owned_trap_archive, search

pytestmark = pytest.mark.gpu


def run_set(plain_entries, keys, pats, phase=0, cap=1 << 18):
    descs, src = build_source(plain_entries, keys, phase)
    buf = DeviceBuffer.from_numpy(src)
    try:
        counts, pcounts, matches, total = mb.find_set_batch(descs, buf.ptr, pats, src_bytes=src.size, max_matches=cap)
    finally:
        buf.free()
    return counts, pcounts, as_list(matches), total


def check_against_oracle(ents, keys, pats, phase=0):
    counts, pcounts, matches, total = run_set(ents, keys, pats, phase)
    want, want_counts, want_p = search(ents, pats)
    assert total == len(want) and matches == want, (phase, len(pats))
    assert counts.tolist() == want_counts.tolist() and pcounts.tolist() == want_p.tolist()
    return want


def make_set(kind, rng):
    if kind.startswith("random"):
        k = int(kind[6:])
        pats = set()
        while len(pats) < k:
            pats.add(bytes(int(x) for x in rng.integers(0, 256, size=int(rng.integers(1, 65)))))
        return sorted(pats, key=lambda p: rng.random())
    if kind == "ones":
        return [bytes([b]) for b in rng.choice(256, size=17, replace=False)]
    if kind.startswith("prefix"):  # 64 patterns sharing their first n bytes
        n = int(kind[6:])
        head = bytes(int(x) for x in rng.integers(0, 256, size=n))
        pats = []
        while len(pats) < 64:
            p = head + bytes(int(x) for x in rng.integers(0, 256, size=int(rng.integers(1, 65 - n))))
            if p not in pats:
                pats.append(p)
        return pats
    if kind == "pairs":
        return [b"ab", b"abc", b"a", b"abcd", b"bc", b"abcde" * 12 + b"abcd"]
    raise ValueError(kind)


def planted(pats, rng, phase, sizes=(64, 63, 1, 17, 100, 8192 + 70, 3 * 8192 + 5, 40000, 333, 16, 0, 5000)):
    """Entries with every pattern planted at position 0, at the end, and across 16-byte chunk and 8 KiB tile
    boundaries (into the halo)."""
    ents = [rng.integers(0, 256, size=s, dtype=np.uint8) for s in sizes]
    for i, e in enumerate(ents):
        h0 = (phase + sum(sizes[:i])) & 15
        for pat in pats:
            L = len(pat)
            starts = {0, e.size - L} | {b - h0 - j for b in list(range(16, e.size, 16 * 97)) + list(range(8192, e.size, 8192))
                                        for j in (1, L // 2, L - 1)}
            for s in sorted(starts)[::max(1, len(pats) // 8)]:
                if 0 <= s and s + L <= e.size:
                    e[s:s + L] = np.frombuffer(pat, np.uint8)
    return ents


SET_KINDS = ["random1", "random2", "random17", "random256", "ones", "prefix2", "prefix4", "prefix8", "pairs"]


@pytest.mark.parametrize("kind", SET_KINDS)
def test_sets_against_the_oracle(kind):
    rng = np.random.default_rng(zlib.crc32(kind.encode()))
    pats = make_set(kind, rng)
    for phase in range(16) if kind in ("random17", "pairs") else (0, 7):
        ents = planted(pats, rng, phase)
        for keys in ([k for k in EDGE_KEYS for _ in range(3)][:len(ents)], synth.entry_keys(len(ents)).tolist()):
            want = check_against_oracle(ents, keys, pats, phase)
            assert len(want) >= 5


def test_entries_shorter_than_lmax_and_matches_at_the_ends():
    """Starts come from Lmin and each pattern's end is checked against the entry's: in entries shorter than Lmax the
    short patterns are found, also ending exactly at the entry end; a 64-byte match may end on the last halo byte."""
    rng = np.random.default_rng(8)
    long_pat = bytes(int(x) for x in rng.integers(0, 256, size=64))
    pats = [b"\x11\x22\x33", long_pat, b"\x44"]
    for phase in (0, 5, 15):
        sizes = [3, 10, 40, 63, 64, 8192 + 200, 2 * 8192 + 64]
        ents = [rng.integers(0, 256, size=s, dtype=np.uint8) for s in sizes]
        for i, e in enumerate(ents):
            e[-3:] = np.frombuffer(pats[0], np.uint8)   # ends exactly at the entry end
            if e.size > 3:
                e[-4] = 0x44
            if e.size >= 64 + 3:
                e[:64] = np.frombuffer(long_pat, np.uint8)
        for i in (5, 6):  # a 64-byte match from the last start of tile 0: its last byte is the last halo byte
            h0 = (phase + sum(sizes[:i])) & 15
            s = 8192 - h0 - 1
            ents[i][s:s + 64] = np.frombuffer(long_pat, np.uint8)
        want = check_against_oracle(ents, synth.entry_keys(len(ents)).tolist(), pats, phase)
        assert all((i, sizes[i] - 3, 0) in want for i in range(len(sizes)))
        assert all((i, 8192 - ((phase + sum(sizes[:i])) & 15) - 1, 1) in want for i in (5, 6))


def _companions(pat, rng, longest):
    """Other patterns for a model case's pattern: a prefix (same 2-byte key) and shorter or longer random ones."""
    L = len(pat)
    out = [pat]
    cands = [pat[:L - 1]] if L > 2 else []
    cands += [bytes(int(x) for x in rng.integers(0, 256, size=n)) for n in {1, max(1, L // 2), min(longest, 64)}]
    for c in cands:
        if 1 <= len(c) <= longest and c not in out:
            out.append(c)
    return out


@pytest.mark.parametrize("cell", sorted(km.reachable_find_cells()), ids=lambda c: "-".join(c))
def test_model_cases_through_the_set_kernel(cell):
    """Every case the kernel model builds for find_batch_kernel (redo cells, halo cells, guard decoys) run through the
    set kernel with the case's pattern inside a set of other lengths: the case's pattern gives the oracle's counts.
    Window cases take only patterns up to the case's length, so that the case's minimal window still holds."""
    case = cases_by_cell()[cell]
    rng = np.random.default_rng(zlib.crc32("-".join(cell).encode()))
    pats = _companions(case.pattern, rng, 64 if case.kind == "batch" else case.L)
    ents = decipher_entries(case.descs, case.image)
    want, want_counts, want_p = search(ents, pats)
    mem = case.memory()
    buf = aligned_buffer(mem)
    try:
        if case.kind == "batch":
            counts, pcounts, matches, total = mb.find_set_batch(model_descs(case.descs), buf.ptr + case.src_ptr, pats,
                                                                src_bytes=case.image_bytes, max_matches=1 << 16)
            assert total == len(want) and as_list(matches) == want, cell
            assert counts.tolist() == want_counts.tolist() and pcounts.tolist() == want_p.tolist()
        else:
            t0, t1, wp, wo, wb = case.win
            lo, hi = case.entry_starts()
            want0 = [(d, p, 0) for d, p, j in want if j == 0 and d == case.target and lo <= p < hi]
            plan = mb.Plan(model_descs(case.descs), case.image_bytes, case.image_bytes, case.dst_align)
            pset = mb.PatternSet(pats)
            res = Results(len(case.descs), 1 << 12)
            pc = DeviceBuffer(8 * len(pats))
            pc.upload(np.zeros(8 * len(pats), np.uint8))
            m = DeviceBuffer(12 * res.cap)
            plan.find_set_window(t0, t1, buf.ptr + wp, wo, wb, pset, res.counts, pc.ptr, m.ptr, res.cap, res.total)
            sync()
            total = int(res.buf.download()[:8].view(np.uint64)[0])
            got = as_list(m.download().view(mb.SET_MATCH_DTYPE)[:min(total, res.cap)])
            assert int(pc.download().view(np.uint64)[0]) == len(want0), cell
            assert sorted(x for x in got if x[2] == 0) == want0, cell
            plan.close()
            pset.close()
            pc.free()
            m.free()
    finally:
        buf.free()


def test_one_pattern_set_equals_find_batch():
    rng = np.random.default_rng(21)
    for L in (1, 2, 5, 17, 64):
        pat = bytes(int(x) for x in rng.integers(0, 256, size=L))
        ents = planted([pat], rng, 3)
        keys = synth.entry_keys(len(ents)).tolist()
        descs, src = build_source(ents, keys, 3)
        buf = DeviceBuffer.from_numpy(src)
        c1, m1, t1 = mb.find_batch(descs, buf.ptr, pat, src_bytes=src.size)
        c2, p2, m2, t2 = mb.find_set_batch(descs, buf.ptr, [pat], src_bytes=src.size)
        buf.free()
        assert t1 == t2 == int(p2[0]) and c1.tolist() == c2.tolist()
        assert [(int(a), int(b)) for a, b in zip(m1["desc"], m1["pos"])] == [(d, p) for d, p, _ in as_list(m2)]
        assert all(j == 0 for _, _, j in as_list(m2)) and t1 >= 5


def test_64_patterns_on_one_gib_equal_64_single_searches():
    total_bytes = 1 << 30
    sizes = synth.entry_sizes_loguniform(10000, total_bytes, seed=7)
    src_off = synth.packed_offsets(sizes)
    keys = synth.entry_keys(len(sizes))
    descs = mb.make_descs(src_off, src_off, sizes, keys)
    n = int(src_off[-1] + sizes[-1])
    buf = DeviceBuffer(n)
    buf.fill_payload()
    rng = np.random.default_rng(64)
    pats = set()
    while len(pats) < 64:
        pats.add(bytes(int(x) for x in rng.integers(0, 256, size=int(rng.choice([2, 2, 3, 4, 9, 33, 64])))))
    pats = sorted(pats)
    counts, pcounts, matches, total = mb.find_set_batch(descs, buf.ptr, pats, src_bytes=n, max_matches=1 << 23)
    want_counts = np.zeros(len(sizes), np.uint64)
    want = []
    for j, pat in enumerate(pats):
        c, m, t = mb.find_batch(descs, buf.ptr, pat, src_bytes=n, max_matches=1 << 20)
        assert int(pcounts[j]) == t
        want_counts += c
        want += [(int(a), int(b), j) for a, b in zip(m["desc"], m["pos"])]
    buf.free()
    want.sort()
    assert total == len(want) == int(pcounts.sum()) and as_list(matches) == want and total > 10 * 64
    assert (counts.astype(np.uint64) == want_counts).all()


def _plan_and_buffers(ents, keys, pats, phase=0, cap=1):
    descs, src = build_source(ents, keys, phase)
    buf = DeviceBuffer.from_numpy(src)
    plan = mb.Plan(descs, src.size, src.size, (buf.ptr) & 15)
    res = Results(len(ents), cap)
    pc = DeviceBuffer(8 * len(pats))
    pc.upload(np.zeros(pc.nbytes, np.uint8))
    m = DeviceBuffer(12 * max(cap, 1))
    return descs, src, buf, plan, res, pc, m


@pytest.mark.parametrize("which", ["0", "1", "n", "n+1"])
def test_cap_and_accumulation(which):
    rng = np.random.default_rng(4)
    pats = [b"\x00", b"\x00\x01", b"\x01\x00\x01"]
    ents = [np.zeros(int(s), np.uint8) for s in rng.integers(100, 9000, size=20)]
    for e in ents:
        e[rng.integers(0, e.size, size=e.size // 3)] = 1
    keys = synth.entry_keys(len(ents)).tolist()
    want, want_counts, want_p = search(ents, pats)
    n = len(want)
    cap = {"0": 0, "1": 1, "n": n, "n+1": n + 1}[which]
    descs, src, buf, plan, res, pc, m = _plan_and_buffers(ents, keys, pats, cap=cap)
    pset = mb.PatternSet(pats)
    for rep in (1, 2):  # results accumulate over calls
        plan.find_set(buf.ptr, pset, res.counts, pc.ptr, m.ptr, cap, res.total)
        sync()
        raw = res.buf.download()
        total = int(raw[:8].view(np.uint64)[0])
        assert total == rep * n
        assert raw[16:16 + 4 * len(ents)].view(np.uint32).tolist() == (rep * want_counts).tolist()
        assert pc.download().view(np.uint64).tolist() == (rep * want_p).tolist()
        got = as_list(m.download().view(mb.SET_MATCH_DTYPE)[:min(total, cap)])
        assert len(got) == min(cap, total) and set(got) <= set(want)
        if rep == 1 and cap >= n:
            assert sorted(got) == want
    for x in (plan, pset):
        x.close()
    for x in (buf, pc, m):
        x.free()


def test_window_bounds_use_lmax():
    """Inside one entry: the minimal window for the set's Lmax is accepted (and equals the whole search of the tiles),
    one byte short at either end is MOD_ERR_ARG."""
    rng = np.random.default_rng(9)
    pats = [b"\x5a", b"\x5a\xa5\x0f", bytes(int(x) for x in rng.integers(0, 256, size=40))]
    lmax = 40
    ent = rng.integers(0, 256, size=6 * 8192, dtype=np.uint8)
    ent[3 * 8192 - 7:3 * 8192 - 7 + 40] = np.frombuffer(pats[2], np.uint8)
    descs, src, buf, plan, res, pc, m = _plan_and_buffers([ent], [0x1234567], pats, phase=0, cap=1 << 12)
    pset = mb.PatternSet(pats)
    t0, t1 = 1, 3
    h0 = int(descs["src_off"][0] + (buf.ptr & 15)) & 15
    lo = 8192 * t0 - h0
    hi = 8192 * t1 - h0 + lmax - 1
    win = DeviceBuffer(hi - lo + 32)
    at = (lo + buf.ptr) & 15  # keep the window on the plan's grid
    win.upload(src[lo:hi], at)
    plan.find_set_window(t0, t1, win.ptr + at, lo, hi - lo, pset, res.counts, pc.ptr, m.ptr, res.cap, res.total)
    sync()
    total = int(res.buf.download()[:8].view(np.uint64)[0])
    got = sorted(as_list(m.download().view(mb.SET_MATCH_DTYPE)[:total]))
    want, _, _ = search([oracle.cycle(src[:ent.size], 0x1234567)], pats)
    assert got == [x for x in want if lo <= x[1] < 8192 * t1 - h0] and (0, 3 * 8192 - 7, 2) in got
    for bad_lo, bad_hi in ((lo + 1, hi), (lo, hi - 1)):
        lib = mb._abi.load()
        rc = lib.mod_plan_find_set_window(plan._handle, t0, t1, win.ptr + at + (bad_lo - lo), bad_lo, bad_hi - bad_lo,
                                          pset._handle, None, res.counts, pc.ptr, m.ptr, res.cap, res.total, None)
        assert rc == MOD_ERR_ARG
    for x in (plan, pset):
        x.close()
    for x in (buf, pc, m, win):
        x.free()


def test_refusals():
    rng = np.random.default_rng(2)
    ents = [rng.integers(0, 256, size=5000, dtype=np.uint8) for _ in range(3)]
    pats = [b"ab", b"c"]
    descs, src, buf, plan, res, pc, m = _plan_and_buffers(ents, [1, 2, 3], pats, cap=4)
    pset = mb.PatternSet(pats)
    lib = mb._abi.load()
    # off the source grid: the plan's chunk grid does not lie on a source shifted by one byte
    assert lib.mod_plan_find_set(plan._handle, buf.ptr + 1, pset._handle, None, res.counts, pc.ptr, m.ptr, 4, res.total,
                                 None) == MOD_ERR_ALIGN
    off = mb.Plan(mb.make_descs(descs["src_off"], descs["src_off"] + 3, descs["len"], descs["key"]), src.size, src.size + 3, 0)
    assert lib.mod_plan_find_set(off._handle, buf.ptr, pset._handle, None, res.counts, pc.ptr, m.ptr, 4, res.total,
                                 None) == MOD_ERR_ALIGN
    # invalid sets are refused on the host
    h = ctypes.c_void_p()
    for data, lens in ((b"abab", [2, 2]), (b"", []), (b"x" * 65, [65]), (b"a", [0])):
        arr = np.frombuffer(data or b"\0", np.uint8)
        ln = np.array(lens or [1], np.uint32)
        assert lib.mod_pattern_set_create(arr.ctypes.data, ln.ctypes.data, len(lens), ctypes.byref(h)) == MOD_ERR_ARG
    many = np.frombuffer(b"".join(b"%03d" % i for i in range(257)), np.uint8)
    assert lib.mod_pattern_set_create(many.ctypes.data, np.full(257, 3, np.uint32).ctypes.data, 257, ctypes.byref(h)) == MOD_ERR_ARG
    assert lib.mod_pattern_set_create(many.ctypes.data, np.full(256, 3, np.uint32).ctypes.data, 256, ctypes.byref(h)) == 0
    lib.mod_pattern_set_destroy(h)
    with pytest.raises(ValueError):
        mb.PatternSet([b"a", b"a"])
    # a set of another device
    if mb.device_count() >= 2:
        mb.init(1)
        other = mb.PatternSet(pats)
        mb.init(0)
        assert lib.mod_plan_find_set(plan._handle, buf.ptr, other._handle, None, res.counts, pc.ptr, m.ptr, 4, res.total,
                                     None) == MOD_ERR_ARG
        other.close()
    for x in (plan, pset, off):
        x.close()
    for x in (buf, pc, m):
        x.free()


def test_facade_find_set_across_every_piece_cut(tmp_path):
    """test_find_set_host's owned-start archive through the CLI on the CUDA library: with 1 MiB groups the pieces
    overlap by Lmax - 1 = 63 bytes and the short patterns planted there are counted once."""
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    rng = np.random.default_rng(3)
    pats = [b"\xe7", bytes(int(x) for x in rng.integers(0, 256, 17)), bytes(int(x) for x in rng.integers(0, 256, 64))]
    key = owned_trap_archive(tmp_path, pats)
    total = check_set(CLI, tmp_path, "ps4", pats, key=key, env=dict(os.environ, MOD_IO_GROUP_MIB="1"))[2]
    assert check_set(CLI, tmp_path, "ps4", pats, key=key)[2] == total


def test_facade_find_set_on_a_ciphered_1gib_archive_on_every_gpu(tmp_path):
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    root = shm_dir(tmp_path)
    try:
        key = 0x5EED1234
        sizes = [int(x) for x in synth.entry_sizes_loguniform(10000, 1 << 30, seed=5)]
        arkfixture.write_archive(root, n_files=len(sizes), n_parts=4, seed=37, body_key=key, sizes=sizes)
        pats = [b"\x5a\xa5\x0f", b"\x5a\xa5", b"\x01\x02\x03\x04\x05", b"\x33\x44\x55\x66"]
        shown = [p.hex() for p in pats]
        want_lines, want_counts, want_total, want_files = expected_output(root, "ps4", pats, key=key, shown=shown)
        with open(os.path.join(root, "l.txt"), "w") as f:
            f.write("\n".join(shown) + "\n")
        all_gpus = hex((1 << mb.device_count()) - 1)
        for extra in ({}, {"MOD_DEVICES": all_gpus}):
            env = dict(os.environ, MOD_TRACE="1", **extra)
            out = subprocess.run([CLI, "-bodykey", str(key), "-findhexlist", "l.txt"], cwd=root, capture_output=True,
                                 timeout=900, env=env)
            assert out.returncode == 0, out.stdout.decode("latin-1")[-3000:] + out.stderr.decode("latin-1")[-3000:]
            stdout = out.stdout.decode("latin-1")
            rows = [ln for ln in stdout.splitlines() if "\t" in ln]
            assert [ln for ln in rows if ln.count("\t") == 1] == want_counts
            assert [ln for ln in rows if ln.count("\t") == 2] == want_lines[:10000]
            assert f"{want_total} matches in {want_files} files" in stdout
            if extra:
                assert f"on {mb.device_count()} GPU(s)" in out.stderr.decode()
    finally:
        shutil.rmtree(root, ignore_errors=True)
