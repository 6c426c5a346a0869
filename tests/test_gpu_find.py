"""GPU: the search kernel (find_batch_kernel behind mod_find_batch / mod_plan_find / mod_plan_find_window) and
the -find facade on the real library, against the oracle: entries deciphered on the CPU, every start compared."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import kernel_model as km
import oracle
import synth
import arkfixture
import modulate_b200 as mb
from gpuutil import DeviceBuffer, sync
from test_find_host import check, oracle_find, piece_cut_archive, SUMMARY

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "modulate_b200", "bin", "modulate")
EDGE_KEYS = [0, 0x7FFFFFFF, -0x80000000, -1, 1]


def plain_find(plain_entries, pat):
    """Oracle matches (desc, pos) and counts of the wanted deciphered entries."""
    out, counts = [], []
    P = np.frombuffer(pat, np.uint8)
    for i, e in enumerate(plain_entries):
        n = 0
        if e.size >= len(pat):
            w = np.lib.stride_tricks.sliding_window_view(e, len(pat))
            pos = np.nonzero((w == P).all(axis=1))[0]
            out += [(i, int(p)) for p in pos]
            n = len(pos)
        counts.append(n)
    return out, np.array(counts, np.uint32)


def build_source(plain_entries, keys, phase):
    """Byte-packed source whose entries decipher to `plain_entries` (Cycle is its own inverse)."""
    sizes = np.array([e.size for e in plain_entries], np.int64)
    src_off = synth.packed_offsets(sizes) + phase
    src = np.zeros(int(phase + sizes.sum() + 64), np.uint8)
    for e, o, k in zip(plain_entries, src_off, keys):
        src[o:o + e.size] = oracle.cycle(e, k)
    return mb.make_descs(src_off, src_off, sizes, keys), src


def run_find(plain_entries, keys, pat, phase=0, cap=1 << 16):
    descs, src = build_source(plain_entries, keys, phase)
    buf = DeviceBuffer.from_numpy(src)
    counts, matches, total = mb.find_batch(descs, buf.ptr, pat, src_bytes=src.size, max_matches=cap)
    buf.free()
    return counts, [(int(m["desc"]), int(m["pos"])) for m in matches], total


def planted_entries(L, pat, rng, phase):
    """Entries with the pattern straddling 16-byte chunk and 8 KiB tile boundaries (so inside the halo), at
    position 0 and len - L, and split across two adjacent entries."""
    sizes = [L, L - 1, 1, 17, 100, 8192 + 70, 3 * 8192 + 5, 40000, 333, 16, 0, 5000]
    ents = [rng.integers(0, 256, size=s, dtype=np.uint8) for s in sizes]
    for i, e in enumerate(ents):
        h0 = (phase + sum(sizes[:i])) & 15
        starts = {0, e.size - L}
        for b in list(range(16, e.size, 16 * 37)) + list(range(8192, e.size, 8192)):
            for j in (1, L // 2, L - 1):
                starts.add(b - h0 - j)
        for s in sorted(starts):
            if 0 <= s and s + L <= e.size:
                e[s:s + L] = np.frombuffer(pat, np.uint8)
    # split across entries 7 | 8 (no match may come of it)
    if L > 1:
        k = L // 2
        ents[7][-k:] = np.frombuffer(pat[:k], np.uint8)
        ents[8][:L - k] = np.frombuffer(pat[k:], np.uint8)
    return ents


@pytest.mark.parametrize("L", [1, 2, 3, 4, 5, 15, 16, 17, 63, 64])
def test_kernel_matches_oracle_planted(L):
    rng = np.random.default_rng(L)
    pat = bytes(int(x) for x in rng.integers(1, 256, size=L))
    for phase in range(16) if L in (5, 17) else (0, 7):
        ents = planted_entries(L, pat, rng, phase)
        for keys in ([k for k in EDGE_KEYS for _ in range(3)][:len(ents)], synth.entry_keys(len(ents)).tolist()):
            counts, matches, total = run_find(ents, keys, pat, phase)
            want, want_counts = plain_find(ents, pat)
            assert matches == want and total == len(want) and (counts == want_counts).all(), (L, phase)
            assert len(want) >= 5


def test_redo_branch_inside_the_tile_and_the_halo():
    """Keys chosen by the model's backward search put a bit-31 state (the exact redo) on a chunk inside a tile
    and on a halo chunk; a match planted over the triggering byte is found.  The model shows that the hot loop's
    speculative bytes differ there, so matching them without the redo would miss it."""
    rng = np.random.default_rng(5)
    h0, size = 5, 3 * 8192
    for tin, chunk, lo, hi, start_of in (
            (0, 300, 0, 16, lambda b: 16 * 300 + 0 - h0),               # interior chunk of tile 0
            (1, 0, 0, 16, lambda b: 8192 - h0 - 20),                    # halo of tile 0 = chunk 0 of tile 1
            (1, 1, 0, 12, lambda b: 8192 - h0 - 20)):                   # its second halo chunk
        st = km.find_tile_state(chunk, lo, hi, rng)[0]
        key = km.key_for_state(int(st), h0, tin)
        trig = np.nonzero(km.triggers(km.chunk_states(int(st), chunk)))[0]
        s = start_of(None)
        L = 64 if tin else 16
        plain = rng.integers(0, 256, size=size, dtype=np.uint8)
        pat = bytes(int(x) for x in rng.integers(1, 256, size=L))
        plain[s:s + L] = np.frombuffer(pat, np.uint8)
        tbyte = 8192 * tin + 16 * chunk + int(trig[0]) - h0
        assert s <= tbyte < s + L
        spec = km.speculative_bytes(km.chunk_states(int(st), chunk))
        canon = km.canonical_bytes(km.chunk_states(int(st), chunk))
        assert spec[trig[0]] != canon[trig[0]]  # the speculative keystream is wrong inside the match
        counts, matches, total = run_find([plain], [km.i32(key)], pat, phase=h0)
        want, _ = plain_find([plain], pat)
        assert (0, s) in want and matches == want and total == len(want)


def test_cap_truncation_keeps_exact_counts():
    rng = np.random.default_rng(3)
    ents = [np.zeros(int(n), np.uint8) for n in rng.integers(100, 20000, size=40)]
    for e in ents:
        e[rng.integers(0, e.size, size=e.size // 3)] = 1
    keys = synth.entry_keys(len(ents)).tolist()
    want, want_counts = plain_find(ents, b"\x00")
    counts, matches, total = run_find(ents, keys, b"\x00", cap=1000)
    assert total == len(want) and (counts == want_counts).all()
    assert len(matches) == 1000 and set(matches) <= set(want) and matches == sorted(matches)


def test_find_window_over_a_slot_ring_equals_the_whole_plan():
    rng = np.random.default_rng(11)
    sizes = [int(x) for x in rng.integers(0, 60000, size=300)]
    pat = b"\x4d\x6f"
    ents = [rng.integers(0, 256, size=s, dtype=np.uint8) for s in sizes]
    keys = synth.entry_keys(len(ents)).tolist()
    descs, src = build_source(ents, keys, 9)
    want, want_counts = plain_find(ents, pat)
    whole = DeviceBuffer.from_numpy(src)
    plan = mb.Plan(descs, src.size, src.size, 0)
    cap = 1 << 16
    out = DeviceBuffer(16 + 4 * len(ents) + 8 * cap)

    def results():
        raw = out.download()
        total = int(raw[:8].view(np.uint64)[0])
        counts = raw[16:16 + 4 * len(ents)].view(np.uint32)
        m = raw[16 + 4 * len(ents):].view(mb.MATCH_DTYPE)[:min(total, cap)]
        return total, counts.copy(), sorted((int(a), int(b)) for a, b in zip(m["desc"], m["pos"]))

    out.upload(np.zeros(out.nbytes, np.uint8))
    plan.find(whole.ptr, pat, out.ptr + 16, out.ptr + 16 + 4 * len(ents), cap, out.ptr)
    sync()
    total, counts, matches = results()
    assert total == len(want) and counts.tolist() == want_counts.tolist() and matches == want
    out.upload(np.zeros(out.nbytes, np.uint8))
    slots = [DeviceBuffer(4 << 20) for _ in range(3)]
    for gi, e0 in enumerate(range(0, len(ents), 23)):
        e1 = min(len(ents), e0 + 23)
        t0, t1 = plan.tile_range(e0, e1)
        lo = int(descs["src_off"][e0])
        hi = int(max(descs["src_off"][e1 - 1] + descs["len"][e1 - 1], lo))
        slot = slots[gi % 3]
        slot.upload(src[lo:hi], lo & 15)
        plan.find_window(t0, t1, slot.ptr + (lo & 15), lo, hi - lo, pat, out.ptr + 16, out.ptr + 16 + 4 * len(ents), cap, out.ptr)
        if gi == 0:
            with pytest.raises(mb.ModError):  # one byte short of the window: the halo / tail check refuses it
                plan.find_window(t0, t1, slot.ptr + (lo & 15), lo, hi - lo - 1, pat, out.ptr + 16,
                                 out.ptr + 16 + 4 * len(ents), cap, out.ptr)
        sync()
    total, counts, matches = results()
    assert total == len(want) and counts.tolist() == want_counts.tolist() and matches == want
    lib = mb._abi.load()
    for bad in (b"", b"x" * 65):
        with pytest.raises(ValueError):
            mb.find_batch(descs, whole.ptr, bad, src_bytes=src.size)
        cnt, tot = np.zeros(len(ents), np.uint32), ctypes.c_uint64()
        assert lib.mod_find_batch(descs.ctypes.data, len(descs), whole.ptr, src.size, bad + b"\0", len(bad), cnt.ctypes.data,
                                  None, 0, ctypes.byref(tot)) == -2  # MOD_ERR_ARG
    plan.close()


def test_one_gib_ten_thousand_entries_against_numpy():
    total_bytes = 1 << 30
    sizes = synth.entry_sizes_loguniform(10000, total_bytes, seed=7)
    src_off = synth.packed_offsets(sizes)
    keys = synth.entry_keys(len(sizes))
    descs = mb.make_descs(src_off, src_off, sizes, keys)
    n = int(src_off[-1] + sizes[-1])
    src = synth.payload(0, n)
    plain = np.empty_like(src)
    for o, s, k in zip(src_off, sizes, keys):
        plain[o:o + s] = oracle.cycle(src[o:o + s], int(k))
    # a 5-byte pattern planted in a few entries (in plain space, then re-enciphered)
    pat5 = b"\x01\x9a\x33\x7e\x02"
    for i in range(0, 10000, 997):
        o, s = int(src_off[i]), int(sizes[i])
        p = o + s // 2
        plain[p:p + 5] = np.frombuffer(pat5, np.uint8)
        src[o:o + s] = oracle.cycle(plain[o:o + s], int(keys[i]))
    buf = DeviceBuffer.from_numpy(src)
    ends = src_off + sizes
    for pat in (b"\xa5\x3c", pat5):
        L = len(pat)
        hit = plain[:n - L + 1] == pat[0]
        for j in range(1, L):
            hit &= plain[j:n - L + 1 + j] == pat[j]
        pos = np.nonzero(hit)[0]
        d = np.searchsorted(src_off, pos, side="right") - 1
        keep = pos + L <= ends[d]
        want = sorted(zip(d[keep].tolist(), (pos[keep] - src_off[d[keep]]).tolist()))
        counts, matches, total = mb.find_batch(descs, buf.ptr, pat, src_bytes=n, max_matches=1 << 20)
        assert total == len(want) and [(int(a), int(b)) for a, b in zip(matches["desc"], matches["pos"])] == want
        assert counts.sum() == total and (np.bincount(d[keep], minlength=len(sizes)) == counts).all()
    buf.free()


def shm_dir(tmp_path):
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else str(tmp_path)
    import tempfile
    return tempfile.mkdtemp(prefix="modfind", dir=base)


def test_facade_find_on_a_ciphered_1gib_archive(tmp_path):
    import shutil
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    root = shm_dir(tmp_path)
    try:
        key = 0x5EED1234
        sizes = [int(x) for x in synth.entry_sizes_loguniform(10000, 1 << 30, seed=5)]
        arkfixture.write_archive(root, n_files=len(sizes), n_parts=4, seed=37, body_key=key, sizes=sizes)
        pat = b"\x5a\xa5\x0f"
        want_lines, want_total, want_files = oracle_find(root, "ps4", pat, key)
        runs = [{}]
        if mb.device_count() >= 2:
            runs.append({"MOD_DEVICES": "0x3"})
        for extra in runs:
            env = dict(os.environ, MOD_TRACE="1", **extra)
            out = subprocess.run([CLI, "-bodykey", str(key), "-findhex", pat.hex()], cwd=root, capture_output=True, timeout=600,
                                 env=env)
            assert out.returncode == 0, out.stdout.decode("latin-1") + out.stderr.decode("latin-1")
            stdout = out.stdout.decode("latin-1")
            assert [ln for ln in stdout.splitlines() if "\t" in ln] == want_lines
            assert SUMMARY.search(stdout).groups() == (str(want_total), str(want_files))
            if extra:
                assert "on 2 GPU(s)" in out.stderr.decode()
    finally:
        shutil.rmtree(root, ignore_errors=True)


@pytest.mark.parametrize("L", [1, 2, 17, 64])
def test_facade_find_across_every_piece_cut(tmp_path, L):
    """The archive of test_find_host's piece-cut case through the CLI on the CUDA library: with 1 MiB groups the
    big entries travel as pieces that overlap by L - 1 bytes, and every match is still found exactly once."""
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    pat, key = piece_cut_archive(tmp_path, L)
    _, total, _, _ = check(CLI, tmp_path, "ps4", pat, key=key, env=dict(os.environ, MOD_IO_GROUP_MIB="1"))
    assert total >= 8
    check(CLI, tmp_path, "ps4", pat, key=key)
