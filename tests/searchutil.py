"""CPU helpers of the search tests: the CLI linked against the oracle-backed mock of the C ABI, the numpy reference
every search is checked against, the CLI output it predicts, and the archives the search tests build."""
from __future__ import annotations

import glob
import os
import re
import subprocess

import numpy as np

import arkfixture
import kernel_model_masked as kmm
import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "modulate_b200", "csrc")
CPP = os.path.join(ROOT, "tests", "cpp")
BUILD = os.path.join(ROOT, "tests", "_build")

MOD_ERR_ARG, MOD_ERR_ALIGN = -2, -3
FOLD = np.array([kmm.fold(b) for b in range(256)], np.uint8)
SUMMARY = re.compile(r"^(\d+) matches in (\d+) files$", re.M)
PIECE_GROUP = 1 << 20  # MOD_IO_GROUP_MIB=1


# ---- the mock CLI ------------------------------------------------------------------------------------------------

def link(name: str, main: str, generation: int = 0) -> str:
    """tests/_build/<name>: the facade (csrc/*.cpp) and `main` linked against the oracle-backed mock ABI with the
    search entry points of library generation `generation` (tests/cpp/mock_find_abi.cpp); g++ only, no CUDA.  Linked
    again when any source is newer than the binary."""
    oracle.build()
    os.makedirs(BUILD, exist_ok=True)
    exe = os.path.join(BUILD, name)
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cpp"))) + [main, os.path.join(CPP, "mock_abi.cpp"),
                                                             os.path.join(CPP, "mock_find_abi.cpp")]
    deps = srcs + glob.glob(os.path.join(CSRC, "*.h")) + glob.glob(os.path.join(CPP, "*")) + \
        [os.path.join(ROOT, "include", "modulate_b200.h")]
    if not os.path.exists(exe) or any(os.path.getmtime(d) > os.path.getmtime(exe) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", f"-DMOCK_SEARCH_ABI={generation}",
                               "-I", CSRC, "-I", os.path.join(ROOT, "include"), "-o", exe, *srcs,
                               "-L", os.path.join(ROOT, "oracle"), "-loracle", f"-Wl,-rpath,{os.path.join(ROOT, 'oracle')}"])
    return exe


def mock_cli(generation: int) -> str:
    """The modulate CLI on the mock ABI of library generation 0 (no search), 1 (single pattern), 2 (pattern sets) or
    3 (masked patterns and case-folded sets)."""
    return link(f"modulate_mock_gen{generation}", os.path.join(CSRC, "cli", "modulate_main.cpp"), generation)


# ---- the reference -----------------------------------------------------------------------------------------------

def search(entries, patterns, masks=None, fold=False, owned=None):
    """Every start p of entry i at which pattern j matches: ((t ^ v) & m) == 0 for each pattern byte v, its mask byte m
    (0xFF without `masks`) and the entry byte t under it, t and v ASCII-folded when `fold`; p < owned[i] when `owned`
    is given.  -> (sorted (i, p, j) matches, counts per entry as uint32, counts per pattern as uint64)."""
    out = []
    for i, e in enumerate(entries):
        e = FOLD[e] if fold else np.asarray(e, np.uint8)
        for j, pat in enumerate(patterns):
            L = len(pat)
            if e.size < L:
                continue
            v = np.frombuffer(pat, np.uint8)
            m = np.frombuffer(masks[j], np.uint8) if masks is not None else np.full(L, 0xFF, np.uint8)
            x = np.lib.stride_tricks.sliding_window_view(e, L) ^ (FOLD[v] if fold else v)
            x &= m
            pos = np.nonzero(~x.any(axis=1))[0]
            if owned is not None:
                pos = pos[pos < owned[i]]
            out += [(i, int(p), j) for p in pos]
    out.sort()
    counts = np.bincount([i for i, _, _ in out], minlength=len(entries)).astype(np.uint32)
    pattern_counts = np.bincount([j for _, _, j in out], minlength=len(patterns)).astype(np.uint64)
    return out, counts, pattern_counts


def search_one(entries, pattern, mask=None, fold=False):
    """search() for one pattern -> (sorted (i, p) matches, counts per entry)."""
    out, counts, _ = search(entries, [pattern], None if mask is None else [mask], fold)
    return [(i, p) for i, p, _ in out], counts


def image_of(root, hdr):
    return np.frombuffer(b"".join(open(os.path.join(root, p), "rb").read() for p, _ in hdr.parts), np.uint8)


def expected_output(root, plat, patterns, masks=None, fold=False, key=0, shown=None):
    """What a search of the archive in `root` prints -> (match lines, per-pattern lines, total, files).  Lines are in
    table order (as Load parses it), then offset, then list order.  A list search prints each pattern as `shown[j]`,
    on its match lines and its count lines; a single-pattern search (`shown` None) prints name and offset only."""
    hdr, _ = arkfixture.read_header(os.path.join(root, f"main_{plat}.hdr"))
    image = image_of(root, hdr)
    plain = [oracle.cycle(image[e.offset:e.offset + e.size], key) if key else image[e.offset:e.offset + e.size]
             for e in hdr.entries]
    matches, counts, pattern_counts = search(plain, patterns, masks, fold)
    if shown is None:
        lines = [f"{hdr.entries[i].name}\t{p}" for i, p, _ in matches]
    else:
        lines = [f"{hdr.entries[i].name}\t{p}\t{shown[j]}" for i, p, j in matches]
    return lines, [f"{c}\t{s}" for c, s in zip(pattern_counts, shown or [])], len(matches), int((counts > 0).sum())


# ---- running the CLI ---------------------------------------------------------------------------------------------

def cli_out(cli, root, *args, env=None, expect=0):
    """Run a search command -> (lines holding a tab, total, files, stdout); total and files are None without the
    summary line."""
    out = subprocess.run([cli, *args], cwd=root, capture_output=True, timeout=600, env=env)
    stdout = out.stdout.decode("latin-1")
    assert out.returncode == (0 if expect == 0 else 255), stdout + out.stderr.decode("latin-1")
    m = SUMMARY.search(stdout)
    lines = [ln for ln in stdout.splitlines() if "\t" in ln]
    return lines, int(m.group(1)) if m else None, int(m.group(2)) if m else None, stdout


def _pre(plat, key):
    return (["-ps3"] if plat == "ps3" else []) + (["-bodykey", str(key)] if key else [])


def cli_find(cli, root, pat: bytes, *pre, env=None, hex_form=False):
    got = cli_out(cli, root, *pre, *(["-findhex", pat.hex()] if hex_form else ["-find", pat]), env=env)
    assert got[1] is not None, got[3]
    return got


def cli_find_set(cli, root, pats, *pre, env=None, hex_form=True, expect=0):
    """Write the list, run the CLI -> (match lines, count lines, total, files, stdout)."""
    path = os.path.join(root, "patterns.txt")
    with open(path, "wb") as f:
        f.write(b"".join((p.hex() if hex_form else p.decode("latin-1")).encode("latin-1") + b"\n" for p in pats))
    rows, total, files, stdout = cli_out(cli, root, *pre, "-findhexlist" if hex_form else "-findlist", path, env=env,
                                         expect=expect)
    return [ln for ln in rows if ln.count("\t") == 2], [ln for ln in rows if ln.count("\t") == 1], total, files, stdout


def wild_hex(value: bytes, mask: bytes) -> str:
    """The -findwild text of (value, mask) with nibble masks only."""
    out = []
    for v, m in zip(value, mask):
        out.append("".join("%x" % ((v >> s) & 15) if (m >> s) & 15 == 15 else "?" for s in (4, 0)))
    return " ".join(out)


# ---- the CLI against the reference -------------------------------------------------------------------------------

def check(cli, root, plat, pat, key=0, env=None, hex_form=True):
    got = cli_find(cli, root, pat, *_pre(plat, key), env=env, hex_form=hex_form)
    want_lines, _, want_total, want_files = expected_output(root, plat, [pat], key=key)
    assert got[1:3] == (want_total, want_files), pat
    if want_total <= 10000:
        assert got[0] == want_lines, pat
    else:
        # more matches than lines: which ones a group that overflows its list keeps is unspecified, but the
        # lines are matches, in table order, and the rest is counted
        rank = {ln: i for i, ln in enumerate(want_lines)}
        idx = [rank[ln] for ln in got[0]]
        assert len(idx) == 10000 and idx == sorted(idx) and len(set(idx)) == len(idx)
        assert f"... {want_total - 10000} more" in got[3]
    return got


def check_set(cli, root, plat, pats, key=0, env=None, hex_form=True):
    shown = [p.hex() for p in pats] if hex_form else [p.decode("latin-1") for p in pats]
    got = cli_find_set(cli, root, pats, *_pre(plat, key), env=env, hex_form=hex_form)
    want = expected_output(root, plat, pats, key=key, shown=shown)
    assert got[1:4] == want[1:], (got[1:4], want[1:])
    if want[2] <= 10000:
        assert got[0] == want[0]
    return got


def check_wild(cli, root, plat, value, mask, key=0, env=None):
    got = cli_out(cli, root, *_pre(plat, key), "-findwild", wild_hex(value, mask), env=env)
    want_lines, _, want_total, want_files = expected_output(root, plat, [value], [mask], key=key)
    assert got[1:3] == (want_total, want_files), (value.hex(), mask.hex())
    if want_total <= 10000:
        assert got[0] == want_lines
    return got


def check_nocase(cli, root, plat, text: bytes, key=0):
    got = cli_out(cli, root, *_pre(plat, key), "-findi", text)
    want_lines, _, want_total, want_files = expected_output(root, plat, [text], fold=True, key=key)
    assert got[1:3] == (want_total, want_files), text
    if want_total <= 10000:
        assert got[0] == want_lines
    assert f"for {len(text)} bytes, ignoring case" in got[3]
    return got


def check_nocase_set(cli, root, plat, pats, key=0):
    (root / "ilist.txt").write_bytes(b"".join(p + b"\n" for p in pats))
    lines, total, files, stdout = cli_out(cli, root, *_pre(plat, key), "-findilist", str(root / "ilist.txt"))
    want_lines, want_counts, want_total, want_files = expected_output(root, plat, pats, fold=True, key=key,
                                                                      shown=[p.decode("latin-1") for p in pats])
    assert (total, files) == (want_total, want_files)
    assert [ln for ln in lines if ln.count("\t") == 1] == want_counts
    if want_total <= 10000:
        assert [ln for ln in lines if ln.count("\t") == 2] == want_lines
    assert f"for {len(pats)} patterns, ignoring case" in stdout
    return total


# ---- archives ----------------------------------------------------------------------------------------------------

def planted_archive(root, key=0, **kw):
    """Entries that hold the pattern at their first byte, at their last bytes, split across the boundary of
    two adjacent entries (which must not match), in overlapping runs, and entries shorter than it."""
    pat = b"SYMBOLab"
    contents = {
        1: pat + bytes(100),                       # at entry start
        2: bytes(77) + pat,                        # at entry end
        3: bytes(40) + pat[:3],                    # boundary: 3 bytes here ...
        4: pat[3:] + bytes(40),                    # ... 5 in the next entry: no match
        5: b"aaaaaaa" + bytes(5) + pat * 3 + pat[:7],  # overlapping runs of "aa", adjacent copies
        6: pat[:5],                                # shorter than the pattern
        8: pat,                                    # exactly the pattern
    }
    sizes = [1000, 108, 85, 43, 45, 12 + 24 + 7, 5, 0, 8, 0, 333] + [5000] * 10
    contents[0] = bytes(1000)
    hdr, payloads, _ = arkfixture.write_archive(str(root), n_files=len(sizes), n_parts=2, seed=47, body_key=key, sizes=sizes,
                                                contents=contents, **kw)
    return hdr, pat


def piece_cut_archive(root, L):
    """An archive whose big entries a 1 MiB group cuts into pieces that overlap by L - 1 bytes, with an L-byte
    pattern planted across every cut, at each piece's first and last possible start and at each entry's end.
    -> (pattern, body key)."""
    G = PIECE_GROUP
    key = 0x2468ACE
    sizes = [3_500_000, 10, 0, 2_200_001, 70_000, 1_572_864, 5] + [30_000] * 6
    rng = np.random.default_rng(L)
    pat = bytes(int(x) for x in rng.integers(1, 256, size=L))
    contents = {}
    for i, s in enumerate(sizes):
        blob = bytearray(rng.integers(0, 256, size=s, dtype=np.uint8).tobytes())
        for cut in range(G, s, G):
            for start in {cut - L // 2 - 1, cut - L, cut - 1, cut}:
                if 0 <= start and start + L <= s:
                    blob[start:start + L] = pat
        if s >= L:
            blob[s - L:] = pat
        contents[i] = bytes(blob)
    arkfixture.write_archive(str(root), n_files=len(sizes), n_parts=2, seed=29, body_key=key, sizes=sizes, contents=contents)
    return pat, key


def owned_trap_archive(root, pats):
    """Big entries that 1 MiB groups cut into pieces overlapping by Lmax - 1 = 63 bytes, with every pattern planted
    in the 63 bytes after every cut: a piece that reported starts in its overlap would count them twice."""
    G = PIECE_GROUP
    key = 0x0BADC0DE
    sizes = [3_500_000, 10, 2_200_001, 1_572_864, 70_000]
    rng = np.random.default_rng(17)
    contents = {}
    for i, s in enumerate(sizes):
        blob = bytearray(rng.integers(0, 256, size=s, dtype=np.uint8).tobytes())
        for cut in range(G, s, G):
            for start, pat in ((cut, pats[0]), (cut + 1, pats[1]), (cut + 30, pats[0]), (cut + 62, pats[0]),
                               (cut + 20, pats[1]), (cut + 40, pats[1]), (cut - 64, pats[2]), (cut + 70, pats[2])):
                if start + len(pat) <= s:
                    blob[start:start + len(pat)] = pat
        contents[i] = bytes(blob)
    arkfixture.write_archive(str(root), n_files=len(sizes), n_parts=2, seed=23, body_key=key, sizes=sizes, contents=contents)
    return key
