"""CPU: the archive search (-find / -findhex, CArk::FindInFiles, the slot-ring GPU step) driven end to end
through the oracle-backed mock of the C ABI (tests/cpp/mock_abi.cpp).  Expected results come from the
oracle: every entry deciphered, then every start position compared, so overlapping matches count."""
import os
import re
import subprocess

import numpy as np
import pytest

import arkfixture
import oracle
from oracle import ark_oracle as ao
from test_facade_host import BUILD, CSRC, ROOT, run

MOCK_FIND = os.path.join(BUILD, "modulate_mock_find")


@pytest.fixture(scope="session")
def cli():
    """modulate CLI linked against the oracle-backed mock ABI plus its search entry points (g++ only, no CUDA)."""
    import glob
    oracle.build()
    os.makedirs(BUILD, exist_ok=True)
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cpp"))) + [os.path.join(CSRC, "cli", "modulate_main.cpp"),
                                                              os.path.join(ROOT, "tests", "cpp", "mock_abi.cpp"),
                                                              os.path.join(ROOT, "tests", "cpp", "mock_find_abi.cpp")]
    deps = srcs + glob.glob(os.path.join(CSRC, "*.h")) + [os.path.join(ROOT, "include", "modulate_b200.h")]
    if not os.path.exists(MOCK_FIND) or any(os.path.getmtime(d) > os.path.getmtime(MOCK_FIND) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"), "-o",
                               MOCK_FIND, *srcs, "-L", os.path.join(ROOT, "oracle"), "-loracle",
                               f"-Wl,-rpath,{os.path.join(ROOT, 'oracle')}"])
    return MOCK_FIND
from test_ref_fixtures import MANIFEST, CASES, fixture_file_bytes, ref_header

SUMMARY = re.compile(r"^(\d+) matches in (\d+) files$", re.M)


def image_of(root, hdr):
    return np.frombuffer(b"".join(open(os.path.join(root, p), "rb").read() for p, _ in hdr.parts), np.uint8)


def positions(data: np.ndarray, pat: bytes):
    L = len(pat)
    if data.size < L:
        return []
    win = np.lib.stride_tricks.sliding_window_view(data, L)
    return [int(i) for i in np.nonzero((win == np.frombuffer(pat, np.uint8)).all(axis=1))[0]]


def oracle_find(root, plat, pat: bytes, key: int = 0, max_lines: int = 10000):
    """(lines, total, files) the CLI must print: table order (as Load parses it), then offset."""
    hdr, _ = arkfixture.read_header(os.path.join(root, f"main_{plat}.hdr"))
    image = image_of(root, hdr)
    lines, total, files = [], 0, 0
    for e in hdr.entries:
        data = oracle.cycle(image[e.offset:e.offset + e.size], key) if key else image[e.offset:e.offset + e.size]
        pos = positions(data, pat)
        total += len(pos)
        files += bool(pos)
        lines += [f"{e.name}\t{p}" for p in pos]
    return lines[:max_lines], total, files


def cli_find(cli, root, pat: bytes, *pre, env=None, hex_form=False):
    args = [*pre, "-findhex", pat.hex()] if hex_form else [*pre, "-find", pat]
    out = subprocess.run([cli, *args], cwd=root, capture_output=True, timeout=600, env=env)
    stdout = out.stdout.decode("latin-1")
    assert out.returncode == 0, stdout + out.stderr.decode("latin-1")
    lines = [ln for ln in stdout.splitlines() if "\t" in ln]
    m = SUMMARY.search(stdout)
    assert m, stdout
    return lines, int(m.group(1)), int(m.group(2)), stdout


def check(cli, root, plat, pat, key=0, env=None, hex_form=True):
    pre = (["-ps3"] if plat == "ps3" else []) + (["-bodykey", str(key)] if key else [])
    got = cli_find(cli, root, pat, *pre, env=env, hex_form=hex_form)
    want = oracle_find(root, plat, pat, key, max_lines=None)
    assert got[1:3] == want[1:], pat
    if want[1] <= 10000:
        assert got[0] == want[0], pat
    else:
        # more matches than lines: which ones a group that overflows its list keeps is unspecified, but the
        # lines are matches, in table order, and the rest is counted
        rank = {ln: i for i, ln in enumerate(want[0])}
        idx = [rank[ln] for ln in got[0]]
        assert len(idx) == 10000 and idx == sorted(idx) and len(set(idx)) == len(idx)
        assert f"... {want[1] - 10000} more" in got[3]
    return got


@pytest.mark.parametrize("case", CASES)
def test_find_in_reference_written_archives(cli, tmp_path, case):
    """The archives exactly as the reference wrote them (PS3 and PS4): -find and -findhex equal the oracle."""
    info = MANIFEST[case]
    plat = info["platform"]
    (tmp_path / f"main_{plat}.hdr").write_bytes(ref_header(case))
    by_name = {f["name"]: f for f in info["input"]}
    image = bytearray(sum(p["size"] for p in info["loaded_parts"]))
    for f in info["loaded_files"]:
        image[f["offset"]:f["offset"] + f["size"]] = fixture_file_bytes(by_name[f["name"]])
    pos = 0
    for part in info["loaded_parts"]:
        (tmp_path / part["path"]).write_bytes(bytes(image[pos:pos + part["size"]]))
        pos += part["size"]
    some = next(bytes(image[f["offset"] + 3:f["offset"] + 9]) for f in info["loaded_files"] if f["size"] > 16)
    for pat in (some, some[:2], b"\x00", b"\x00\x00\x00\x00\x00", b"not in there at all"):
        _, total, _, _ = check(cli, tmp_path, plat, pat)
        if pat == some:
            assert total >= 1
    text = next(bytes(image[i:i + 4]) for i in range(len(image) - 4) if 0 not in image[i:i + 4])
    check(cli, tmp_path, plat, text, hex_form=False)  # argv bytes as they are


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


def test_planted_patterns_boundaries_overlaps_and_short_entries(cli, tmp_path):
    hdr, pat = planted_archive(tmp_path)
    lines, total, files, _ = check(cli, tmp_path, "ps4", pat)
    assert total >= 5
    check(cli, tmp_path, "ps4", b"aa")           # 6 overlapping starts in "aaaaaaa"
    check(cli, tmp_path, "ps4", pat * 2)         # longer than most entries
    check(cli, tmp_path, "ps4", b"\x00")         # L = 1: very many matches, zero-size entries included
    _, total, _, _ = check(cli, tmp_path, "ps4", pat[:3] + pat[3:5])
    # the split copy across entries 3 / 4 is not a match
    assert not any(ln.startswith(hdr.entries[3].name + "\t") for ln in cli_find(cli, tmp_path, pat)[0])


@pytest.mark.parametrize("key", [0x7FFFFFFF, -0x80000000, -1, 1, 0x12345678])
def test_body_key_edge_keys(cli, tmp_path, key):
    _, pat = planted_archive(tmp_path, key=key)
    _, total, _, _ = check(cli, tmp_path, "ps4", pat, key=key)
    assert total >= 5


def test_ps3_archive(cli, tmp_path):
    _, pat = planted_archive(tmp_path, ps4=False)
    check(cli, tmp_path, "ps3", pat)


PIECE_GROUP = 1 << 20  # MOD_IO_GROUP_MIB=1


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


@pytest.mark.parametrize("L", [1, 2, 17, 64])
def test_matches_across_every_piece_cut(cli, tmp_path, L):
    """MOD_IO_GROUP_MIB=1 cuts the big entries into 1 MiB pieces that overlap by L - 1 bytes: a match planted
    across every cut is found exactly once, and so is one at each piece's first and last possible start."""
    pat, key = piece_cut_archive(tmp_path, L)
    env = dict(os.environ, MOD_IO_GROUP_MIB="1")
    _, total, _, _ = check(cli, tmp_path, "ps4", pat, key=key, env=env)
    assert total >= 8
    check(cli, tmp_path, "ps4", pat, key=key)  # default groups: the same answer


def test_two_mock_devices(cli, tmp_path):
    """Above the 256 MiB multi-GPU threshold the groups are dealt to every device; each device's counts are
    summed at the end."""
    key = 0x1357BDF
    sizes = [1_000_000] * 270
    sizes[5] = 0
    hdr, _, _ = arkfixture.write_archive(str(tmp_path), n_files=len(sizes), n_parts=3, seed=31, body_key=key, sizes=sizes)
    env = dict(os.environ, MOD_MOCK_DEVICES="2", MOD_TRACE="1")
    pat = b"\x17\x2a"
    out = subprocess.run([cli, "-bodykey", str(key), "-findhex", pat.hex()], cwd=tmp_path, capture_output=True, timeout=600, env=env)
    assert out.returncode == 0
    assert "find pipeline" in out.stderr.decode() and "on 2 GPU(s)" in out.stderr.decode()
    stdout = out.stdout.decode("latin-1")
    want_lines, want_total, want_files = oracle_find(tmp_path, "ps4", pat, key)
    assert [ln for ln in stdout.splitlines() if "\t" in ln] == want_lines
    assert SUMMARY.search(stdout).groups() == (str(want_total), str(want_files))
    assert want_total > 1000


def test_pattern_length_limits(cli, tmp_path):
    planted_archive(tmp_path)
    assert "1 to 64 bytes" in run(cli, tmp_path, "-findhex", "", expect=1)
    assert "1 to 64 bytes" in run(cli, tmp_path, "-find", "x" * 65, expect=1)
    assert "pairs of hex digits" in run(cli, tmp_path, "-findhex", "abc", expect=1)
    run(cli, tmp_path, "-find", "x" * 64)
    assert "0 matches in 0 files" in run(cli, tmp_path, "-find", "no such text anywhere")
    assert "-findhex <hex>" in run(cli, tmp_path)


def test_corrupt_header_fails_like_unpack(cli, tmp_path):
    arkfixture.write_archive(str(tmp_path), n_files=10, seed=9)
    path = tmp_path / "main_ps4.hdr"
    good = path.read_bytes()
    for bad in (b"\x01\x02\x03\x04" + good[4:], good[:len(good) // 2]):
        path.write_bytes(bad)
        unpack = run(cli, tmp_path, "-unpack", "o", expect=1)
        find = run(cli, tmp_path, "-find", "abc", expect=1)
        assert unpack.splitlines()[-1] == find.splitlines()[-1]
    os.remove(path)
    assert "Failed to open file" in run(cli, tmp_path, "-find", "abc", expect=1)


def test_entry_outside_the_archive_is_refused(cli, tmp_path):
    entries = [ao.Entry(name="ps4/a.bin", offset=0, size=100), ao.Entry(name="ps4/b.bin", offset=90, size=100)]
    hdr = ao.Header(ps4=True, parts=[("main_ps4_0.ark", 150)], entries=entries)
    plain = ao.serialise_header(hdr)
    (tmp_path / "main_ps4.hdr").write_bytes(plain[:4] + oracle.cycle(np.frombuffer(plain[4:], np.uint8), ao.KEY_PS4).tobytes())
    (tmp_path / "main_ps4_0.ark").write_bytes(bytes(150))
    assert "lies outside the archive data" in run(cli, tmp_path, "-find", "abc", expect=1)


def test_duplicate_names_are_each_reported(cli, tmp_path):
    first, second = b"xxNEEDLExx", b"NEEDLE" + b"." * 20
    entries = [ao.Entry(name="ps4/dup.bin", offset=0, size=len(first)),
               ao.Entry(name="ps4/dup.bin", offset=len(first), size=len(second))]
    image = first + second
    hdr = ao.Header(ps4=True, parts=[("main_ps4_0.ark", len(image))], entries=entries)
    plain = ao.serialise_header(hdr)
    (tmp_path / "main_ps4.hdr").write_bytes(plain[:4] + oracle.cycle(np.frombuffer(plain[4:], np.uint8), ao.KEY_PS4).tobytes())
    (tmp_path / "main_ps4_0.ark").write_bytes(image)
    lines, total, files, _ = check(cli, tmp_path, "ps4", b"NEEDLE")
    assert total == 2 and files == 2 and sorted(lines) == ["ps4/dup.bin\t0", "ps4/dup.bin\t2"]


def test_facade_without_the_search_entry_points(cli, tmp_path):
    """Linked against an ABI implementation that predates the search (here the mock without mock_find_abi.cpp),
    the facade still links and loads, and -find reports that the search is missing."""
    import glob
    exe = os.path.join(BUILD, "modulate_mock_nosearch")
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cpp"))) + [os.path.join(CSRC, "cli", "modulate_main.cpp"),
                                                              os.path.join(ROOT, "tests", "cpp", "mock_abi.cpp")]
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           *srcs, "-L", os.path.join(ROOT, "oracle"), "-loracle", f"-Wl,-rpath,{os.path.join(ROOT, 'oracle')}"])
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=12, n_parts=2, seed=3)
    assert "has no search" in run(exe, tmp_path, "-find", "abc", expect=1)
    run(exe, tmp_path, "-unpack", "out")
    for e, p in zip(hdr.entries, payloads):
        assert (tmp_path / "out" / e.name).read_bytes() == p
