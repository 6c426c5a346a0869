"""CPU: the pattern-set search (-findlist / -findhexlist, CArk::FindSetInFiles, the owned-start bounds of the
slot-ring GPU step) driven end to end through the oracle-backed mock of the C ABI (tests/cpp/mock_abi.cpp,
mock_find_abi.cpp, mock_find_set_abi.cpp).  Expected results come from numpy over the oracle-deciphered entries:
every start compared with every pattern, so overlapping matches and several patterns at one start all count."""
import glob
import os
import re
import subprocess

import numpy as np
import pytest

import arkfixture
import oracle
from test_facade_host import BUILD, CSRC, ROOT, run
from test_find_host import MOCK_FIND, PIECE_GROUP, SUMMARY, cli as find_cli, image_of, planted_archive, positions  # noqa: F401
from test_ref_fixtures import CASES, MANIFEST, fixture_file_bytes, ref_header

MOCK_FIND_SET = os.path.join(BUILD, "modulate_mock_find_set")


@pytest.fixture(scope="session")
def cli():
    """modulate CLI linked against the oracle-backed mock ABI with its search and set-search entry points."""
    oracle.build()
    os.makedirs(BUILD, exist_ok=True)
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cpp"))) + [os.path.join(CSRC, "cli", "modulate_main.cpp")] + \
        [os.path.join(ROOT, "tests", "cpp", f) for f in ("mock_abi.cpp", "mock_find_abi.cpp", "mock_find_set_abi.cpp")]
    deps = srcs + glob.glob(os.path.join(CSRC, "*.h")) + [os.path.join(ROOT, "include", "modulate_b200.h")]
    if not os.path.exists(MOCK_FIND_SET) or any(os.path.getmtime(d) > os.path.getmtime(MOCK_FIND_SET) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"), "-o",
                               MOCK_FIND_SET, *srcs, "-L", os.path.join(ROOT, "oracle"), "-loracle",
                               f"-Wl,-rpath,{os.path.join(ROOT, 'oracle')}"])
    return MOCK_FIND_SET


def oracle_find_set(root, plat, pats, shown, key=0):
    """(match lines, per-pattern lines, total, files) the CLI must print."""
    hdr, _ = arkfixture.read_header(os.path.join(root, f"main_{plat}.hdr"))
    image = image_of(root, hdr)
    lines, counts, total, files = [], [0] * len(pats), 0, 0
    for e in hdr.entries:
        data = oracle.cycle(image[e.offset:e.offset + e.size], key) if key else image[e.offset:e.offset + e.size]
        hits = sorted((p, j) for j, pat in enumerate(pats) for p in positions(data, pat))
        for p, j in hits:
            counts[j] += 1
        total += len(hits)
        files += bool(hits)
        lines += [f"{e.name}\t{p}\t{shown[j]}" for p, j in hits]
    return lines, [f"{c}\t{s}" for c, s in zip(counts, shown)], total, files


def cli_find_set(cli, root, pats, *pre, env=None, hex_form=True, expect=0):
    """Write the list, run the CLI -> (match lines, count lines, total, files, stdout)."""
    path = os.path.join(root, "patterns.txt")
    with open(path, "wb") as f:
        f.write(b"".join((p.hex() if hex_form else p.decode("latin-1")).encode("latin-1") + b"\n" for p in pats))
    out = subprocess.run([cli, *pre, "-findhexlist" if hex_form else "-findlist", path], cwd=root, capture_output=True,
                         timeout=600, env=env)
    stdout = out.stdout.decode("latin-1")
    assert out.returncode == (0 if expect == 0 else 255), stdout + out.stderr.decode("latin-1")
    rows = [ln for ln in stdout.splitlines() if "\t" in ln]
    match_lines = [ln for ln in rows if ln.count("\t") == 2]
    count_lines = [ln for ln in rows if ln.count("\t") == 1]
    m = SUMMARY.search(stdout)
    return match_lines, count_lines, int(m.group(1)) if m else None, int(m.group(2)) if m else None, stdout


def check_set(cli, root, plat, pats, key=0, env=None, hex_form=True):
    pre = (["-ps3"] if plat == "ps3" else []) + (["-bodykey", str(key)] if key else [])
    shown = [p.hex() for p in pats] if hex_form else [p.decode("latin-1") for p in pats]
    got = cli_find_set(cli, root, pats, *pre, env=env, hex_form=hex_form)
    want = oracle_find_set(root, plat, pats, shown, key)
    assert got[1:4] == want[1:], (got[1:4], want[1:])
    if want[2] <= 10000:
        assert got[0] == want[0]
    return got


@pytest.mark.parametrize("case", CASES)
def test_find_set_in_reference_written_archives(cli, tmp_path, case):
    """The archives exactly as the reference wrote them: a mixed-length list equals numpy over the oracle."""
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
    pats = [some, some[:2], b"\x00", b"\x00\x00\x00\x00\x00", b"not in there at all", some[:1]]
    pats = list(dict.fromkeys(pats))
    _, _, total, _, _ = check_set(cli, tmp_path, plat, pats)
    assert total >= 1
    text = next(bytes(image[i:i + 4]) for i in range(len(image) - 4) if all(32 < b < 127 for b in image[i:i + 4]))
    check_set(cli, tmp_path, plat, [text, text[:3], text[1:]], hex_form=False)


def test_prefix_pairs_and_several_patterns_at_one_start(cli, tmp_path):
    hdr, pat = planted_archive(tmp_path)
    pats = [pat, pat[:2], pat[:3], b"aa", b"a", pat * 2, b"\x00"]
    lines, counts, total, files, _ = check_set(cli, tmp_path, "ps4", pats)
    # entry 1 starts with the pattern: every prefix of it is listed at offset 0, in list order
    first = [ln for ln in lines if ln.startswith(hdr.entries[1].name + "\t0\t")]
    assert first == [f"{hdr.entries[1].name}\t0\t{p.hex()}" for p in (pat, pat[:2], pat[:3])]


def test_list_parsing(cli, tmp_path):
    planted_archive(tmp_path)
    lst = tmp_path / "l.txt"

    def findlist(content, *args, hex_form=False, expect=0):
        lst.write_bytes(content)
        return run(cli, tmp_path, *args, "-findhexlist" if hex_form else "-findlist", str(lst), expect=expect)

    # CRLF and empty lines: the same as the plain list
    plain = findlist(b"SYMBOL\naa\n")
    assert findlist(b"\r\nSYMBOL\r\n\r\n\naa\r\n") == plain
    assert "\t2\tSYMBOL\n" not in plain and "SYMBOL" in plain
    hexed = findlist(b"53 59 4D\n\nAA bb\r\n", hex_form=True)
    assert "\t53594d\n" in hexed and "\taabb\n" in hexed
    assert "line 2 is not pairs of hex digits" in findlist(b"00\nabc\n", hex_form=True, expect=1)
    assert "line 2 is not pairs of hex digits" in findlist(b"00\nzz\n", hex_form=True, expect=1)
    assert "line 3 repeats the pattern of line 1" in findlist(b"abc\nabd\nabc\n", expect=1)
    assert "line 3 repeats the pattern of line 1" in findlist(b"0a0b\n0c\n0A 0B\n", hex_form=True, expect=1)
    assert "line 257: a list holds at most 256" in findlist(b"".join(b"p%03d\n" % i for i in range(257)), expect=1)
    findlist(b"".join(b"p%03d\n" % i for i in range(256)))
    assert "line 2: the pattern must be 1 to 64 bytes" in findlist(b"ok\n" + b"x" * 65 + b"\n", expect=1)
    findlist(b"x" * 64 + b"\n")
    assert "holds no pattern" in findlist(b"\n\r\n", expect=1)
    assert "cannot read" in run(cli, tmp_path, "-findlist", str(tmp_path / "missing.txt"), expect=1)
    usage = run(cli, tmp_path)
    assert "-findlist <file>" in usage and "-findhexlist <file>" in usage


def test_output_order_and_the_line_cut(cli, tmp_path):
    """More than 10 000 matches: the first 10 000 lines in (table, offset, list) order, '... N more', then the
    exact count of every pattern and the summary."""
    sizes = [3000] * 8
    contents = {i: bytes([0x41]) * 3000 for i in range(8)}
    arkfixture.write_archive(str(tmp_path), n_files=len(sizes), n_parts=2, seed=5, sizes=sizes, contents=contents)
    pats = [b"AA", b"A", b"AAAA", b"B"]
    lines, counts, total, files, stdout = cli_find_set(cli, tmp_path, pats)
    want_lines, want_counts, want_total, want_files = oracle_find_set(tmp_path, "ps4", pats, [p.hex() for p in pats])
    assert (counts, total, files) == (want_counts, want_total, want_files)
    assert want_total > 10000 and lines == want_lines[:10000]
    assert f"... {want_total - 10000} more" in stdout
    tail = stdout.splitlines()
    at = tail.index(counts[0])
    assert tail[at:at + 5] == counts + [f"{total} matches in {files} files"]
    assert counts[3] == "0\t42"


@pytest.mark.parametrize("key", [0x7FFFFFFF, -0x80000000, -1, 1, 0x12345678])
def test_body_key_edge_keys(cli, tmp_path, key):
    _, pat = planted_archive(tmp_path, key=key)
    _, _, total, _, _ = check_set(cli, tmp_path, "ps4", [pat, pat[2:5], b"\x00", b"ab"], key=key)
    assert total >= 5


def test_two_mock_devices(cli, tmp_path):
    key = 0x1357BDF
    sizes = [1_000_000] * 270
    sizes[5] = 0
    arkfixture.write_archive(str(tmp_path), n_files=len(sizes), n_parts=3, seed=31, body_key=key, sizes=sizes)
    env = dict(os.environ, MOD_MOCK_DEVICES="2", MOD_TRACE="1")
    pats = [b"\x17\x2a", b"\x99", b"\x01\x02\x03"]
    out = subprocess.run([cli, "-bodykey", str(key), "-findhexlist", "/dev/stdin"], cwd=tmp_path, capture_output=True,
                         timeout=600, env=env, input=b"".join(p.hex().encode() + b"\n" for p in pats))
    assert out.returncode == 0, out.stdout.decode("latin-1")
    assert "on 2 GPU(s)" in out.stderr.decode()
    stdout = out.stdout.decode("latin-1")
    want_lines, want_counts, want_total, want_files = oracle_find_set(tmp_path, "ps4", pats, [p.hex() for p in pats], key)
    rows = [ln for ln in stdout.splitlines() if "\t" in ln]
    assert [ln for ln in rows if ln.count("\t") == 1] == want_counts
    assert SUMMARY.search(stdout).groups() == (str(want_total), str(want_files))
    assert want_total > 10000


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


def test_owned_starts_at_every_piece_cut(cli, tmp_path):
    """A set of lengths {1, 17, 64} with MOD_IO_GROUP_MIB=1: the pieces overlap by 63 bytes, and the 1- and 17-byte
    patterns planted in those 63 bytes must be counted once (the owned-start bounds), like with whole entries."""
    rng = np.random.default_rng(3)
    pats = [b"\xe7", bytes(int(x) for x in rng.integers(0, 256, 17)), bytes(int(x) for x in rng.integers(0, 256, 64))]
    key = owned_trap_archive(tmp_path, pats)
    env = dict(os.environ, MOD_IO_GROUP_MIB="1")
    _, counts, total, _, _ = check_set(cli, tmp_path, "ps4", pats, key=key, env=env)
    assert int(counts[1].split("\t")[0]) >= 6 and int(counts[2].split("\t")[0]) >= 2
    assert check_set(cli, tmp_path, "ps4", pats, key=key)[2] == total  # whole entries: the same answer


def test_facade_without_the_set_search_entry_points(find_cli, tmp_path):
    """Linked against an ABI implementation with the single-pattern search but without the set entry points (the
    mock without mock_find_set_abi.cpp), the facade still links, -find works and -findlist says what is missing."""
    arkfixture.write_archive(str(tmp_path), n_files=12, n_parts=2, seed=3)
    (tmp_path / "l.txt").write_bytes(b"abc\n")
    assert "has no set search" in run(find_cli, tmp_path, "-findlist", str(tmp_path / "l.txt"), expect=1)
    assert re.search(r"\d+ matches in \d+ files", run(find_cli, tmp_path, "-find", "abc"))
