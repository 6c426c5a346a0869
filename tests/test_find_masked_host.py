"""CPU: the wildcard and case-insensitive searches (-findwild / -findi / -findilist, CArk::FindMaskedInFiles,
CArk::FindSetInFiles with lbIgnoreCase) driven end to end through the oracle-backed mock of the C ABI
(tests/cpp/mock_abi.cpp, mock_find_abi.cpp and mock_find_masked_abi.cpp, which also answers the set entry points with
sets that may be folded).  Expected results come from numpy over the oracle-deciphered entries: every start compared
under the mask, or after ASCII case folding."""
import glob
import os
import re
import subprocess

import numpy as np
import pytest

import arkfixture
import kernel_model_masked as kmm
import oracle
from test_facade_host import BUILD, CSRC, ROOT, run
from test_find_host import PIECE_GROUP, SUMMARY, image_of, piece_cut_archive, planted_archive  # noqa: F401
from test_ref_fixtures import CASES, MANIFEST, fixture_file_bytes, ref_header

MOCK_FIND_MASKED = os.path.join(BUILD, "modulate_mock_find_masked")
MOCK_NO_MASKED = os.path.join(BUILD, "modulate_mock_no_masked")
FOLD = np.array([kmm.fold(b) for b in range(256)], np.uint8)


def _link(out, mocks):
    oracle.build()
    os.makedirs(BUILD, exist_ok=True)
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cpp"))) + [os.path.join(CSRC, "cli", "modulate_main.cpp")] + \
        [os.path.join(ROOT, "tests", "cpp", f) for f in mocks]
    deps = srcs + glob.glob(os.path.join(CSRC, "*.h")) + [os.path.join(ROOT, "include", "modulate_b200.h")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"), "-o",
                               out, *srcs, "-L", os.path.join(ROOT, "oracle"), "-loracle",
                               f"-Wl,-rpath,{os.path.join(ROOT, 'oracle')}"])
    return out


@pytest.fixture(scope="session")
def cli():
    """modulate CLI linked against the mock ABI with every search entry point, the masked ones included
    (mock_find_masked_abi.cpp takes the place of mock_find_set_abi.cpp)."""
    return _link(MOCK_FIND_MASKED, ("mock_abi.cpp", "mock_find_abi.cpp", "mock_find_masked_abi.cpp"))


@pytest.fixture(scope="session")
def old_cli():
    """The same without mock_find_masked_abi.cpp: a library that predates the masked entry points."""
    return _link(MOCK_NO_MASKED, ("mock_abi.cpp", "mock_find_abi.cpp", "mock_find_set_abi.cpp"))


def wild_hex(value: bytes, mask: bytes) -> str:
    """The -findwild text of (value, mask) with nibble masks only."""
    out = []
    for v, m in zip(value, mask):
        out.append("".join("%x" % ((v >> s) & 15) if (m >> s) & 15 == 15 else "?" for s in (4, 0)))
    return " ".join(out)


def entries(root, plat, key):
    hdr, _ = arkfixture.read_header(os.path.join(root, f"main_{plat}.hdr"))
    image = image_of(root, hdr)
    for e in hdr.entries:
        yield e, (oracle.cycle(image[e.offset:e.offset + e.size], key) if key else image[e.offset:e.offset + e.size])


def oracle_masked(root, plat, value, mask, key=0):
    """(lines, total, files) the CLI must print for a masked search."""
    lines, total, files = [], 0, 0
    for e, data in entries(root, plat, key):
        pos = kmm.masked_positions(data, value, mask)
        total += len(pos)
        files += bool(pos)
        lines += [f"{e.name}\t{p}" for p in pos]
    return lines, total, files


def cli_out(cli, root, *args, env=None, expect=0):
    out = subprocess.run([cli, *args], cwd=root, capture_output=True, timeout=600, env=env)
    stdout = out.stdout.decode("latin-1")
    assert out.returncode == (0 if expect == 0 else 255), stdout + out.stderr.decode("latin-1")
    m = SUMMARY.search(stdout)
    lines = [ln for ln in stdout.splitlines() if "\t" in ln]
    return lines, int(m.group(1)) if m else None, int(m.group(2)) if m else None, stdout


def _pre(plat, key):
    return (["-ps3"] if plat == "ps3" else []) + (["-bodykey", str(key)] if key else [])


def check_wild(cli, root, plat, value, mask, key=0, env=None):
    got = cli_out(cli, root, *_pre(plat, key), "-findwild", wild_hex(value, mask), env=env)
    want = oracle_masked(root, plat, bytes(v & m for v, m in zip(value, mask)), mask, key)
    assert got[1:3] == want[1:], (value.hex(), mask.hex())
    if want[1] <= 10000:
        assert got[0] == want[0]
    return got


def check_nocase(cli, root, plat, text: bytes, key=0):
    got = cli_out(cli, root, *_pre(plat, key), "-findi", text)
    folded = bytes(FOLD[np.frombuffer(text, np.uint8)])
    mask = bytes(0xDF if 0x41 <= b <= 0x5A else 0xFF for b in folded)
    want = oracle_masked(root, plat, folded, mask, key)
    assert got[1:3] == want[1:], text
    if want[1] <= 10000:
        assert got[0] == want[0]
    assert f"for {len(text)} bytes, ignoring case" in got[3]
    return got


def oracle_nocase_set(root, plat, pats, key=0):
    lines, counts, total, files = [], [0] * len(pats), 0, 0
    for e, data in entries(root, plat, key):
        fdata = FOLD[data]
        hits = sorted((p, j) for j, pat in enumerate(pats)
                      for p in kmm.masked_positions(fdata, bytes(FOLD[np.frombuffer(pat, np.uint8)]), b"\xff" * len(pat)))
        for _, j in hits:
            counts[j] += 1
        total += len(hits)
        files += bool(hits)
        lines += [f"{e.name}\t{p}\t{pats[j].decode('latin-1')}" for p, j in hits]
    return lines, [f"{c}\t{p.decode('latin-1')}" for c, p in zip(counts, pats)], total, files


def check_nocase_set(cli, root, plat, pats, key=0):
    (root / "ilist.txt").write_bytes(b"".join(p + b"\n" for p in pats))
    lines, total, files, stdout = cli_out(cli, root, *_pre(plat, key), "-findilist", str(root / "ilist.txt"))
    want_lines, want_counts, want_total, want_files = oracle_nocase_set(root, plat, pats, key)
    assert (total, files) == (want_total, want_files)
    assert [ln for ln in lines if ln.count("\t") == 1] == want_counts
    if want_total <= 10000:
        assert [ln for ln in lines if ln.count("\t") == 2] == want_lines
    assert f"for {len(pats)} patterns, ignoring case" in stdout
    return total


def _reference_archive(tmp_path, case):
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
    return plat, bytes(image)


@pytest.mark.parametrize("case", CASES)
def test_masked_searches_in_reference_written_archives(cli, tmp_path, case):
    """The archives exactly as the reference wrote them: -findwild, -findi and -findilist equal numpy."""
    plat, image = _reference_archive(tmp_path, case)
    some = next(image[i:i + 6] for i in range(0, len(image) - 6, 97) if len(set(image[i:i + 6])) > 3)
    _, total, _, _ = check_wild(cli, tmp_path, plat, some, b"\x00\xff\xf0\xff\x0f\x00")
    assert total >= 1
    check_wild(cli, tmp_path, plat, some[:2], b"\xff\x00")
    check_wild(cli, tmp_path, plat, b"\x00", b"\xf0")
    text = next(image[i:i + 5] for i in range(len(image) - 5) if all(0x41 <= (b & 0xDF) <= 0x5A for b in image[i:i + 5]))
    assert check_nocase(cli, tmp_path, plat, text.swapcase())[1] >= 1
    check_nocase(cli, tmp_path, plat, text[:1].lower())
    assert check_nocase_set(cli, tmp_path, plat, [text.swapcase(), text[1:4].lower(), b"@", b"[", text[:1]]) >= 1


def test_case_folding_and_non_letters(cli, tmp_path):
    """-findi folds A-Z / a-z only: '@' / '`', '[' / '{' and bytes >= 0x80 match only themselves."""
    contents = {0: b"Amplitude AMPLITUDE amplitude aMpLiTuDe", 1: b"@`[{\xc1\xe1\xdf\xff_\x7f" * 3, 2: b"symbol SYMBOL"}
    arkfixture.write_archive(str(tmp_path), n_files=4, n_parts=1, seed=7, sizes=[len(contents[0]), 30, 13, 100],
                             contents=contents)
    assert check_nocase(cli, tmp_path, "ps4", b"amplitude")[1] == 4
    for b in (b"@", b"`", b"[", b"{", b"\xc1", b"\xe1", b"\xdf", b"\xff", b"_", b"\x7f"):
        check_nocase(cli, tmp_path, "ps4", b)
    assert check_nocase_set(cli, tmp_path, "ps4", [b"AMPLITUDE", b"sym", b"s", b"@`", b"\xc1"]) >= 8


def test_parse_errors(cli, tmp_path):
    planted_archive(tmp_path)

    def wild(text, expect=0):
        return run(cli, tmp_path, "-findwild", text, expect=expect)

    assert "-findwild takes pairs of hex digits, any of them ?" in wild("0a?", expect=1)
    assert "-findwild takes pairs of hex digits, any of them ?" in wild("0x??", expect=1)
    assert "-findwild takes pairs of hex digits, any of them ?" in wild("g0", expect=1)
    assert "The pattern must be 1 to 64 bytes long" in wild("", expect=1)
    assert "The pattern must be 1 to 64 bytes long" in wild("??" * 64 + "00", expect=1)
    assert "has no hex digit that is not ?" in wild("?? ??", expect=1)
    assert re.search(r"\d+ matches in \d+ files", wild("?? 5? 4D"))
    assert re.search(r"\d+ matches in \d+ files", wild("??" * 63 + "0?"))
    assert "-findhex takes pairs of hex digits" in run(cli, tmp_path, "-findhex", "4?", expect=1)
    assert "The pattern must be 1 to 64 bytes long" in run(cli, tmp_path, "-findi", "x" * 65, expect=1)
    lst = tmp_path / "l.txt"
    lst.write_bytes(b"Symbol\nother\nSYMBOL\n")
    assert "-findilist: line 3 repeats the pattern of line 1 ignoring case" in \
        run(cli, tmp_path, "-findilist", str(lst), expect=1)
    lst.write_bytes(b"ok\n" + b"x" * 65 + b"\n")
    assert "-findilist: line 2: the pattern must be 1 to 64 bytes" in run(cli, tmp_path, "-findilist", str(lst), expect=1)
    lst.write_bytes(b"@\n`\n[\n{\n")  # not letters: four different patterns
    run(cli, tmp_path, "-findilist", str(lst))
    usage = run(cli, tmp_path)
    assert "-findi <text>" in usage and "-findilist <file>" in usage and "-findwild <hex>" in usage


@pytest.mark.parametrize("L", [1, 2, 17, 64])
def test_wildcards_at_both_ends_across_every_piece_cut(cli, tmp_path, L):
    """MOD_IO_GROUP_MIB=1: pieces overlap by L - 1 bytes; a masked pattern with wildcards at both ends finds every
    planted match exactly once, as with whole entries."""
    pat, key = piece_cut_archive(tmp_path, L)
    mask = b"\x0f" if L == 1 else b"\x00\xff" if L == 2 else b"\x00" + b"\xff" * (L - 2) + b"\x00"
    env = dict(os.environ, MOD_IO_GROUP_MIB="1")
    _, total, _, _ = check_wild(cli, tmp_path, "ps4", pat, mask, key=key, env=env)
    assert total >= 8
    assert check_wild(cli, tmp_path, "ps4", pat, mask, key=key)[1] == total


def test_two_mock_devices(cli, tmp_path):
    key = 0x1357BDF
    sizes = [1_000_000] * 270
    arkfixture.write_archive(str(tmp_path), n_files=len(sizes), n_parts=3, seed=31, body_key=key, sizes=sizes)
    env = dict(os.environ, MOD_MOCK_DEVICES="2", MOD_TRACE="1")
    out = subprocess.run([cli, "-bodykey", str(key), "-findwild", "17 ?a"], cwd=tmp_path, capture_output=True, timeout=600,
                         env=env)
    assert out.returncode == 0 and "on 2 GPU(s)" in out.stderr.decode()
    want = oracle_masked(tmp_path, "ps4", b"\x17\x0a", b"\xff\x0f", key)
    assert SUMMARY.search(out.stdout.decode("latin-1")).groups() == (str(want[1]), str(want[2]))
    assert want[1] > 10000


def test_facade_without_the_masked_entry_points(old_cli, tmp_path):
    """Linked against an ABI implementation without the masked and case-folded entry points, the facade still links,
    -find and -findlist work, and the new commands say what is missing."""
    arkfixture.write_archive(str(tmp_path), n_files=12, n_parts=2, seed=3)
    (tmp_path / "l.txt").write_bytes(b"abc\n")
    assert re.search(r"\d+ matches in \d+ files", run(old_cli, tmp_path, "-find", "abc"))
    assert re.search(r"\d+ matches in \d+ files", run(old_cli, tmp_path, "-findlist", str(tmp_path / "l.txt")))
    assert "has no masked search (mod_plan_find_masked_window)" in run(old_cli, tmp_path, "-findwild", "0?", expect=1)
    assert "has no masked search" in run(old_cli, tmp_path, "-findi", "Abc", expect=1)
    assert "has no case-insensitive set search (mod_pattern_set_create_nocase)" in \
        run(old_cli, tmp_path, "-findilist", str(tmp_path / "l.txt"), expect=1)
