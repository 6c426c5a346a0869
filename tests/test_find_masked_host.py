"""CPU: the wildcard and case-insensitive searches (-findwild / -findi / -findilist, CArk::FindMaskedInFiles,
CArk::FindSetInFiles with lbIgnoreCase) driven end to end through the oracle-backed mock of the C ABI
(tests/cpp/mock_abi.cpp, mock_find_abi.cpp).  Expected results come from the numpy reference of tests/searchutil.py
over the oracle-deciphered entries: every start compared under the mask, or after ASCII case folding."""
import os
import re
import subprocess

import pytest

import arkfixture
from arkfixture import MANIFEST, CASES, fixture_file_bytes, ref_header, run
from searchutil import (SUMMARY, check_nocase, check_nocase_set, check_wild, expected_output, mock_cli, piece_cut_archive,
                        planted_archive)


@pytest.fixture(scope="session")
def cli():
    """modulate CLI on the mock ABI with every search entry point, the masked ones and folded sets included."""
    return mock_cli(3)


@pytest.fixture(scope="session")
def old_cli():
    """The same on a library that predates the masked entry points (single-pattern and set search only)."""
    return mock_cli(2)


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
    _, _, want_total, want_files = expected_output(tmp_path, "ps4", [b"\x17\x0a"], [b"\xff\x0f"], key=key)
    assert SUMMARY.search(out.stdout.decode("latin-1")).groups() == (str(want_total), str(want_files))
    assert want_total > 10000


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
