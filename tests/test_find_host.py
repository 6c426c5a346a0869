"""CPU: the archive search (-find / -findhex, CArk::FindInFiles, the slot-ring GPU step) driven end to end
through the oracle-backed mock of the C ABI (tests/cpp/mock_abi.cpp, mock_find_abi.cpp).  Expected results come
from the oracle: every entry deciphered, then every start position compared, so overlapping matches count."""
import os
import subprocess

import numpy as np
import pytest

import arkfixture
import oracle
from oracle import ark_oracle as ao
from arkfixture import CASES, MANIFEST, fixture_file_bytes, ref_header, run
from searchutil import SUMMARY, check, cli_find, expected_output, mock_cli, piece_cut_archive, planted_archive


@pytest.fixture(scope="session")
def cli():
    """modulate CLI on the mock ABI of a library with the single-pattern search (g++ only, no CUDA)."""
    return mock_cli(1)


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
    want_lines, _, want_total, want_files = expected_output(tmp_path, "ps4", [pat], key=key)
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
    """Linked against an ABI implementation that predates the search (here the mock of generation 0),
    the facade still links and loads, and -find reports that the search is missing."""
    exe = mock_cli(0)
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=12, n_parts=2, seed=3)
    assert "has no search" in run(exe, tmp_path, "-find", "abc", expect=1)
    run(exe, tmp_path, "-unpack", "out")
    for e, p in zip(hdr.entries, payloads):
        assert (tmp_path / "out" / e.name).read_bytes() == p
