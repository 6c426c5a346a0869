"""CPU: everything either side of the cipher, against fixtures PRODUCED BY THE REFERENCE ITSELF.

tests/golden/ark/ and tests/golden/dtb/ were written by tests/golden/make_ark_golden.py, which runs
the reference's own CArk.cpp / CDtaFile.cpp (compiled by `make -C oracle ark_ref`): the .hdr files
are what its SaveArk wrote, `loaded_files` what its Load parsed back, `built_parts` what its BuildArk
assigned, `extracted_sha256` what its ExtractFiles wrote, *.ref.dtb what CDtaFile::Load + Save made of
*.in.dtb.  Checked here, bit-exact:

  * the Python restatement (oracle/ark_oracle.py, oracle/dta_oracle.py): reader, PS3 and PS4 writers,
    BuildArk offsets and part split, DTB codec;
  * the product's host-side C++ (csrc/ArkHeader.cpp, CArk.cpp, CDtaFile.cpp, the CLI) through the
    mock of the C ABI: -pack / -pack_add reproduce the reference's header bytes and part files,
    -unpack of a reference-written archive reproduces its extracted files, -dtacopy its DTB bytes.

Header bytes 12..27 (mChecksumData) are uninitialised stack in the reference (CArk.cpp:911-921) and
are masked on both sides.
"""
import hashlib
import json
import os
import shutil

import numpy as np
import pytest

import oracle
import synth
from oracle import ark_oracle as ao
from oracle import dta_oracle as do
from arkfixture import CASES, GOLD, MANIFEST, fixture_file_bytes, ref_header, run
from searchutil import mock_cli

with open(os.path.join(GOLD, "dtb", "index.json")) as _f:
    DTB_INDEX = json.load(_f)
SONGS = MANIFEST["songs"]


@pytest.fixture(scope="session")
def cli():
    """modulate CLI on the mock ABI, without the search entry points."""
    return mock_cli(0)


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def masked(hdr: bytes) -> bytes:
    b = bytearray(hdr)
    b[12:28] = b"\0" * 16
    return bytes(b)


def decipher(raw: bytes) -> bytes:
    magic = int.from_bytes(raw[:4], "little")
    return raw[:4] + oracle.cycle(np.frombuffer(raw[4:], dtype=np.uint8), ao.platform_key(magic)).tobytes()


def entries_of(table):
    return [ao.Entry(name=f["name"], offset=f["offset"], size=f["size"], flags1=f["flags1"], flags2=f["flags2"],
                     hash=f["hash"]) for f in table]


# ---- the Python restatement against the reference's output -------------------------------------------

@pytest.mark.parametrize("case", CASES)
def test_restated_reader_matches_reference_load(case):
    info = MANIFEST[case]
    hdr = ao.parse_header(decipher(ref_header(case)))
    got = [dict(name=e.name, offset=e.offset, size=e.size, flags1=e.flags1, flags2=e.flags2, hash=e.hash)
           for e in hdr.entries]
    assert got == info["loaded_files"]
    assert [{"path": p, "size": s} for p, s in hdr.parts] == info["loaded_parts"]
    assert hdr.ps4 == (info["platform"] == "ps4")


@pytest.mark.parametrize("case", CASES)
def test_restated_writer_matches_reference_save(case):
    """Entries in the order BuildArk left them (built_files) -> lSaveHeader's bytes, PS3 bucket order
    and PS4 path order included, bucket chains and the trailing bucket-head table included."""
    info = MANIFEST[case]
    hdr = ao.Header(ps4=info["platform"] == "ps4", parts=[(p["path"], p["size"]) for p in info["built_parts"]],
                    entries=entries_of(info["built_files"]))
    assert masked(ao.serialise_header(hdr)) == masked(decipher(ref_header(case)))


@pytest.mark.parametrize("case", CASES)
def test_restated_build_ark_matches_reference(case):
    """ConstructFromDirectory's allowance plan (CArk.cpp:211-217) + BuildArk's byte-packed offsets and
    exceed-then-close part split (CArk.cpp:784-824)."""
    info = MANIFEST[case]
    sizes = [f["size"] for f in info["built_files"]]
    offsets, parts = ao.build_ark(sizes, ao.plan_part_sizes(sum(sizes), len(info["built_parts"])))
    assert offsets == [f["offset"] for f in info["built_files"]]
    assert parts == [p["size"] for p in info["built_parts"]]
    assert len(parts) >= 3 and min(parts) > 0  # the fixtures do exercise the split


def test_fixtures_cover_the_edge_cases():
    for case in CASES:
        info = MANIFEST[case]
        files = info["loaded_files"]
        assert any(f["size"] == 0 and f["offset"] == 0 and f["hash"] == 0 for f in files)  # zero-size entries
        n = len(files)
        buckets = [ao.file_hash(f["name"], n) for f in files]
        assert len(set(buckets)) < n  # colliding name-hash buckets -> flags1 chains
        assert any(f["flags1"] != -1 for f in files)
    # -pack: the song list came from the DTA configs (CUSTOM1 is configured, Custom_Two is not), the
    # built-in songs are always kept, new files are ignored
    for plat in ("ps3", "ps4"):
        names = {f["name"] for f in MANIFEST[f"{plat}_pack"]["loaded_files"]}
        assert not any("/songs/Custom_Two/" in n or "zz_new_file" in n for n in names)
        assert any("/songs/credits/" in n for n in names) and any("/songs/Custom1/" in n for n in names)


# ---- the product's host-side C++ against the reference's output ------------------------------------------

def stage_case(tmp_path, case):
    """cwd for the CLI: the seed header as main_<plat>.hdr and the regenerated input tree in in/."""
    info = MANIFEST[case]
    plat = info["platform"]
    shutil.copy(os.path.join(GOLD, "ark", case, "seed.hdr"), tmp_path / f"main_{plat}.hdr")
    for f in info["input"]:
        path = tmp_path / "in" / f["name"]
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_bytes(fixture_file_bytes(f))
    args = ([] if plat == "ps4" else ["-ps3"]) + (["-packall"] if info["pack_all"] else [])
    args += ["-pack" if info["ignore_new"] else "-pack_add", "in", "out"]
    return info, plat, args


@pytest.mark.parametrize("case", CASES)
def test_cpp_pack_reproduces_reference_header_and_parts(cli, tmp_path, case):
    info, plat, args = stage_case(tmp_path, case)
    run(cli, tmp_path, *args)
    got = (tmp_path / "out" / f"main_{plat}.hdr").read_bytes()
    want = ref_header(case)
    assert len(got) == len(want)
    assert masked(decipher(got)) == masked(decipher(want))  # plaintext view: readable diffs
    assert got[:12] == want[:12] and got[28:] == want[28:]   # and the ciphered bytes as written
    for part, digest in zip(info["loaded_parts"], info["part_sha256"]):
        blob = (tmp_path / "out" / part["path"]).read_bytes()
        assert len(blob) == part["size"] and sha(blob) == digest, part


@pytest.mark.parametrize("case", CASES)
def test_cpp_unpack_of_reference_written_archive(cli, tmp_path, case):
    """The archive exactly as the reference wrote it (its header; its part files, rebuilt from the
    manifest and verified by sha256) -> the files the reference's own ExtractFiles produced."""
    info = MANIFEST[case]
    plat = info["platform"]
    (tmp_path / f"main_{plat}.hdr").write_bytes(ref_header(case))
    by_name = {f["name"]: f for f in info["input"]}
    image = bytearray(sum(p["size"] for p in info["loaded_parts"]))
    for f in info["loaded_files"]:
        src = by_name[f["name"]]
        image[f["offset"]:f["offset"] + f["size"]] = fixture_file_bytes(src)
    pos = 0
    for part, digest in zip(info["loaded_parts"], info["part_sha256"]):
        blob = bytes(image[pos:pos + part["size"]])
        assert sha(blob) == digest
        (tmp_path / part["path"]).write_bytes(blob)
        pos += part["size"]
    run(cli, tmp_path, *([] if plat == "ps4" else ["-ps3"]), "-unpack", "ext")
    for name, digest in info["extracted_sha256"].items():
        assert sha((tmp_path / "ext" / name).read_bytes()) == digest, name


def test_cpp_song_list_matches_reference_getsongs(cli, tmp_path):
    """GetSongs + GetSongData (CDtaFile.cpp:102-181, :248-294) through the CLI's -listsongs, against the
    list the reference derived from the same two configs."""
    import arkfixture
    cfg, songs_cfg = arkfixture.song_config_blobs()
    d = tmp_path / "in" / "ps4" / "config"
    d.mkdir(parents=True)
    (d / "amp_config.dta_dta_ps4").write_bytes(cfg)
    (d / "amp_songs_config.dta_dta_ps4").write_bytes(songs_cfg)
    out = run(cli, tmp_path, "-listsongs", "in")
    assert len(SONGS) == 3 and SONGS[0]["path"] == "../songs/custom1/custom1.moggsong"  # lower-cased by GetSongData
    for i, sg in enumerate(SONGS):
        want = (f"Song {i + 1}\t  {sg['id']} - {sg['name']} - {sg['type']}\n\t  {sg['path']}\n\t  Unlocked by "
                f"{sg['unlock_method']} {sg['unlock_count']}\n\t  Arena: {sg['arena']}\n")
        assert want in out, (want, out)
    assert f"Song {len(SONGS) + 1}" not in out


# ---- DTB ----------------------------------------------------------------------------------------------------

DTB_CASES = sorted(k for k in DTB_INDEX if not k.startswith("reject_"))


@pytest.mark.parametrize("name", DTB_CASES)
def test_dtb_codecs_match_reference_load_save(cli, tmp_path, name):
    src = open(os.path.join(GOLD, "dtb", name + ".in.dtb"), "rb").read()
    want = open(os.path.join(GOLD, "dtb", name + ".ref.dtb"), "rb").read()
    assert sha(src) == DTB_INDEX[name]["in_sha256"] and sha(want) == DTB_INDEX[name]["ref_sha256"]
    assert do.save_like_reference(do.parse(src)) == want
    (tmp_path / "in.dtb").write_bytes(src)
    run(cli, tmp_path, "-dtacopy", "in.dtb", "out.dtb")
    assert (tmp_path / "out.dtb").read_bytes() == want


def test_dtb_two_top_level_trees_lose_their_separator_like_the_reference():
    """CDtaFile::Save writes the root's children back to back (CDtaFile.cpp:371-374) although Load
    expects (type, 1) between top-level trees (:93-94): the reference does not round-trip such files."""
    assert not DTB_INDEX["two_trees"]["identical"]
    assert all(DTB_INDEX[k]["identical"] for k in DTB_CASES if k != "two_trees")


@pytest.mark.parametrize("name", sorted(k for k in DTB_INDEX if k.startswith("reject_")))
def test_dtb_inputs_the_reference_rejects(cli, tmp_path, name):
    assert DTB_INDEX[name]["rc"] == 6  # eError_InvalidData
    blob = open(os.path.join(GOLD, "dtb", name + ".dtb"), "rb").read()
    with pytest.raises(do.DtaError):
        do.parse(blob)
    (tmp_path / "bad.dtb").write_bytes(blob)
    assert "Bad data" in run(cli, tmp_path, "-dtacopy", "bad.dtb", "o.dtb", expect=1)
