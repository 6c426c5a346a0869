"""CPU: the host-side C++ (CArk facade, ArkHeader codec, CLI) driven end to end through a MOCK of
the C ABI that answers with the oracle (tests/cpp/mock_abi.cpp).  Same flows run on the GPU with
the real library in tests/test_gpu_facade.py."""
import os
import subprocess

import numpy as np
import pytest

import oracle
import synth
from oracle import ark_oracle as ao
import arkfixture
from arkfixture import check_unpacked, reconstruct_walk, run
from searchutil import ROOT, link, mock_cli


@pytest.fixture(scope="session")
def cli():
    """modulate CLI linked against the oracle-backed mock ABI, without the search entry points (g++ only, no CUDA)."""
    return mock_cli(0)


@pytest.mark.parametrize("ps4", [True, False])
def test_unpack_matches_oracle_gather(cli, tmp_path, ps4):
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), ps4=ps4, n_files=80, n_parts=3, seed=3)
    # the oracle's own view of the archive: parts -> flat image -> gather by (offset, size)
    blobs = [open(tmp_path / p, "rb").read() for p, _ in hdr.parts]
    assert ao.extract(hdr.entries, ao.load_ark_data(blobs)) == payloads
    args = ([] if ps4 else ["-ps3"]) + ["-unpack", "out"]
    stdout = run(cli, tmp_path, *args)
    assert "Complete!" in stdout
    check_unpacked(tmp_path / "out", hdr, payloads)


def test_unpack_with_body_key(cli, tmp_path):
    key = 0x12345678
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=40, n_parts=2, seed=5, body_key=key)
    run(cli, tmp_path, "-bodykey", str(key), "-unpack", "out")
    check_unpacked(tmp_path / "out", hdr, payloads)


def test_decode_matches_oracle(cli, tmp_path):
    for ps4 in (True, False):
        d = tmp_path / ("p4" if ps4 else "p3")
        _, _, plain = arkfixture.write_archive(str(d), ps4=ps4, n_files=30, seed=7)
        run(cli, d, *([] if ps4 else ["-ps3"]), "-decode")
        plat = "ps4" if ps4 else "ps3"
        assert open(d / f"main_{plat}.hdr.dec", "rb").read() == plain


def test_load_rejects_bad_headers(cli, tmp_path):
    hdr, _, plain = arkfixture.write_archive(str(tmp_path), n_files=10, seed=9)
    path = tmp_path / "main_ps4.hdr"
    good = path.read_bytes()
    path.write_bytes(b"\x01\x02\x03\x04" + good[4:])                # unknown magic
    assert "Unknown version number" in run(cli, tmp_path, "-unpack", "o", expect=1)
    bad = bytearray(plain)
    bad[4 + 24:4 + 28] = (101).to_bytes(4, "little")                # numArks > 100
    enc = bytes(bad[:4]) + oracle.cycle(np.frombuffer(bytes(bad[4:]), np.uint8), ao.KEY_PS4).tobytes()
    path.write_bytes(enc)
    assert "Value of out bounds" in run(cli, tmp_path, "-unpack", "o", expect=1)
    path.write_bytes(good[:len(good) // 2])                          # truncated: bounds-checked, not UB
    assert "Bad data" in run(cli, tmp_path, "-unpack", "o", expect=1)
    os.remove(path)
    assert "Failed to open file" in run(cli, tmp_path, "-unpack", "o", expect=1)


@pytest.mark.parametrize("ps4", [True, False])
def test_pack_roundtrip_offsets_parts_and_header_bytes(cli, tmp_path, ps4):
    """unpack -> pack_add -packall -> the rebuilt set: offsets and part sizes follow the oracle's
    BuildArk restatement, the image is the byte-packed payloads, and the header bytes equal the
    oracle's serialiser (PS3: its own bucket order; PS4: the order the C++ chose)."""
    plat = "ps4" if ps4 else "ps3"
    pre = [] if ps4 else ["-ps3"]
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), ps4=ps4, n_files=70, n_parts=3, seed=11)
    run(cli, tmp_path, *pre, "-unpack", "unpacked")
    run(cli, tmp_path, *pre, "-packall", "-pack_add", "unpacked", "repacked")
    new, plain = arkfixture.read_header(str(tmp_path / "repacked" / f"main_{plat}.hdr"))
    by_name = {e.name: p for e, p in zip(hdr.entries, payloads)}
    assert sorted(e.name for e in new.entries) == sorted(by_name)
    # the C++ packs files in its directory-walk order; recover it from the offsets
    packed = sorted([e for e in new.entries if e.size], key=lambda e: e.offset)
    walk = [e.name for e in packed]
    sizes_in_walk = [len(by_name[n]) for n in walk]
    total = sum(sizes_in_walk)
    want_off, want_parts = ao.build_ark(sizes_in_walk, ao.plan_part_sizes(total, len(hdr.parts)))
    assert [e.offset for e in packed] == want_off
    assert [s for _, s in new.parts] == want_parts
    assert all(e.offset == 0 for e in new.entries if e.size == 0)
    image = b"".join(open(tmp_path / "repacked" / p, "rb").read() for p, _ in new.parts)
    assert image == b"".join(by_name[n] for n in walk)
    # header bytes: feed the oracle serialiser the same table (in C++ table order = walk order incl. empties)
    table_order_names = [e.name for e in new.entries]
    ref_entries = {e.name: e for e in new.entries}
    # reconstruct the in-memory table the C++ serialised: directory-walk order (files first, then dirs)
    table = reconstruct_walk(sorted(by_name), by_name)
    tbl = [ao.Entry(name=n, offset=ref_entries[n].offset, size=ref_entries[n].size) for n in table]
    model = ao.Header(ps4=ps4, parts=new.parts, entries=tbl)
    order = None if not ps4 else [table.index(n) for n in table_order_names]
    assert ao.serialise_header(model, order=order) == plain
    # and it round-trips through unpack again
    os.makedirs(tmp_path / "again", exist_ok=True)
    for p, _ in new.parts:
        os.replace(tmp_path / "repacked" / p, tmp_path / "again" / p)
    os.replace(tmp_path / "repacked" / f"main_{plat}.hdr", tmp_path / "again" / f"main_{plat}.hdr")
    run(cli, tmp_path / "again", *pre, "-unpack", "out")
    check_unpacked(tmp_path / "again" / "out", hdr, payloads)


def test_pack_filters_unknown_files_and_songs(cli, tmp_path):
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=50, n_parts=2, seed=13)
    run(cli, tmp_path, "-unpack", "unpacked")
    (tmp_path / "unpacked" / "ps4" / "brand_new.bin").write_bytes(b"new file")
    # like the reference (Modulate.cpp:410-432), -pack without -packall takes its song list from the two DTA
    # configs of the input tree and fails loudly without them (it used to drop every song silently)
    assert "Failed to open file" in run(cli, tmp_path, "-pack", "unpacked", "r0", expect=1)
    cfg, songs_cfg = arkfixture.song_config_blobs()
    (tmp_path / "unpacked" / "ps4" / "config").mkdir(parents=True, exist_ok=True)
    (tmp_path / "unpacked" / "ps4" / "config" / "amp_config.dta_dta_ps4").write_bytes(cfg)
    (tmp_path / "unpacked" / "ps4" / "config" / "amp_songs_config.dta_dta_ps4").write_bytes(songs_cfg)
    run(cli, tmp_path, "-pack", "unpacked", "r1")                       # default: ignore new + /songs/ filter
    new, _ = arkfixture.read_header(str(tmp_path / "r1" / "main_ps4.hdr"))
    names = {e.name for e in new.entries}
    assert "ps4/brand_new.bin" not in names
    # CUSTOM1 is in the configs, so its folder is kept (an unconfigured folder being dropped is pinned by the
    # reference-generated fixtures: tests/test_ref_fixtures.py, /songs/Custom_Two/)
    assert {n for n in names if "/songs/custom1/" in n} == {e.name for e in hdr.entries if "/songs/custom1/" in e.name}
    assert any("/songs/credits/" in n for n in names) or not any("/songs/credits/" in e.name for e in hdr.entries)
    run(cli, tmp_path, "-packall", "-pack_add", "unpacked", "r2")      # everything
    new2, _ = arkfixture.read_header(str(tmp_path / "r2" / "main_ps4.hdr"))
    assert {e.name for e in new2.entries} == {e.name for e in hdr.entries} | {
        "ps4/brand_new.bin", "ps4/config/amp_config.dta_dta_ps4", "ps4/config/amp_songs_config.dta_dta_ps4"}


def test_unpack_duplicate_names_resolve_in_table_order(cli, tmp_path):
    """Two entries with one name: the reference writes in table order with overwriting on (its default,
    CArk.cpp:435-501, Settings.cpp:7), so the LAST entry's bytes stay on disk -- whatever order the
    pipeline's writer threads run in, and without two threads ever writing one path."""
    first, second, other = b"F" * 70000, b"S" * 50000, b"o" * 1000
    entries = [ao.Entry(name="ps4/dup.bin", offset=0, size=len(first)),
               ao.Entry(name="ps4/other.bin", offset=len(first), size=len(other)),
               ao.Entry(name="ps4/dup.bin", offset=len(first) + len(other), size=len(second)),
               ao.Entry(name="ps4/empty_dup.bin", offset=0, size=0),
               ao.Entry(name="ps4/empty_dup.bin", offset=0, size=0)]
    image = first + other + second
    hdr = ao.Header(ps4=True, parts=[("main_ps4_0.ark", len(image))], entries=entries)
    plain = ao.serialise_header(hdr)
    cipher = plain[:4] + oracle.cycle(np.frombuffer(plain[4:], dtype=np.uint8), ao.KEY_PS4).tobytes()
    (tmp_path / "main_ps4.hdr").write_bytes(cipher)
    (tmp_path / "main_ps4_0.ark").write_bytes(image)
    for _ in range(3):  # thread scheduling must not matter
        run(cli, tmp_path, "-unpack", "out")
        assert (tmp_path / "out" / "ps4" / "dup.bin").read_bytes() == second
        assert (tmp_path / "out" / "ps4" / "other.bin").read_bytes() == other
        assert (tmp_path / "out" / "ps4" / "empty_dup.bin").read_bytes() == b""


def test_large_entries_travel_in_pieces(cli, tmp_path, monkeypatch):
    """Entries larger than a pipeline group are cut into pieces (jumped keys) so that a slot never has to hold
    a whole big file: same files out of -unpack, same archive out of -pack_add.  MOD_IO_GROUP_MIB=1 makes a
    few-MiB entry 'large'."""
    import subprocess
    key = 0x2468ACE
    sizes = [3_500_000, 10, 0, 2_200_001, 70_000, 1_572_864, 5] + [30_000] * 20
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=len(sizes), n_parts=2, seed=29, body_key=key, sizes=sizes)
    env = dict(os.environ, MOD_IO_GROUP_MIB="1")

    def run_env(*args):
        out = subprocess.run([cli, *args], cwd=tmp_path, capture_output=True, text=True, timeout=300, env=env)
        assert out.returncode == 0, out.stdout + out.stderr

    run_env("-bodykey", str(key), "-unpack", "out")
    check_unpacked(tmp_path / "out", hdr, payloads)
    run_env("-bodykey", str(key), "-packall", "-pack_add", "out", "re")
    run(cli, tmp_path / "re", "-bodykey", str(key), "-unpack", "again")       # default group size reads it back
    check_unpacked(tmp_path / "re" / "again", hdr, payloads)
    new, _ = arkfixture.read_header(str(tmp_path / "re" / "main_ps4.hdr"))
    image = np.frombuffer(b"".join(open(tmp_path / "re" / p, "rb").read() for p, _ in new.parts), np.uint8)
    by_name = {e.name: p for e, p in zip(hdr.entries, payloads)}
    for e in new.entries:  # every entry, big ones included, is one continuous keystream from its first byte
        assert oracle.cycle(image[e.offset:e.offset + e.size], key).tobytes() == by_name[e.name], e.name


def test_pipelines_deal_groups_to_two_devices(cli, tmp_path):
    """An archive above the facade's 256 MiB multi-GPU threshold is spread over every device, in both
    directions: each slot's group must run on the slot's device with that device's plan and stream (the
    mock, like the real library, refuses a plan or stream of another device)."""
    key = 0x1357BDF
    sizes = [900_000] * 300
    sizes[7] = sizes[150] = 0
    sizes[100] = 60 << 20  # cut into pieces
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=len(sizes), n_parts=3, seed=31, body_key=key, sizes=sizes)
    assert sum(sizes) > 256 << 20
    env = dict(os.environ, MOD_MOCK_DEVICES="2", MOD_TRACE="1")

    def run_env(cwd, *args):
        out = subprocess.run([cli, "-bodykey", str(key), *args], cwd=cwd, capture_output=True, text=True, timeout=300, env=env)
        assert out.returncode == 0, out.stdout + out.stderr
        return out.stderr

    assert "on 2 GPU(s)" in run_env(tmp_path, "-unpack", "out")
    check_unpacked(tmp_path / "out", hdr, payloads)
    assert "on 2 GPU(s)" in run_env(tmp_path, "-packall", "-pack_add", "out", "re")
    assert "on 2 GPU(s)" in run_env(tmp_path / "re", "-unpack", "again")
    check_unpacked(tmp_path / "re" / "again", hdr, payloads)


def test_pack_fails_loudly_on_an_unreadable_file(cli, tmp_path):
    """BuildArk gives up on the first input it cannot open (reference CArk.cpp:799-804)."""
    if os.geteuid() == 0:
        pytest.skip("root can read everything")
    hdr, _, _ = arkfixture.write_archive(str(tmp_path), n_files=20, n_parts=2, seed=23)
    run(cli, tmp_path, "-unpack", "unpacked")
    victim = next(e for e in hdr.entries if e.size)
    os.chmod(tmp_path / "unpacked" / victim.name, 0)
    assert "Failed to open file" in run(cli, tmp_path, "-packall", "-pack", "unpacked", "out", expect=1)


def test_header_codec_roundtrip_python_side():
    """Load's reader parses what lSaveHeader's writer emits (oracle restatement of both)."""
    for ps4 in (True, False):
        names = arkfixture.make_names(200, seed=21)
        entries = [ao.Entry(name=n, offset=i * 100, size=(i % 7) * 10) for i, n in enumerate(names)]
        hdr = ao.Header(ps4=ps4, parts=[("a.ark", 1000), ("b.ark", 2000)], entries=entries)
        back = ao.parse_header(ao.serialise_header(hdr))
        assert back.parts == hdr.parts and back.ps4 == ps4
        assert sorted((e.name, e.offset, e.size) for e in back.entries) == sorted((e.name, e.offset, e.size) for e in entries)
        # every bucket chain reaches every entry of the bucket exactly once
        n = len(back.entries)
        reached = set()
        for b in range(n):
            idx = back.entries[b].flags2 if b < n else -1
            while idx != -1:
                assert idx not in reached
                reached.add(idx)
                assert ao.file_hash(back.entries[idx].name, n) == b
                idx = back.entries[idx].flags1
        assert reached == set(range(n))


def test_header_fuzz_never_crashes(cli, tmp_path):
    """Random corruptions of a valid (deciphered-then-reciphered) header: the loader must answer
    with an eError or succeed, never crash or hang (the reference reads out of bounds here)."""
    hdr, _, plain = arkfixture.write_archive(str(tmp_path), n_files=40, n_parts=2, seed=17)
    path = tmp_path / "main_ps4.hdr"
    rng = np.random.default_rng(99)
    crashes = []
    for trial in range(120):
        bad = bytearray(plain)
        kind = trial % 4
        if kind == 0:      # flip a few random bytes after the magic
            for _ in range(int(rng.integers(1, 6))):
                bad[int(rng.integers(4, len(bad)))] = int(rng.integers(0, 256))
        elif kind == 1:    # overwrite a random aligned word with an extreme value
            pos = int(rng.integers(1, len(bad) // 4)) * 4
            bad[pos:pos + 4] = int(rng.choice([0x7FFFFFFF, 0xFFFFFFFF, 0x80000000, 25001, 101])).to_bytes(4, "little")
        elif kind == 2:    # truncate
            bad = bad[:int(rng.integers(4, len(bad)))]
        else:              # append garbage
            bad += bytes(int(x) for x in rng.integers(0, 256, size=int(rng.integers(1, 64))))
        enc = bytes(bad[:4]) + oracle.cycle(np.frombuffer(bytes(bad[4:]), np.uint8), ao.KEY_PS4).tobytes()
        path.write_bytes(enc)
        out = subprocess.run([cli, "-unpack", f"o{trial}"], cwd=tmp_path, capture_output=True, text=True, timeout=60)
        if out.returncode not in (0, 255):
            crashes.append((trial, kind, out.returncode))
    assert not crashes, crashes


def test_external_caller_compiles_against_facade_headers(cli, tmp_path):
    """A caller that only includes the facade headers (reference class names and signatures)."""
    exe = link("facade_sample", os.path.join(ROOT, "tests", "cpp", "facade_sample.cpp"))
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=25, n_parts=2, seed=41)
    out = subprocess.run([exe, "main_ps4.hdr", "out/"], cwd=tmp_path, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "keystream: 7a cc ad 6f af 91 a7 e3" in out.stdout          # PS4 key KAT (SURVEY.md 8(c))
    assert f"files: {len(hdr.entries)}, has first: 1" in out.stdout
    check_unpacked(tmp_path / "out", hdr, payloads)
