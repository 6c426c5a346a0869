"""GPU: the C++ facade (CEncryptionCycler / CArk) and the CLI linked against the REAL CUDA library:
the same archive flows as tests/test_facade_host.py, checked against the oracle."""
import os
import subprocess

import numpy as np
import pytest

import oracle
import synth
from oracle import ark_oracle as ao
import arkfixture
from arkfixture import check_unpacked, reconstruct_walk

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "modulate_b200", "bin", "modulate")


def run(cwd, *args, expect=0):
    if not os.path.exists(CLI):
        from modulate_b200 import build as _build
        _build.build()
    assert os.path.exists(CLI), "modulate CLI not built (python -m modulate_b200.build)"
    out = subprocess.run([CLI, *args], cwd=cwd, capture_output=True, text=True, timeout=600)
    assert out.returncode == (0 if expect == 0 else 255), out.stdout + out.stderr
    return out.stdout


def test_cli_links_the_cuda_library():
    out = subprocess.run(["ldd", CLI], capture_output=True, text=True).stdout
    assert "libmodulate_b200.so" in out and "not found" not in out.split("libmodulate_b200.so")[1].split("\n")[0]


@pytest.mark.parametrize("ps4", [True, False])
def test_unpack_on_gpu(tmp_path, ps4):
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), ps4=ps4, n_files=300, n_parts=4, seed=31)
    run(tmp_path, *([] if ps4 else ["-ps3"]), "-unpack", "out")
    check_unpacked(tmp_path / "out", hdr, payloads)


def test_unpack_ciphered_bodies_on_gpu(tmp_path):
    key = -559038737  # 0xDEADBEEF as int
    sizes = [int(x) for x in np.random.default_rng(2).integers(0, 300000, size=120)]
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=120, n_parts=3, seed=33, body_key=key, sizes=sizes)
    run(tmp_path, "-bodykey", str(key), "-unpack", "out")
    check_unpacked(tmp_path / "out", hdr, payloads)


def test_decode_on_gpu(tmp_path):
    _, _, plain = arkfixture.write_archive(str(tmp_path), n_files=500, seed=35)
    run(tmp_path, "-decode")
    assert open(tmp_path / "main_ps4.hdr.dec", "rb").read() == plain


@pytest.mark.parametrize("ps4", [True, False])
def test_repack_on_gpu_end_to_end(tmp_path, ps4):
    """BASELINE config 5 in miniature: extract, patch one DTA-like entry on the host, rebuild offsets
    and parts, re-encipher bodies + header, write; then read it all back."""
    plat = "ps4" if ps4 else "ps3"
    pre = [] if ps4 else ["-ps3"]
    key = 0x0BADF00D
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), ps4=ps4, n_files=150, n_parts=3, seed=37, body_key=key)
    run(tmp_path, *pre, "-bodykey", str(key), "-unpack", "unpacked")
    # the host-side patch: one entry is a binary DTA script; change a value in it with the DTB codec
    from oracle import dta_oracle as do
    from arkfixture import song_config_tree
    victim = next(e for e in hdr.entries if e.size > 100)
    tree = song_config_tree()
    open(tmp_path / "unpacked" / victim.name, "wb").write(do.serialise([tree]))
    run(tmp_path, "-dtaset", os.path.join("unpacked", victim.name), "bpm", "174")
    kids, i = do.find_node(tree, b"bpm")
    kids[i + 1] = ("int", 0, 174)
    patched = do.serialise([tree])
    assert open(tmp_path / "unpacked" / victim.name, "rb").read() == patched
    run(tmp_path, *pre, "-bodykey", str(key), "-packall", "-pack_add", "unpacked", "repacked")
    new, plain = arkfixture.read_header(str(tmp_path / "repacked" / f"main_{plat}.hdr"))
    by_name = {e.name: p for e, p in zip(hdr.entries, payloads)}
    by_name[victim.name] = patched
    packed = sorted([e for e in new.entries if e.size], key=lambda e: e.offset)
    sizes_in_walk = [len(by_name[e.name]) for e in packed]
    want_off, want_parts = ao.build_ark(sizes_in_walk, ao.plan_part_sizes(sum(sizes_in_walk), len(hdr.parts)))
    assert [e.offset for e in packed] == want_off and [s for _, s in new.parts] == want_parts
    image = np.frombuffer(b"".join(open(tmp_path / "repacked" / p, "rb").read() for p, _ in new.parts), np.uint8)
    for e in packed:  # bodies are ciphered per entry with the body key
        assert oracle.cycle(image[e.offset:e.offset + e.size], key).tobytes() == by_name[e.name], e.name
    table = reconstruct_walk(sorted(by_name), by_name)
    ref = {e.name: e for e in new.entries}
    model = ao.Header(ps4=ps4, parts=new.parts, entries=[ao.Entry(name=n, offset=ref[n].offset, size=ref[n].size) for n in table])
    order = None if not ps4 else [table.index(e.name) for e in new.entries]
    assert ao.serialise_header(model, order=order) == plain


def test_config5_repack_through_the_c_binding(mb):
    """BASELINE config 5 through include/modulate_ark.h (what bench.py's extra.cfg5 times at 1 GiB), here
    on a 48 MiB / 700-entry archive: unpack, DTA patch, repack; every byte of the repacked HDR and ARK
    parts is compared with the oracle inside measure_cfg5."""
    import types

    import bench
    r = bench.measure_cfg5(types.SimpleNamespace(mb=mb), total=48 << 20, n_files=700)
    assert r["parity_bytes_checked"] > 48 << 20 and r["value"] > 0
    assert r["entries"] == 700


def test_unpack_large_archive_uses_every_gpu(tmp_path, mb):
    """An archive above the facade's 256 MiB multi-GPU threshold: groups are dealt to slots on every
    visible device (one device here unless the box has more); output must not depend on it."""
    sizes = [int(x) for x in synth.entry_sizes_loguniform(600, 300 << 20, lo=1 << 10, hi=4 << 20, seed=41)]
    key = 0x1234567
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=600, n_parts=2, seed=43, body_key=key, sizes=sizes)
    mb.ark_unpack(str(tmp_path / "main_ps4.hdr"), str(tmp_path), str(tmp_path / "out"), key)
    check_unpacked(tmp_path / "out", hdr, payloads)


def test_large_entries_travel_in_pieces_on_gpu(tmp_path, mb, monkeypatch):
    """Entries larger than a pipeline group are cut into jumped-key pieces in both file pipelines
    (MOD_IO_GROUP_MIB=1 makes a few-MiB entry 'large'); the bytes must not change."""
    monkeypatch.setenv("MOD_IO_GROUP_MIB", "1")
    key = 0x2468ACE
    sizes = [3_500_000, 10, 0, 2_200_001, 70_000, 1_572_864, 5] + [30_000] * 20
    hdr, payloads, _ = arkfixture.write_archive(str(tmp_path), n_files=len(sizes), n_parts=2, seed=29, body_key=key, sizes=sizes)
    mb.ark_unpack(str(tmp_path / "main_ps4.hdr"), str(tmp_path), str(tmp_path / "out"), key)
    check_unpacked(tmp_path / "out", hdr, payloads)
    os.makedirs(tmp_path / "re")
    mb.ark_pack(str(tmp_path / "main_ps4.hdr"), str(tmp_path / "out"), str(tmp_path / "re"), "main_ps4.hdr",
                pack_all=True, ignore_new_files=False, body_key=key)
    monkeypatch.delenv("MOD_IO_GROUP_MIB")
    mb.ark_unpack(str(tmp_path / "re" / "main_ps4.hdr"), str(tmp_path / "re"), str(tmp_path / "again"), key)
    check_unpacked(tmp_path / "again", hdr, payloads)
