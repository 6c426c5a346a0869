"""Synthetic HDR + ARK sets on disk for the facade / CLI tests (built with the oracle)."""
from __future__ import annotations

import json
import os
import subprocess
from typing import List, Optional, Sequence

import numpy as np

import oracle
import synth
from oracle import ark_oracle as ao

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# the reference-generated archive fixtures (tests/golden/make_ark_golden.py): one case per key, and the song list
# the reference derived from the two DTA configs under "songs"
with open(os.path.join(GOLD, "ark", "manifest.json")) as _f:
    MANIFEST = json.load(_f)
CASES = sorted(k for k in MANIFEST if k != "songs")

DIRS = ["ps4/config", "ps4/songs/credits", "ps4/songs/tut0", "ps4/songs/custom1", "ps4/ui", "ps4/ui/textures", "ps4"]
EXTS = ["dta_dta_ps4", "mogg", "png_ps4", "bin", "moggsong"]


def make_names(n: int, seed: int = 1) -> List[str]:
    """n distinct entry names; distinct also when compared case-insensitively (they have to coexist in
    one NTFS directory tree, and the PS4 header order compares with _stricmp)."""
    rng = np.random.default_rng(seed)
    names = {}
    while len(names) < n:
        d = DIRS[int(rng.integers(0, len(DIRS)))]
        stem = "".join(chr(int(c)) for c in rng.integers(97, 123, size=int(rng.integers(3, 10))))
        if rng.random() < 0.2:
            stem = stem.capitalize()
        name = f"{d}/{stem}.{EXTS[int(rng.integers(0, len(EXTS)))]}"
        names.setdefault(name.upper(), name)
    return sorted(names.values())


def cipher_entries(image: np.ndarray, offsets, sizes, key: int) -> None:
    """In place: one Cycle() per entry with `key` -- the unmodified reference cipher over all host
    threads when it is built (oracle/_ref), else the C restatement."""
    import os as _os
    if oracle.have_ref():
        parts = np.zeros(len(sizes), dtype=oracle.PART_DTYPE)
        parts["off"] = np.asarray(offsets, dtype=np.uint64)
        parts["len"] = np.asarray(sizes, dtype=np.uint32)
        parts["key"] = synth.i32(key)
        oracle.ref_cycle_parts(image, parts, _os.cpu_count() or 1)
    else:
        for o, s in zip(offsets, sizes):
            if s:
                image[int(o):int(o) + int(s)] = oracle.cycle(image[int(o):int(o) + int(s)], key)


def reconstruct_walk(names, by_name=None):
    """Directory walk order of the facade's ConstructFromDirectory: per directory, files then
    sub-directories, each in NTFS index order (by upper-cased name)."""
    tree = {}
    for n in names:
        node = tree
        parts = n.split("/")
        for p in parts[:-1]:
            node = node.setdefault(("d", p), {})
        node[("f", parts[-1])] = n
    out = []

    def walk(node):
        files = sorted([k for k in node if k[0] == "f"], key=lambda k: (k[1].upper(), k[1]))
        dirs = sorted([k for k in node if k[0] == "d"], key=lambda k: (k[1].upper(), k[1]))
        for k in files:
            out.append(node[k])
        for k in dirs:
            walk(node[k])
    walk(tree)
    return out


def write_archive(root: str, *, ps4: bool = True, n_files: int = 60, n_parts: int = 3, seed: int = 1,
                  body_key: int = 0, sizes: Optional[Sequence[int]] = None, contents=None):
    """Write main_<plat>.hdr + part files under `root`.  `contents` maps entry index -> bytes for
    entries that must hold something specific (e.g. a DTB).  Returns (Header, plain payload list, plain header)."""
    os.makedirs(root, exist_ok=True)
    plat = "ps4" if ps4 else "ps3"
    rng = np.random.default_rng(seed)
    names = make_names(n_files, seed)
    if sizes is None:
        sizes = [int(x) for x in rng.integers(0, 40000, size=n_files)]
        for i in range(0, n_files, 9):
            sizes[i] = 0  # zero-size entries exist in real headers (offset 0, marker 0)
    offsets = synth.packed_offsets(np.array(sizes, dtype=np.int64))
    total = int(sum(sizes))
    payloads = [synth.payload(int(o) + 1000 * seed, int(s)).tobytes() for o, s in zip(offsets, sizes)]
    if contents:
        for i, blob in contents.items():
            assert len(blob) == sizes[i]
            payloads[i] = blob
    image = np.frombuffer(b"".join(payloads), dtype=np.uint8).copy()
    if body_key and total:
        cipher_entries(image, offsets, sizes, body_key)
    image = image.tobytes()
    # parts: equal shares, the last takes the remainder
    share = total // n_parts
    part_sizes = [share] * (n_parts - 1) + [total - share * (n_parts - 1)]
    parts = [(f"main_{plat}_{i}.ark", s) for i, s in enumerate(part_sizes)]
    entries = [ao.Entry(name=n, offset=(int(o) if s else 0), size=int(s)) for n, o, s in zip(names, offsets, sizes)]
    hdr = ao.Header(ps4=ps4, parts=parts, entries=entries)
    plain = ao.serialise_header(hdr)
    cipher = bytearray(plain)
    cipher[4:] = oracle.cycle(np.frombuffer(plain[4:], dtype=np.uint8), ao.KEY_PS4 if ps4 else ao.KEY_PS3).tobytes()
    with open(os.path.join(root, f"main_{plat}.hdr"), "wb") as f:
        f.write(cipher)
    pos = 0
    for pth, s in parts:
        with open(os.path.join(root, pth), "wb") as f:
            f.write(image[pos:pos + s])
        pos += s
    return hdr, payloads, plain


def read_header(path: str) -> ao.Header:
    raw = open(path, "rb").read()
    magic = int.from_bytes(raw[:4], "little")
    plain = raw[:4] + oracle.cycle(np.frombuffer(raw[4:], dtype=np.uint8), ao.platform_key(magic)).tobytes()
    return ao.parse_header(plain), plain


# ---- the two DTA configs `-pack` reads its song list from (reference Modulate.cpp:410-432) -----------------

SONGS = [
    {"id": "CUSTOM1", "name": "Custom One", "path": "../songs/Custom1/custom1.moggsong", "arena": "World1",
     "type": "kSongNormal", "unlock_method": "play_num", "unlock_count": 3},
    {"id": "CREDITS", "name": "Credits", "path": "songs/credits/credits.moggsong", "arena": "World2",
     "type": "kSongBoss", "unlock_method": "", "unlock_count": -1},
    {"id": "NOT_IN_SONGS_CONFIG", "name": "Orphan", "path": "", "arena": "", "type": "",
     "unlock_method": "beat_num", "unlock_count": 7},
]


def song_config_blobs():
    """(amp_config, amp_songs_config) DTB blobs shaped the way CDtaFile::GetSongs / GetSongData walk them
    (CDtaFile.cpp:102-181, :248-294): six-field song records beside "unlock_tokens" (ids without lower-case
    letters are songs), four-field unlock records beside "campaign", {id, path, (type T)} records inside
    arena groups."""
    from oracle import dta_oracle as do

    def sym(text, t=5):
        return ("str", t, text.encode())

    records = [sym("unlock_tokens")]
    for i, sg in enumerate(SONGS):
        records.append(("tree", 16, 10 + i, [sym(sg["id"]), sym(sg["name"]), sym("unlock_extra"), sym("unlock_extra_desc"),
                                             sym("ui/textures/black_square.png"), sym("CAMPVO_song_extra")]))
    records.append(("tree", 16, 30, [sym("freq_arena"), sym("an arena, not a song"), sym("a"), sym("b"), sym("c"), sym("d")]))
    records.append(("tree", 16, 31, [sym("SHORT"), sym("five fields only"), sym("a"), sym("b"), sym("c")]))
    unlocks = [sym("campaign")]
    for i, sg in enumerate(SONGS):
        if sg["unlock_method"]:
            unlocks.append(("tree", 16, 60 + i, [sym(sg["unlock_method"]), ("int", 0, sg["unlock_count"]),
                                                 sym("kUnlockArena"), sym(sg["id"])]))
    amp_config = ("tree", 16, 1, [("tree", 16, 2, records), ("tree", 16, 50, unlocks), ("int", 6, 12345)])

    arenas = {}
    for sg in SONGS:
        if sg["path"]:
            arenas.setdefault(sg["arena"], []).append(sg)
    groups = []
    for gi, (arena, members) in enumerate(sorted(arenas.items())):
        kids = [sym(arena)]
        for mi, sg in enumerate(members):
            kids.append(("tree", 16, 100 + 10 * gi + mi, [sym(sg["id"]), sym(sg["path"], 33),
                                                         ("tree", 16, 200 + 10 * gi + mi, [sym("type"), sym(sg["type"])])]))
        groups.append(("tree", 16, 90 + gi, kids))
    amp_songs_config = ("tree", 16, 1, groups)
    return do.serialise([amp_config]), do.serialise([amp_songs_config])


def fixture_file_bytes(f) -> bytes:
    """Contents of one input file of the reference-generated fixtures (tests/golden/ark/manifest.json): the
    two DTA configs are real DTB (song_config_blobs), everything else is synth.payload(seed, size)."""
    if f.get("content") == "amp_config":
        return song_config_blobs()[0]
    if f.get("content") == "amp_songs_config":
        return song_config_blobs()[1]
    return synth.payload(f["seed"], f["size"]).tobytes()


def song_config_tree():
    """A small amp_config-like DTA script: (key value) pairs inside nested trees (dta_oracle tuple form)."""
    import struct

    def sym(s):
        return ("str", 5, s.encode())
    song = ("tree", 16, 12, [sym("song"), ("tree", 16, 13, [sym("name"), ("str", 18, b"Perfect Brain")]),
                             ("tree", 16, 14, [sym("bpm"), ("int", 0, 120)]),
                             ("tree", 16, 15, [sym("preview_start_ms"), ("int", 6, 30000)]),
                             ("tree", 17, 16, [sym("boss_level"), ("int", 0, -1), ("float", 1, struct.pack("<f", 0.5))])])
    return ("tree", 16, 1, [sym("songs"), song, ("tree", 16, 20, [sym("unlock_tokens"), ("int", 0, 3)])])


def ref_header(case: str) -> bytes:
    """The header bytes the reference's SaveArk wrote for fixture `case`."""
    plat = MANIFEST[case]["platform"]
    with open(os.path.join(GOLD, "ark", case, f"main_{plat}.hdr"), "rb") as f:
        return f.read()


# ---- running the CLI -----------------------------------------------------------------------------------------

def run(cli, cwd, *args, expect=0):
    """stdout of the CLI `cli` run in `cwd`; exit code 0, or the CLI's error exit when `expect` is not 0."""
    out = subprocess.run([cli, *args], cwd=cwd, capture_output=True, text=True, timeout=300)
    assert out.returncode == (expect if expect == 0 else 255), out.stdout + out.stderr
    return out.stdout


def check_unpacked(out_dir, hdr, payloads):
    for e, p in zip(hdr.entries, payloads):
        got = open(os.path.join(out_dir, e.name), "rb").read()
        assert got == p, e.name
