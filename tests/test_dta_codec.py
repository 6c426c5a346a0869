"""CPU: the host-side DTB codec (csrc/CDtaFile.cpp) through the CLI built against the mock ABI,
checked against the oracle restatement of the reference's reader/writer (oracle/dta_oracle.py), which
tests/test_ref_fixtures.py in turn checks against DTB files the reference itself loaded and saved."""
import struct

import numpy as np
import pytest

from oracle import dta_oracle as do
from arkfixture import run, song_config_tree  # song_config_tree: shared with bench.py's cfg5 workload
from searchutil import mock_cli


@pytest.fixture(scope="session")
def cli():
    """modulate CLI on the mock ABI, without the search entry points."""
    return mock_cli(0)


def random_tree(rng, depth=0, ttype=16):
    n = int(rng.integers(1, 7))
    children = []
    for _ in range(n):
        kind = rng.integers(0, 10)
        if kind < 3:
            children.append(("int", int(rng.choice(do.INT_TYPES)), int(rng.integers(-2**31, 2**31))))
        elif kind < 4:
            children.append(("float", 1, struct.pack("<f", float(rng.normal()))))
        elif kind < 7:
            ln = int(rng.integers(0, 24))
            s = bytes(int(x) for x in rng.integers(97, 123, size=ln))
            children.append(("str", int(rng.choice(do.STR_TYPES)), s))
        elif depth < 5:
            children.append(random_tree(rng, depth + 1, int(rng.choice(do.TREE_TYPES))))
        else:
            children.append(("int", 0, 7))
    return ("tree", ttype, int(rng.integers(0, 3000)), children)


def test_oracle_roundtrip_and_known_bytes():
    t = ("tree", 16, 1, [("str", 5, b"a"), ("int", 0, 5), ("tree", 17, 2, [("float", 1, struct.pack("<f", 1.5))])])
    blob = do.serialise([t])
    assert blob == (b"\x01\x01\x00\x00\x00" + b"\x03\x00\x01\x00" + b"\x05\x00\x00\x00\x01\x00\x00\x00a" +
                    b"\x00\x00\x00\x00\x05\x00\x00\x00" + b"\x11\x00\x00\x00\x01\x00\x00\x00" + b"\x01\x00\x02\x00" +
                    b"\x01\x00\x00\x00\x00\x00\xc0\x3f")
    assert do.parse(blob) == [t]


@pytest.mark.parametrize("seed", range(5))
def test_cpp_codec_roundtrips_random_trees(cli, tmp_path, seed):
    rng = np.random.default_rng(seed)
    trees = [random_tree(rng)] + ([random_tree(rng, ttype=17)] if seed % 2 else [])
    blob = do.serialise(trees)
    assert do.parse(blob) == trees
    (tmp_path / "in.dtb").write_bytes(blob)
    run(cli, tmp_path, "-dtacopy", "in.dtb", "out.dtb")
    # what the reference's Save writes: identical for one tree, separator-less for several (pinned by
    # tests/golden/dtb/two_trees, tests/test_ref_fixtures.py)
    assert (tmp_path / "out.dtb").read_bytes() == do.save_like_reference(trees)
    if len(trees) == 1:
        assert do.save_like_reference(trees) == blob


def test_cpp_dtaset_patches_like_the_oracle(cli, tmp_path):
    tree = song_config_tree()
    (tmp_path / "cfg.dtb").write_bytes(do.serialise([tree]))
    run(cli, tmp_path, "-dtaset", "cfg.dtb", "bpm", "174", "-dtaset", "cfg.dtb", "name", "Patched Song")
    got = do.parse((tmp_path / "cfg.dtb").read_bytes())
    kids, i = do.find_node(tree, b"bpm")
    kids[i + 1] = ("int", 0, 174)
    kids, i = do.find_node(tree, b"name")
    kids[i + 1] = ("str", 18, b"Patched Song")
    assert got == [tree]
    assert "No value of a matching type" in run(cli, tmp_path, "-dtaset", "cfg.dtb", "missing_key", "1", expect=1)


def test_cpp_rejects_corrupt_dtb(cli, tmp_path):
    good = do.serialise([song_config_tree()])
    cases = {
        "zero_children": good[:5] + b"\x00\x00" + good[7:],
        "bad_type": good[:9] + struct.pack("<i", 99) + good[13:],
        "truncated": good[:len(good) - 3],
        "negative_strlen": good[:13] + struct.pack("<i", -4) + good[17:],
    }
    for name, blob in cases.items():
        with pytest.raises(do.DtaError):
            do.parse(blob)
        (tmp_path / f"{name}.dtb").write_bytes(blob)
        out = run(cli, tmp_path, "-dtacopy", f"{name}.dtb", "o.dtb", expect=1)
        assert "Bad data" in out, name
