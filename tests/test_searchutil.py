"""CPU: the numpy search reference of tests/searchutil.py, which every search test compares the CLI and the kernels
against, checked against a plain per-byte loop on small random entries."""
import numpy as np
import pytest

from searchutil import search, search_one

ALPHABET = np.frombuffer(b"aAbBzZ@`[{\x00\x01\x10\x1f\x80\xc1\xe1\xff", np.uint8)


def fold(b):
    return b - 0x20 if ord("a") <= b <= ord("z") else b


def loop_search(entries, patterns, masks, fold_case, owned):
    out = []
    for i, e in enumerate(entries):
        for p in range(len(e)):
            for j, pat in enumerate(patterns):
                if p + len(pat) > len(e) or (owned is not None and p >= owned[i]):
                    continue
                mask = masks[j] if masks is not None else b"\xff" * len(pat)
                key = fold if fold_case else (lambda b: b)
                if all((key(int(e[p + k])) ^ key(pat[k])) & mask[k] == 0 for k in range(len(pat))):
                    out.append((i, p, j))
    return out


def pattern_set(rng):
    """Mixed lengths 1..9, half of them sharing a 2-byte prefix, the rest random."""
    head = bytes(rng.choice(ALPHABET, size=2))
    pats = set()
    while len(pats) < 12:
        pat = bytes(rng.choice(ALPHABET, size=int(rng.integers(1, 10))))
        pats.add(head[:len(pat)] + pat[2:] if len(pats) % 2 else pat)
    return sorted(pats, key=lambda p: rng.random())


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("fold_case", [False, True])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("bounded", [False, True])
def test_search_equals_a_per_byte_loop(seed, fold_case, masked, bounded):
    rng = np.random.default_rng(seed)
    entries = [rng.choice(ALPHABET, size=int(s)).astype(np.uint8) for s in (0, 1, 2, 9, 64, 200, 333)]
    pats = pattern_set(rng)
    for e in entries[3:]:  # plant each pattern at a few starts, some of them at the end
        for pat in pats[:6]:
            at = int(rng.integers(0, e.size - len(pat) + 1))
            e[at:at + len(pat)] = np.frombuffer(pat, np.uint8)
    # wildcard, nibble and fold-mask bytes, never an all-zero mask
    weak = np.array([0xFF, 0xFF, 0x00, 0xF0, 0x0F, 0xDF], np.uint8)
    masks = [bytes(rng.choice(weak, size=len(p))) for p in pats] if masked else None
    if masks is not None:
        masks = [m if any(m) else b"\xff" + m[1:] for m in masks]
    owned = [int(rng.integers(0, len(e) + 2)) for e in entries] if bounded else None
    got, counts, pattern_counts = search(entries, pats, masks, fold_case, owned)
    want = loop_search(entries, pats, masks, fold_case, owned)
    assert got == sorted(want) and len(want) >= 10
    assert counts.dtype == np.uint32 and counts.tolist() == [sum(1 for i, _, _ in want if i == n) for n in range(len(entries))]
    assert pattern_counts.dtype == np.uint64
    assert pattern_counts.tolist() == [sum(1 for _, _, j in want if j == n) for n in range(len(pats))]
    one, one_counts = search_one(entries, pats[0], None if masks is None else masks[0], fold_case)
    first = loop_search(entries, pats[:1], None if masks is None else masks[:1], fold_case, None)
    assert one == [(i, p) for i, p, _ in first]
    assert one_counts.tolist() == [sum(1 for i, _, _ in first if i == n) for n in range(len(entries))]
