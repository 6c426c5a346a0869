"""Throughput of the masked search and the case-folded sets against the exact kernels.

    python tools/find_masked_timing.py [--reps 10] [--skip-16g]

Kernel-only, device-resident, inputs larger than L2, CUDA events, medians of `reps`, the variants alternated in one
process.  Sets of entries: 1 GiB in 10 000 and 16 GiB in 160 000, byte-packed, per-entry keys, random bytes.
Single pattern (8 bytes): the exact kernel (mod_plan_find), the masked kernel with a fold mask on letters, a wildcard
pattern whose anchor is a >= 1 (two leading ?? bytes), and a weak-anchor pattern whose every byte keeps one nibble.
Sets: K = 16 and 256 random letter patterns of 4 to 32 bytes, exact against folded.  TB/s are payload bytes over
kernel time.  Prints the GPU name and power limit first.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import modulate_b200 as mb  # noqa: E402
import synth  # noqa: E402
from find_set_timing import timed  # noqa: E402
from find_timing import gpu_info  # noqa: E402

SINGLE = {
    "exact": (b"AmpLitUd", None),
    "fold": mb.ignore_case_pattern(b"AmpLitUd"),
    "wild_a2": mb.wildcard_pattern("?? ?? 41 6d 70 4c 69 74"),
    "nibble": mb.wildcard_pattern("4? 6? 7? 4? 6? 7? 5? 6?"),
}


def letter_sets(rng) -> dict:
    out = {}
    for k in (16, 256):
        pats, seen = [], set()
        while len(pats) < k:
            p = bytes(int(x) for x in rng.integers(0x41, 0x5B, size=int(rng.integers(4, 33))))
            p = bytes(b | (0x20 * int(rng.integers(2))) for b in p)
            if p.upper() not in seen:
                seen.add(p.upper())
                pats.append(p)
        out[k] = pats
    return out


def stats(ts, payload):
    t = float(np.median(ts))
    return {"median_s": t, "min_s": float(np.min(ts)), "payload_TBps": payload / t / 1e12}


def time_workload(total: int, n: int, reps: int, sets: dict) -> dict:
    sizes = synth.entry_sizes_loguniform(n, total, seed=7)
    off = synth.packed_offsets(sizes)
    nbytes = int(off[-1] + sizes[-1])
    descs = mb.make_descs(off, off, sizes, synth.entry_keys(n))
    buf = torch.empty(nbytes + 64, dtype=torch.uint8, device="cuda").random_(0, 256)
    plan = mb.Plan(descs, nbytes, nbytes, buf.data_ptr() & 15)
    cap = 1 << 20
    res = torch.zeros(16 + 4 * n + 8 * 256 + 12 * cap, dtype=torch.uint8, device="cuda")
    base = res.data_ptr()
    counts, pcounts, lst = base + 16, base + 16 + 4 * n, base + 16 + 4 * n + 8 * 256
    payload = int(np.sum(sizes, dtype=np.int64))

    fns = {}
    for name, (value, mask) in SINGLE.items():
        fns[name] = (lambda v=value, m=mask: plan.find(buf.data_ptr(), v, counts, lst, cap, base, mask=m))
    psets = {}
    for k, pats in sets.items():
        psets[(k, False)] = mb.PatternSet(pats)
        psets[(k, True)] = mb.PatternSet(pats, ignore_case=True)
        for fold in (False, True):
            s = psets[(k, fold)]
            fns[f"set{k}_{'fold' if fold else 'exact'}"] = (lambda s=s: plan.find_set(buf.data_ptr(), s, counts, pcounts, lst,
                                                                                     cap, base))
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            timed(fn, reps, times[k])
    out = {"payload_bytes": payload, "entries": n, "kernels": {k: stats(ts, payload) for k, ts in times.items()}}
    kt = out["kernels"]
    out["over_exact"] = {k: kt[k]["median_s"] / kt["exact"]["median_s"] for k in SINGLE}
    out["fold_over_exact_set"] = {k: kt[f"set{k}_fold"]["median_s"] / kt[f"set{k}_exact"]["median_s"] for k in sets}
    for s in psets.values():
        s.close()
    plan.close()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--skip-16g", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("find_masked_timing.py needs a GPU")
    mb.init(0)
    print("GPU:", gpu_info(), flush=True)
    sets = letter_sets(np.random.default_rng(14))
    workloads = [("1GiB/10000", 1 << 30, 10000)] + ([] if args.skip_16g else [("16GiB/160000", 16 << 30, 160000)])
    for name, total, n in workloads:
        r = time_workload(total, n, args.reps, sets)
        r["workload"] = name
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
