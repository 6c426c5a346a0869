"""Throughput of the pattern-set search against single-pattern passes.

    python tools/find_set_timing.py [--reps 10] [--skip-16g] [--cli]

Kernel-only, device-resident, inputs larger than L2, CUDA events, medians of `reps`, the kernels alternated in one
process.  Sets of entries: 1 GiB in 10 000 and 16 GiB in 160 000, byte-packed, per-entry keys.  Pattern sets: K = 1,
16 and 256 random patterns of 4 to 32 bytes, and 64 patterns sharing their first 8 bytes.  Each set is timed as one
mod_plan_find_set pass, against one mod_plan_find pass (its first pattern) and against K sequential mod_plan_find
passes.  TB/s are payload bytes over kernel time.  With --cli, -findhexlist with 256 patterns against -find and
-unpack of the same ciphered 1 GiB archive in /dev/shm, wall time of the command.  Prints the GPU name and power
limit first.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import modulate_b200 as mb  # noqa: E402
import synth  # noqa: E402
from find_timing import gpu_info  # noqa: E402


def pattern_sets(rng) -> dict:
    def rand(k):
        out = []
        while len(out) < k:
            p = bytes(int(x) for x in rng.integers(0, 256, size=int(rng.integers(4, 33))))
            if p not in out:
                out.append(p)
        return out
    head = bytes(int(x) for x in rng.integers(0, 256, size=8))
    prefix = []
    while len(prefix) < 64:
        p = head + bytes(int(x) for x in rng.integers(0, 256, size=int(rng.integers(1, 25))))
        if p not in prefix:
            prefix.append(p)
    return {"random1": rand(1), "random16": rand(16), "random256": rand(256), "prefix64": prefix}


def timed(fn, reps, sink) -> None:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    sink.append(a.elapsed_time(b) / 1e3)


def time_set(total: int, n: int, reps: int, sets: dict) -> dict:
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
    out = {"payload_bytes": payload, "entries": n, "sets": {}}
    for name, pats in sets.items():
        pset = mb.PatternSet(pats)

        def one():
            plan.find(buf.data_ptr(), pats[0], counts, lst, cap, base)

        def seq():
            for p in pats:
                plan.find(buf.data_ptr(), p, counts, lst, cap, base)

        def setpass():
            plan.find_set(buf.data_ptr(), pset, counts, pcounts, lst, cap, base)

        fns = {"set": setpass, "single": one, "sequential": seq}
        for fn in fns.values():
            fn()
        torch.cuda.synchronize()
        times = {k: [] for k in fns}
        for _ in range(reps):
            for k, fn in fns.items():
                timed(fn, reps, times[k])
        r = {"K": len(pats)}
        for k, ts in times.items():
            t = float(np.median(ts))
            r[k] = {"median_s": t, "min_s": float(np.min(ts)), "payload_TBps": payload / t / 1e12}
        r["set_over_single"] = r["set"]["median_s"] / r["single"]["median_s"]
        r["set_over_sequential"] = r["set"]["median_s"] / r["sequential"]["median_s"]
        out["sets"][name] = r
        pset.close()
    plan.close()
    return out


def cli_timing(pats) -> dict:
    import arkfixture
    cli = os.path.join(ROOT, "modulate_b200", "bin", "modulate")
    root = tempfile.mkdtemp(prefix="findsettiming", dir="/dev/shm" if os.access("/dev/shm", os.W_OK) else None)
    try:
        key = 0x5EED1234
        sizes = [int(x) for x in synth.entry_sizes_loguniform(10000, 1 << 30, seed=5)]
        arkfixture.write_archive(root, n_files=len(sizes), n_parts=4, seed=37, body_key=key, sizes=sizes)
        with open(os.path.join(root, "list.txt"), "w") as f:
            f.write("\n".join(p.hex() for p in pats) + "\n")
        out = {}
        runs = (("findhexlist256", ["-findhexlist", "list.txt"]), ("find", ["-findhex", pats[0].hex()]), ("unpack", ["-unpack", "out"]))
        for name, args in runs * 2:
            shutil.rmtree(os.path.join(root, "out"), ignore_errors=True)
            t0 = time.perf_counter()
            r = subprocess.run([cli, "-bodykey", str(key), *args], cwd=root, capture_output=True)
            dt = time.perf_counter() - t0
            assert r.returncode == 0, r.stdout[-2000:]
            out.setdefault(name, []).append(dt)
        return {k: {"wall_s": v} for k, v in out.items()}
    finally:
        shutil.rmtree(root, ignore_errors=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--skip-16g", action="store_true")
    ap.add_argument("--cli", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("find_set_timing.py needs a GPU")
    mb.init(0)
    print("GPU:", gpu_info(), flush=True)
    sets = pattern_sets(np.random.default_rng(256))
    workloads = [("1GiB/10000", 1 << 30, 10000)] + ([] if args.skip_16g else [("16GiB/160000", 16 << 30, 160000)])
    for name, total, n in workloads:
        r = time_set(total, n, args.reps, sets)
        r["workload"] = name
        print(json.dumps(r), flush=True)
    if args.cli:
        print(json.dumps({"cli_1GiB_dev_shm": cli_timing(sets["random256"])}), flush=True)


if __name__ == "__main__":
    main()
