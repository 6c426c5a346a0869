"""Throughput of the archive search against the batched cipher kernel and against its read-only bound.

    python tools/find_timing.py [--reps 20] [--skip-16g] [--cli]

Kernel-only, device-resident, inputs larger than L2: the search kernel (mod_plan_find) and the batched
cipher kernel (mod_plan_run, in place) over the same byte-packed set with per-entry keys, alternated in one
process and timed with CUDA events.  Sets: 1 GiB in 10 000 entries and 16 GiB in 160 000 entries.  The
bounds: the search reads each payload byte once (1 HBM byte per byte; the cipher kernel moves 2), and the
keystream needs one modular multiply (IMAD.WIDE) per byte.  With --cli, -find against -unpack of the same
ciphered 1 GiB archive in /dev/shm, wall time of the command.  Prints the GPU name and power limit first.
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
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import modulate_b200 as mb  # noqa: E402
import synth  # noqa: E402


def gpu_info() -> str:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def peak_read_bw() -> float | None:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if not os.path.exists(path):
        return None
    peaks = json.load(open(path))
    for k in ("hbm_read_bw", "read_bw", "hbm_bw", "dram_bw"):
        if k in peaks:
            v = float(peaks[k])
            return v * 1e9 if v < 1e6 else v
    return None


def time_set(total: int, n: int, reps: int) -> dict:
    sizes = synth.entry_sizes_loguniform(n, total, seed=7)
    off = synth.packed_offsets(sizes)
    nbytes = int(off[-1] + sizes[-1])
    descs = mb.make_descs(off, off, sizes, synth.entry_keys(n))
    buf = torch.empty(nbytes + 64, dtype=torch.uint8, device="cuda").random_(0, 256)
    plan = mb.Plan(descs, nbytes, nbytes, buf.data_ptr() & 15)
    cap = 1 << 20
    res = torch.zeros(16 + 4 * n + 8 * cap, dtype=torch.uint8, device="cuda")
    base = res.data_ptr()
    pat = b"\xa5\x3c\x5a\x0f\x96"

    def find():
        plan.find(buf.data_ptr(), pat, base + 16, base + 16 + 4 * n, cap, base)

    def cipher():
        plan.run(buf.data_ptr(), buf.data_ptr())

    payload = int(np.sum(sizes, dtype=np.int64))
    times = {"find": [], "cipher": []}
    for fn in (find, cipher):
        fn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for name, fn in (("find", find), ("cipher", cipher)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / 1e3)
    plan.close()
    out = {"payload_bytes": payload, "entries": n}
    for name, ts in times.items():
        t = float(np.median(ts))
        out[name] = {"median_s": t, "min_s": float(np.min(ts)), "payload_TBps": payload / t / 1e12}
    return out


def cli_timing() -> dict:
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import arkfixture
    cli = os.path.join(ROOT, "modulate_b200", "bin", "modulate")
    root = tempfile.mkdtemp(prefix="findtiming", dir="/dev/shm" if os.access("/dev/shm", os.W_OK) else None)
    try:
        key = 0x5EED1234
        sizes = [int(x) for x in synth.entry_sizes_loguniform(10000, 1 << 30, seed=5)]
        arkfixture.write_archive(root, n_files=len(sizes), n_parts=4, seed=37, body_key=key, sizes=sizes)
        out = {}
        for name, args in (("find", ["-findhex", "5aa50f"]), ("unpack", ["-unpack", "out"])) * 2:
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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--skip-16g", action="store_true")
    ap.add_argument("--cli", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("find_timing.py needs a GPU")
    mb.init(0)
    print("GPU:", gpu_info(), flush=True)
    peak = peak_read_bw()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sets = [("1GiB/10000", 1 << 30, 10000)] + ([] if args.skip_16g else [("16GiB/160000", 16 << 30, 160000)])
    for name, total, n in sets:
        r = time_set(total, n, args.reps)
        r["set"] = name
        if peak:
            r["read_bound_s"] = r["payload_bytes"] / peak  # 1 HBM byte per payload byte
            r["find_share_of_read_bound"] = r["read_bound_s"] / r["find"]["median_s"]
        r["sms"] = sms
        print(json.dumps(r), flush=True)
    if args.cli:
        print(json.dumps({"cli_1GiB_dev_shm": cli_timing()}), flush=True)


if __name__ == "__main__":
    main()
