#!/usr/bin/env python
"""bench.py -- ARK/DTB decrypt throughput on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg4]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (config.workload = "cfg3", BASELINE.json configs[2], the north_star target): a
16 GiB multi-part ARK set = 32 parts x 512 MiB (kuMaxArkSize, reference CArk.cpp:19), one
(offset, len, key) per part, ciphered in place.  One STEP = one pass of the hot path over the set:
    1. CEncryptionCycler::Cycle over the 384 KiB HDR past its 4-byte magic (CArk::Load, CArk.cpp:338-339;
       rank 0 only -- there is one header);
    2. one launch of the variable-length batched kernel over this rank's share of the set.
The two are independent (different buffers, different keys) and are issued on two CUDA streams that are
joined inside the timed region.
STRONG scaling: the set is fixed; at N GPUs it is cut into N equal-payload offset ranges by
mod_shard_descs (cuts fall inside parts: the tail piece starts from the jumped key), one process per
GPU, no collective on the data path.  `value` times the steps with the set resident in HBM; `e2e`
times the same work through the public C ABI on pinned HOST buffers, H2D and D2H copies included.

Parity is checked IN THIS RUN, at every N, on every rank, before the timed region: >= 64 MiB of
windows of the rank's own shard (both sides of every interior cut and part boundary, plus random
windows) are byte-compared with the CPU oracle -- the unmodified reference cipher (oracle/_ref) for
windows that start a part, its closed-form restatement (pinned against it) for windows deep inside
one.  `parity_bytes_checked` is the sum over ranks; any mismatch ends the run with rc != 0.

--dump-outputs DIR writes, after the K timed steps of the headline workload, what they left in the output
buffers (dump_outputs()).  Inputs are seeded, so two builds run with the same arguments can be compared file
by file.

At N == 1 the line also carries `extra.cfg2` (1 GiB / 10 000 entries, misaligned gather; BASELINE
configs[1]) and `extra.cfg4` (1 000 000 entries of 1..64 KiB, one launch; configs[3]), each with its
own roofline (burst from a short timed region + a 1.5 s sustained run), clocks and parity count,
`extra.cfg5` (configs[4]: unpack -> DTA patch -> repack of a 1 GiB archive through the CArk facade on a
RAM-backed file system, every output byte checked), `roofline.sustained` (>= 3 s of back-to-back
launches with NVML clock / power samples) next to the burst figure, and `cpu_baseline` (the unmodified reference cipher on the
host cores, bounded sample).  The CPU numbers are a baseline, not the target -- the target is
roofline.frac.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree (which may be read-only)

import synth  # noqa: E402  (synthetic inputs shared with the tests)

GIB = 1 << 30
MIB = 1 << 20
HDR_BYTES = 384 * 1024  # a real main_ps4.hdr is 0.3-0.5 MB (SURVEY.md section 3)
PART = 512 * MIB        # kuMaxArkSize, reference CArk.cpp:19
N_PARTS = 32
CPU_SAMPLE_PER_PART = 32 * MIB
PARITY_TARGET = 64 * MIB
METRIC = "ark_dtb_decrypt_throughput"


# ---- workload construction --------------------------------------------------------------------

def cfg2_entries():
    """Entry table of the 1 GiB archive: (src_off, size, key)."""
    sizes = synth.entry_sizes_loguniform(10_000, GIB, lo=1 << 10, hi=1 << 20, seed=7)
    return synth.packed_offsets(sizes), sizes, synth.entry_keys(len(sizes), seed=synth.SEED)


def cfg4_entries(n: int = 1_000_000):
    """BASELINE configs[3]: n byte-packed entries of 1..64 KiB with per-entry keys (~32.5 GiB at 1M)."""
    rng = np.random.default_rng(40)
    sizes = rng.integers(1 << 10, (64 << 10) + 1, size=n).astype(np.int64)
    return synth.packed_offsets(sizes), sizes, synth.entry_keys(n, seed=synth.SEED + 99)


def aligned_slots(sizes: np.ndarray) -> np.ndarray:
    """Each extracted file gets its own 16-byte-aligned slot (separately allocated outputs)."""
    return synth.packed_offsets((sizes + 15) & ~np.int64(15))


def global_descs(mb, workload: str, cfg4_n: int = 1_000_000) -> np.ndarray:
    if workload == "cfg3":
        off = np.arange(N_PARTS, dtype=np.int64) * PART
        return mb.make_descs(off, off, np.full(N_PARTS, PART, np.int64), synth.entry_keys(N_PARTS, seed=synth.SEED + 3))
    if workload == "cfg2":
        off, size, key = cfg2_entries()
        return mb.make_descs(off, aligned_slots(size), size, key)
    off, size, key = cfg4_entries(cfg4_n)
    return mb.make_descs(off, off, size, key)  # in place, like config 3


def config_block(workload: str, descs: np.ndarray, world: int) -> dict:
    """Identical in both arms (ours / reference) so the driver sees the same config."""
    layout = {
        "cfg3": "16 GiB = 32 parts x 512 MiB (kuMaxArkSize), one (offset, len, key) per part, ciphered in place; "
                "HDR Cycle + one batched launch per step",
        "cfg2": "1 GiB image, 10 000 byte-packed entries (log-uniform 1 KiB..1 MiB), per-entry keys, gathered into "
                "16-byte-aligned extract slots; HDR Cycle + one batched launch per step",
        "cfg4": "byte-packed entries of 1..64 KiB, per-entry keys, ciphered in place; HDR Cycle + one batched launch per step",
    }[workload]
    return {"workload": workload, "entries": int(len(descs)), "payload_bytes": int(descs["len"].sum()),
            "hdr_bytes": HDR_BYTES, "layout": layout,
            "l2": "every step reads and writes far more than the 126 MB L2 (>= 2 GiB per GPU); no flush needed",
            "sharding": "mod_shard_descs equal-payload offset ranges over n_gpus, no collective (strong scaling)"}


def rebase(descs: np.ndarray):
    """Shift a shard's descriptors so its source / destination windows start at 0."""
    if len(descs) == 0:
        return descs.copy(), 0, 0, 0, 0
    s0 = int(descs["src_off"].min()) & ~15
    d0 = int(descs["dst_off"].min()) & ~15
    out = descs.copy()
    out["src_off"] -= s0
    out["dst_off"] -= d0
    src_bytes = int((out["src_off"] + out["len"]).max())
    dst_bytes = int((out["dst_off"] + out["len"]).max())
    return out, s0, d0, src_bytes, dst_bytes


# ---- synthetic payload on the device ---------------------------------------------------------------

def _i64(c: int) -> int:
    c &= (1 << 64) - 1
    return c - (1 << 64) if c >> 63 else c


def device_payload(torch, out, offset: int, seed: int = synth.SEED, slice_bytes: int = 256 * MIB) -> None:
    """Fill the uint8 tensor `out` with synth.payload(offset, len(out)) -- the same counter-based
    splitmix64 stream, generated where the tensor lives (two's-complement int64 arithmetic wraps like
    uint64; logical shifts are arithmetic shifts with the sign bits masked off)."""
    n = out.numel()

    def lsr(z, k):
        return (z >> k) & ((1 << (64 - k)) - 1)

    pos = 0
    while pos < n:
        m = min(slice_bytes, n - pos)
        w0 = (offset + pos) // 8
        w1 = (offset + pos + m + 7) // 8
        x = torch.arange(w0, w1, dtype=torch.int64, device=out.device)
        x = (x ^ _i64(seed)) + _i64(0x9E3779B97F4A7C15)
        z = (x ^ lsr(x, 30)) * _i64(0xBF58476D1CE4E5B9)
        z = (z ^ lsr(z, 27)) * _i64(0x94D049BB133111EB)
        z = z ^ lsr(z, 31)
        b = z.view(torch.uint8)
        lo = (offset + pos) - w0 * 8
        out[pos:pos + m].copy_(b[lo:lo + m])
        pos += m
        del x, z, b


# ---- clocks -------------------------------------------------------------------------------------

class ClockSampler:
    """Samples SM clock, power and throttle reasons of one GPU through NVML while a region runs."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period_s: float = 0.002):
        self.samples, self.power, self.reason_counts = [], [], {}
        self.max_mhz = None
        self.period = period_s
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _sample(self):
        nv = self.nv
        try:
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(
                nv, "nvmlDeviceGetCurrentClocksEventReasons") else int(
                nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            for bit, name in self.REASONS.items():
                if mask & bit and name != "gpu_idle":
                    self.reason_counts[name] = self.reason_counts.get(name, 0) + 1
            self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            self._sample()
            time.sleep(self.period)

    def start(self):
        if self.nv is not None:
            self._sample()
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)
        if self.nv is not None:
            self._sample()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reason_counts),
                "reason_samples": dict(self.reason_counts), "samples": len(self.samples),
                "sm_mhz_min": min(self.samples) if self.samples else None,
                "power_w_max": max(self.power) if self.power else None,
                "power_w_mean": float(np.mean(self.power)) if self.power else None}


# ---- CPU arm: the unmodified reference cipher on the host cores ------------------------------------

def cpu_sample(descs: np.ndarray, workload: str):
    """Bounded sample of the workload for the CPU arm: one reference Cycle() per entry / part prefix,
    fanned out over all host threads (the reference has no jump-ahead, so a part can only be sampled
    from its start).  cfg3: the first 32 MiB of each of the 32 parts (1 GiB).  cfg2: every entry (1 GiB).
    cfg4: the first 32 768 entries (~1 GiB)."""
    import oracle
    d = descs
    if workload == "cfg3":
        d = descs.copy()
        d["len"] = np.minimum(d["len"], CPU_SAMPLE_PER_PART)
        what = f"the first {CPU_SAMPLE_PER_PART >> 20} MiB of each of the {len(d)} parts"
    elif workload == "cfg4":
        d = descs[:32768]
        what = f"the first {len(d)} entries"
    else:
        what = f"all {len(d)} entries"
    parts = np.zeros(len(d), dtype=oracle.PART_DTYPE)
    parts["off"] = synth.packed_offsets(d["len"].astype(np.int64))  # sample bytes packed back to back
    parts["len"] = d["len"]
    parts["key"] = d["key"]
    nbytes = int(d["len"].sum())
    return {"descs": d, "parts": parts, "bytes": nbytes,
            "sample": f"{what} of the {workload} set ({nbytes} payload bytes) per step, one reference Cycle() each"}


def cpu_fill_plain(sample, buf: np.ndarray) -> None:
    """The sample's plaintext: synth.payload at each entry's SOURCE offset in the full set."""
    for p, d in zip(sample["parts"], sample["descs"]):
        o, n = int(p["off"]), int(p["len"])
        buf[o:o + n] = synth.payload(int(d["src_off"]), n)


def cpu_step(sample, work: np.ndarray, cores: int, kind: str) -> float:
    import oracle
    t0 = time.perf_counter()
    if kind == "reference":
        oracle.ref_cycle_parts(work, sample["parts"], cores)
    else:  # oracle port, single-threaded C restatement
        for p in sample["parts"]:
            oracle.lib().oracle_cycle(work.ctypes.data + int(p["off"]), int(p["len"]), int(p["key"]))
    return time.perf_counter() - t0


def run_reference_arm(args) -> None:
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import modulate_b200 as mb  # host-only use: make_descs (no GPU work on this arm)
    import oracle
    kind = "reference" if oracle.have_ref() else "port"
    if args.workload == "cfg5":  # the repack set is the cfg2 archive: the CPU arm ciphers its entries
        args.workload = "cfg2"
    descs = global_descs(mb, args.workload)
    sample = cpu_sample(descs, args.workload)
    cores = min(os.cpu_count() or 1, len(sample["parts"]))  # one reference Cycle() per part: at most that many threads
    work = np.empty(sample["bytes"], dtype=np.uint8)
    cpu_fill_plain(sample, work)
    for _ in range(args.warmup):
        cpu_step(sample, work, cores, kind)
    t = 0.0
    for _ in range(args.steps):
        t += cpu_step(sample, work, cores, kind)  # the cipher is an involution: no refill needed
    gbs = sample["bytes"] * args.steps / t / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_block(args.workload, descs, args.gpus),
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": cores if kind == "reference" else 1, "kind": kind,
                         "sample": sample["sample"]},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- GPU arm -----------------------------------------------------------------------------------------

def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs: torch copy_ of 2 GiB, best of 10)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class Ctx:
    """Per-process state shared by the measurement helpers."""

    def __init__(self):
        import torch
        import modulate_b200 as mb
        self.torch, self.mb = torch, mb
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        torch.cuda.set_device(self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        # NUMA placement: run this rank (and first-touch its pinned buffers) on the CPUs closest to its GPU
        self.all_cpus = os.sched_getaffinity(0)
        self.numa_pinned = False
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(self.local))
            self.numa_pinned = os.sched_getaffinity(0) != self.all_cpus
        except Exception:
            pass
        mb.init(self.local)
        self.dev = torch.device("cuda", self.local)
        self.stream = torch.cuda.current_stream()
        self.sh = self.stream.cuda_stream
        # the HDR Cycle of a step is independent of the body launch (different buffer, different key): it runs on
        # a second stream so the batched launches queue back to back; timed_steps() joins the two streams inside
        # the timed region
        self.side = torch.cuda.Stream(device=self.dev)
        self.side_h = self.side.cuda_stream
        self.peak, self.peak_src = load_peaks()

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, value: float, op: str) -> float:
        if self.dist is None:
            return float(value)
        t = self.torch.tensor([value], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def finish(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def parity_windows(descs: np.ndarray, target: int, rng) -> list:
    """(entry index, position in entry, length) windows of a shard: both ends of every piece (= both
    sides of every interior cut and part boundary, the neighbour rank checks the other side), then
    random windows until `target` bytes."""
    wins, total = [], 0
    edge = 256 << 10
    for i, d in enumerate(descs):
        n = int(d["len"])
        if n == 0:
            continue
        if n <= 2 * edge:
            wins.append((i, 0, n))
            total += n
        else:
            wins.append((i, 0, edge))
            wins.append((i, n - edge, edge))
            total += 2 * edge
        if total >= target and len(descs) > 4096:  # many-entry sets: a sample of entries is enough
            break
    big = [i for i, d in enumerate(descs) if int(d["len"]) > 4 * MIB]
    while total < target and big:
        i = big[int(rng.integers(0, len(big)))]
        n = int(descs[i]["len"])
        w = min(4 * MIB, n)
        wins.append((i, int(rng.integers(0, n - w + 1)), w))
        total += w
    return wins


def check_parity(c: Ctx, shard_global: np.ndarray, shard_local: np.ndarray, d_out, label: str) -> int:
    """Byte-compare windows of this rank's OUTPUT (after one ciphering pass) with the CPU oracle.
    shard_global carries offsets / jumped keys in the full set (what the plaintext generator and the
    oracle need), shard_local the same pieces rebased to this rank's buffers."""
    import oracle
    rng = np.random.default_rng(1234 + c.rank)
    have_ref = oracle.have_ref()
    checked = 0
    for i, pos, n in parity_windows(shard_local, PARITY_TARGET, rng):
        g, l = shard_global[i], shard_local[i]
        plain = synth.payload(int(g["src_off"]) + pos, n)
        key = int(g["key"])
        want = oracle.cycle_at(plain, key, pos)
        if pos == 0 and have_ref and n <= 8 * MIB:  # stream start: the unmodified reference itself
            if not np.array_equal(oracle.cycle(plain, key, use_ref=True), want):
                raise SystemExit(f"ORACLE DISAGREES WITH THE REFERENCE ({label}, piece {i})")
        o = int(l["dst_off"]) + pos
        got = d_out[o:o + n].cpu().numpy()
        if not np.array_equal(got, want):
            bad = int(np.flatnonzero(got != want)[0])
            raise SystemExit(f"PARITY FAILURE ({label}): rank {c.rank} piece {i} (set offset {int(g['dst_off']) + pos + bad}) "
                             f"differs from the reference cipher")
        checked += n
    return checked


def timed_steps(c: Ctx, step, kernel, steps: int, warmup: int):
    """K steps between two events on the launching stream; `kernel` (the batched launch) is also
    bracketed per step.  Returns (max-over-ranks ms for K steps, mean kernel ms on this rank, clocks, launches)."""
    torch, mb = c.torch, c.mb
    for _ in range(max(warmup, 3)):
        step(None)
    c.barrier()
    clocks = ClockSampler(c.local)
    launches0 = mb.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    c.barrier()
    clocks.start()
    ev0.record(c.stream)
    c.side.wait_event(ev0)       # nothing of the timed steps starts before ev0 ...
    for i in range(steps):
        step(kev[i])
    c.stream.wait_stream(c.side)  # ... and ev1 waits for everything they launched, on both streams
    ev1.record(c.stream)
    torch.cuda.synchronize()
    info = clocks.stop()
    launches = mb.launch_count() - launches0
    ms_total = c.reduce(ev0.elapsed_time(ev1), "max")
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    return ms_total, kernel_ms, info, launches


DUMP_WINDOWS = 1024       # over all ranks
DUMP_WINDOW_BYTES = 4096  # 4 MiB of payload in all: 16 MiB as float32


def dump_windows(descs: np.ndarray, world: int):
    """(entry index, position in entry, length) arrays of the seeded windows dump_outputs() samples."""
    rng = np.random.default_rng(2718)
    idx = rng.integers(0, len(descs), size=max(1, DUMP_WINDOWS // world))
    lens = descs["len"][idx].astype(np.int64)
    width = np.minimum(lens, DUMP_WINDOW_BYTES)
    return idx, rng.integers(0, lens - width + 1), width


def dump_outputs(c: Ctx, out_dir: str, descs: np.ndarray, d_dst, d_hdr) -> None:
    """Write what the last timed step left in this rank's output buffers, as float32 byte values:
    `hdr.npy`, the whole HDR (rank 0), and `payload.npy`, a fixed sample of the payload -- the dump_windows()
    of the entries, concatenated (bytes between extract slots are never written and stay out of it).  With
    N > 1 ranks each rank writes `payload_rank<r>.npy` of its shard.  In-place workloads hold ciphertext or
    plaintext depending on whether the passes so far (parity check, restore, warm-up, timed steps) are odd or
    even in number: the cipher is an involution."""
    torch = c.torch
    idx, pos, width = dump_windows(descs, c.world)
    start = descs["dst_off"][idx].astype(np.int64) + pos
    at = np.concatenate([np.arange(s, s + n) for s, n in zip(start, width)])
    os.makedirs(out_dir, exist_ok=True)
    sample = d_dst[torch.from_numpy(at).to(c.dev)].cpu().numpy().astype(np.float32)
    np.save(os.path.join(out_dir, f"payload_rank{c.rank}.npy" if c.world > 1 else "payload.npy"), sample)
    if d_hdr is not None:
        np.save(os.path.join(out_dir, "hdr.npy"), d_hdr.cpu().numpy().astype(np.float32))


def sustained(c: Ctx, kernel, payload: int, kernel_ms: float, seconds: float = 3.0) -> dict:
    """>= `seconds` of back-to-back launches of the dominant kernel, with NVML samples."""
    torch = c.torch
    # back-to-back launches overlap each other's ramp-up and tail, so one costs a little LESS than the isolated
    # launch kernel_ms was measured on: 10 % more of them than seconds / kernel_ms keeps the run above `seconds`
    iters = max(10, int(1.1 * seconds * 1e3 / max(kernel_ms, 1e-3)) + 1)
    clocks = ClockSampler(c.local, period_s=0.02)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    clocks.start()
    a.record(c.stream)
    for _ in range(iters):
        kernel()
    b.record(c.stream)
    torch.cuda.synchronize()
    info = clocks.stop()
    ms = a.elapsed_time(b) / iters
    achieved = 2.0 * payload / (ms * 1e-3) / 1e9
    return {"seconds": a.elapsed_time(b) / 1e3, "launches": iters, "kernel_ms": ms, "achieved": achieved,
            "frac": achieved / c.peak, "payload_gbs": payload / (ms * 1e-3) / 1e9, "clocks": info}


def roofline_block(c: Ctx, payload: int, kernel_ms: float, workload: str, clock_info: dict) -> dict:
    achieved = 2.0 * payload / (kernel_ms * 1e-3) / 1e9
    r = {"bound": "hbm", "achieved": achieved, "peak": c.peak, "unit": "GB/s", "frac": achieved / c.peak,
         "traffic": None, "kernel": "modk::cycle_batch_kernel", "kernel_ms": kernel_ms,
         "algorithmic_bytes_per_launch": 2 * payload, "peak_source": c.peak_src,
         "payload_gbs": payload / (kernel_ms * 1e-3) / 1e9,
         "frac_of_nominal_8tbs": achieved / 8000.0}
    try:  # the co-limiting integer roofline: one IMAD.WIDE per payload byte at the measured issue rate
        with open(os.path.join(ROOT, "profiles", "imad.json")) as f:
            lanes = float(json.load(f)["imad_wide_thread_instr_per_clk_per_sm"])
        sm_count = c.torch.cuda.get_device_properties(c.dev).multi_processor_count
        mhz = clock_info.get("sm_mhz") or clock_info.get("sm_max_mhz") or 1965.0
        imad_peak = sm_count * lanes * mhz * 1e6 / 1e9
        r["imad"] = {"peak_payload_gbs": imad_peak, "frac": r["payload_gbs"] / imad_peak,
                     "imad_wide_per_clk_per_sm": lanes, "note": "HBM is the binding roofline"}
    except Exception:
        pass
    if c.world == 1:  # the committed ncu captures are of the single-GPU launch (profiles/traffic.json)
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                r["traffic"] = json.load(f).get(workload)
        except Exception:
            pass
    return r


def piece_count(descs: np.ndarray, group: int = 16 * MIB) -> int:
    """Descriptors after the host batch path has cut entries larger than a group (mod_abi.cu batch_host)."""
    n = descs["len"].astype(np.int64)
    return int(np.where(n > group + group // 2, np.maximum(1, n // group), 1).sum())


def measure_workload(c: Ctx, args, workload: str, *, full: bool, cfg4_n: int = 1_000_000, sustain_s: float = 3.0,
                     cooldown_s: float = 0.0, dump_dir: str | None = None) -> dict:
    """Device-resident value, per-launch roofline, parity, the sustained run (`sustain_s` seconds of back-to-back
    launches; 0 = skip) and, if `full`, e2e for one workload.  `dump_dir`: see dump_outputs()."""
    torch, mb = c.torch, c.mb
    gdescs = global_descs(mb, workload, cfg4_n)
    shard = mb.shard_descs(gdescs, c.rank, c.world) if c.world > 1 else gdescs
    descs, s0, d0, src_bytes, dst_bytes = rebase(shard)
    payload = int(descs["len"].sum())
    in_place = workload in ("cfg3", "cfg4")

    d_src = torch.empty(src_bytes, dtype=torch.uint8, device=c.dev)
    device_payload(torch, d_src, s0)
    d_dst = d_src if in_place else torch.empty(dst_bytes, dtype=torch.uint8, device=c.dev)
    hdr_np = synth.payload(1 << 40, HDR_BYTES)
    d_hdr = torch.from_numpy(hdr_np).to(c.dev)
    plan = mb.Plan(descs, src_bytes, dst_bytes)
    hdr_key = synth.PS4_KEY
    do_hdr = c.rank == 0

    def kernel():
        plan.run(d_src.data_ptr(), d_dst.data_ptr(), c.sh)

    def step(ev):
        if do_hdr:
            mb.cycle_device(d_hdr.data_ptr() + 4, d_hdr.data_ptr() + 4, HDR_BYTES - 4, hdr_key, c.side_h)
        if ev is not None:
            ev[0].record(c.stream)
        kernel()
        if ev is not None:
            ev[1].record(c.stream)

    # -- parity, before anything is timed: one pass over the plaintext, windows against the CPU oracle
    step(None)
    torch.cuda.synchronize()
    checked = check_parity(c, shard, descs, d_dst, workload)
    if do_hdr:
        import oracle
        want = hdr_np.copy()
        want[4:] = oracle.cycle(hdr_np[4:], hdr_key)
        if not np.array_equal(d_hdr.cpu().numpy(), want):
            raise SystemExit("PARITY FAILURE: HDR Cycle differs from the reference cipher")
        checked += HDR_BYTES - 4
    checked_total = int(c.reduce(float(checked), "sum"))
    step(None)  # in-place sets: back to plaintext (the cipher is an involution)

    if cooldown_s > 0:  # generating tens of GiB of payload is power-hungry too: idle until the power controller's
        torch.cuda.synchronize()  # averaging window has forgotten it, so the burst figure is a burst figure
        time.sleep(cooldown_s)
    ms_total, kernel_ms, clock_info, launches = timed_steps(c, step, kernel, args.steps, args.warmup)
    if dump_dir:  # before the sustained run, whose launch count depends on the measured kernel time
        dump_outputs(c, dump_dir, descs, d_dst, d_hdr if do_hdr else None)
    total_payload = int(gdescs["len"].sum())
    value = (total_payload + (HDR_BYTES - 4)) * args.steps / (ms_total * 1e-3) / 1e9
    out = {"value": value, "ms_per_step": ms_total / args.steps, "kernel_ms": kernel_ms,
           "payload_bytes_this_rank": payload, "entries_this_rank": int(len(descs)),
           "parity_bytes_checked": checked_total, "gpu_launches": int(launches), "clocks": clock_info,
           "roofline": roofline_block(c, payload, kernel_ms, workload, clock_info),
           "config": config_block(workload, gdescs, c.world)}
    if args.kernel_only:
        return out
    if sustain_s > 0:
        out["roofline"]["sustained"] = sustained(c, kernel, payload, kernel_ms, sustain_s)
        c.barrier()

    # -- end to end through the public C ABI with HOST (pinned) buffers: H2D + kernels + D2H per step
    if full:
        h_src = torch.empty(src_bytes, dtype=torch.uint8).pin_memory()
        if (workload in ("cfg3", "cfg4")) and (int(args.steps) % 2 == 1 or True):
            device_payload(torch, d_src, s0)  # whatever parity the timed loop left: start from plaintext
        h_src.copy_(d_src)
        h_dst = h_src if in_place else torch.empty(dst_bytes, dtype=torch.uint8).pin_memory()
        h_hdr = torch.from_numpy(hdr_np.copy()).pin_memory()
        del d_src, d_dst, plan
        torch.cuda.empty_cache()

        def e2e_step():
            if do_hdr:
                mb.cycle(h_hdr.data_ptr() + 4, HDR_BYTES - 4, hdr_key)
            mb.cycle_batch(descs, h_src.data_ptr(), h_dst.data_ptr(), src_bytes, dst_bytes)

        e2e_step()  # warm-up 1 doubles as the e2e parity pass: host output against the oracle
        h_out = h_dst.numpy()
        import oracle
        rng = np.random.default_rng(99 + c.rank)
        e2e_checked = 0
        for i, pos, n in parity_windows(descs, 16 * MIB, rng):
            g, l = shard[i], descs[i]
            want = oracle.cycle_at(synth.payload(int(g["src_off"]) + pos, n), int(g["key"]), pos)
            o = int(l["dst_off"]) + pos
            if not np.array_equal(h_out[o:o + n], want):
                raise SystemExit(f"PARITY FAILURE (e2e {workload}): rank {c.rank} piece {i}")
            e2e_checked += n
        e2e_step()  # warm-up 2 (in-place sets: back to plaintext)
        e2e_steps = args.steps
        c.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = c.reduce(time.perf_counter() - t0, "max")
        out["e2e"] = {"value": (total_payload + (HDR_BYTES - 4)) * e2e_steps / e2e_s / 1e9, "unit": "GB/s",
                      "h2d_bytes_per_step": payload + (HDR_BYTES - 4 if do_hdr else 0) + piece_count(descs) * 32,
                      "d2h_bytes_per_step": payload + (HDR_BYTES - 4 if do_hdr else 0),
                      "steps": e2e_steps, "api": "mod_cycle + mod_cycle_batch on pinned host buffers, one process per GPU",
                      "parity_bytes_checked": int(c.reduce(float(e2e_checked), "sum"))}
        ceiling = pcie_ceiling(c.world)
        if ceiling:
            out["e2e"]["copy_ceiling_gbs"] = ceiling
            out["e2e"]["frac_of_copy_ceiling"] = out["e2e"]["value"] / ceiling
        del h_src, h_dst
    return out


def pcie_ceiling(world: int):
    """Raw duplex pinned-copy ceiling (payload GB/s with one H2D and one D2H stream per GPU running at
    once) measured by tools/pcie_probe.py on this pool and committed in profiles/pcie.json."""
    try:
        with open(os.path.join(ROOT, "profiles", "pcie.json")) as f:
            return float(json.load(f)["duplex_payload_gbs"][str(world)])
    except Exception:
        return None


def inprocess_e2e(c: Ctx, args) -> dict:
    """The same 16 GiB set through the IN-PROCESS multi-GPU entry point (mod_cycle_batch_sharded: one host
    thread + stream set per device inside this one process), run by rank 0 alone while the other ranks
    wait.  Reported beside the one-process-per-GPU e2e."""
    torch, mb = c.torch, c.mb
    n_dev = min(c.world, mb.device_count())
    gdescs = global_descs(mb, "cfg3")
    total = int(gdescs["len"].sum())
    h = torch.empty(total, dtype=torch.uint8).pin_memory()
    h.zero_()
    mask = (1 << n_dev) - 1
    p = h.data_ptr()
    mb.cycle_batch_sharded(gdescs, p, p, total, total, mask)  # warm-up + parity (zero plaintext -> keystream)
    import oracle
    hv = h.numpy()
    for k in (0, 7, 31):
        o = k * PART + 12345
        if not np.array_equal(hv[o:o + 65536], oracle.cycle_at(np.zeros(65536, np.uint8), int(gdescs[k]["key"]), 12345)):
            raise SystemExit("PARITY FAILURE (in-process sharded e2e)")
    mb.cycle_batch_sharded(gdescs, p, p, total, total, mask)
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        mb.cycle_batch_sharded(gdescs, p, p, total, total, mask)
    dt = time.perf_counter() - t0
    return {"value": total * reps / dt / 1e9, "unit": "GB/s", "devices": n_dev, "steps": reps,
            "api": "mod_cycle_batch_sharded on one pinned host buffer, ONE process driving all devices"}


def measure_cfg5(c: Ctx, total: int = GIB, n_files: int = 10_000) -> dict:
    """BASELINE configs[4], end to end through the archive-level facade (include/modulate_ark.h) on a
    RAM-backed file system: a 1 GiB / 10 000-entry archive whose bodies are ciphered per entry is
    (1) unpacked -- CArk::Load + ExtractFiles: part files -> pinned slots -> GPU gather + decipher ->
    files, (2) one binary DTA entry is patched on the host (CDtaFile), (3) repacked --
    ConstructFromDirectory + BuildArk + SaveArk: files -> pinned slots -> GPU encipher -> part files,
    header re-serialised and re-enciphered.  Afterwards (untimed) every output byte is compared with
    what the CPU oracle says the repacked HDR and ARK must be."""
    import shutil
    import tempfile

    import arkfixture
    import oracle
    from oracle import ark_oracle as ao
    from oracle import dta_oracle as do
    from arkfixture import song_config_tree

    mb = c.mb
    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    root = tempfile.mkdtemp(prefix="mod_cfg5_", dir=base)
    key = 0x0BADF00D
    try:
        sizes = [int(x) for x in synth.entry_sizes_loguniform(n_files, total, lo=1 << 10, hi=1 << 20, seed=7)]
        tree = song_config_tree()
        dtb = do.serialise([tree])
        victim = 1234 % n_files
        sizes[0] += sizes[victim] - len(dtb)  # keep the total: the DTB entry has its own size
        sizes[victim] = len(dtb)
        hdr, payloads, _ = arkfixture.write_archive(root, n_files=n_files, n_parts=2, seed=5, body_key=key, sizes=sizes,
                                                    contents={victim: dtb})
        victim_name = hdr.entries[victim].name
        hdr_path = os.path.join(root, "main_ps4.hdr")
        out_dir, re_dir = os.path.join(root, "out"), os.path.join(root, "re")
        os.makedirs(re_dir)
        mb.ark_unpack(hdr_path, root, os.path.join(root, "warm"), key)  # warm-up: CUDA context, page cache, pinned pools
        shutil.rmtree(os.path.join(root, "warm"))

        # two timed repetitions, best one reported (both listed): on these VMs one call in four or so stalls for
        # ~0.8 s somewhere in the kernel's page handling (seen with and without the GPU legs before it)
        samples = []
        for rep in range(2):
            if rep:
                shutil.rmtree(out_dir)
                shutil.rmtree(re_dir)
                os.makedirs(re_dir)
            t0 = time.perf_counter()
            mb.ark_unpack(hdr_path, root, out_dir, key)
            t1 = time.perf_counter()
            mb.dta_set_int(os.path.join(out_dir, victim_name), "bpm", 174)
            t2 = time.perf_counter()
            mb.ark_pack(hdr_path, out_dir, re_dir, "main_ps4.hdr", ps4=True, pack_all=True, ignore_new_files=False, body_key=key)
            t3 = time.perf_counter()
            samples.append((t0, t1, t2, t3))
        t0, t1, t2, t3 = min(samples, key=lambda s: s[3] - s[0])

        # -- what the repacked archive must be, from the oracle: walk order, BuildArk offsets / parts, bodies
        #    re-enciphered per entry, header serialised in PS4 order and enciphered
        kids, i = do.find_node(tree, b"bpm")
        kids[i + 1] = ("int", 0, 174)
        by_name = {e.name: p for e, p in zip(hdr.entries, payloads)}
        by_name[victim_name] = do.serialise([tree])
        walk = arkfixture.reconstruct_walk(sorted(by_name))
        wsizes = [len(by_name[n]) for n in walk]
        offsets, parts = ao.build_ark(wsizes, ao.plan_part_sizes(sum(wsizes), len(hdr.parts)))
        image = np.frombuffer(b"".join(by_name[n] for n in walk), dtype=np.uint8).copy()
        packed_off = synth.packed_offsets(np.array(wsizes, dtype=np.int64))
        arkfixture.cipher_entries(image, packed_off, wsizes, key)
        model = ao.Header(ps4=True, parts=[(p, s) for (p, _), s in zip(hdr.parts, parts)],
                          entries=[ao.Entry(name=n, offset=o, size=s) for n, o, s in zip(walk, offsets, wsizes)])
        plain = ao.serialise_header(model)
        want_hdr = plain[:4] + oracle.cycle(np.frombuffer(plain[4:], dtype=np.uint8), ao.KEY_PS4).tobytes()
        got_hdr = open(os.path.join(re_dir, "main_ps4.hdr"), "rb").read()
        if got_hdr != want_hdr:
            raise SystemExit("PARITY FAILURE (cfg5): repacked HDR differs from the oracle")
        checked = len(got_hdr)
        pos = 0
        for (pth, _), psize in zip(hdr.parts, parts):
            got = np.fromfile(os.path.join(re_dir, pth), dtype=np.uint8)
            if got.size != psize or not np.array_equal(got, image[pos:pos + psize]):
                raise SystemExit(f"PARITY FAILURE (cfg5): repacked part {pth} differs from the oracle")
            pos += psize
            checked += psize
        for e, p in list(zip(hdr.entries, payloads))[::97]:  # and a sample of the extracted files
            want = by_name[e.name] if e.name == victim_name else p
            if open(os.path.join(out_dir, e.name), "rb").read() != want:
                raise SystemExit(f"PARITY FAILURE (cfg5): extracted {e.name} differs")
            checked += len(want)
        payload = sum(wsizes)
        return {"value": 2 * payload / (t3 - t0) / 1e9, "unit": "GB/s",
                "what": "payload bytes extracted + payload bytes repacked, per second of wall clock (unpack + DTA patch + pack)",
                "unpack_s": t1 - t0, "dta_patch_s": t2 - t1, "pack_s": t3 - t2,
                "samples_s": [{"unpack": b - a, "pack": d - c_} for a, b, c_, d in samples],
                "unpack_gbs": payload / (t1 - t0) / 1e9, "pack_gbs": payload / (t3 - t2) / 1e9,
                "entries": n_files, "payload_bytes": payload, "parity_bytes_checked": checked,
                "file_system": base, "host_threads": os.cpu_count(),
                "api": "mod_ark_unpack + mod_dta_set_int + mod_ark_pack (CArk / CDtaFile facade) on files"}
    finally:
        shutil.rmtree(root, ignore_errors=True)


def torch_mod():
    import torch
    return torch


def run_gpu_arm(args) -> None:
    c = Ctx()
    if args.workload == "cfg5":
        if c.rank == 0:
            r = measure_cfg5(c)
            print(json.dumps({"metric": METRIC, "value": r["value"], "unit": "GB/s", "n_gpus": 1, "steps": 1, "warmup": 1,
                              "ms_per_step": 1e3 * (r["unpack_s"] + r["dta_patch_s"] + r["pack_s"]), "higher_is_better": True,
                              "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                              "config": {"workload": "cfg5", "entries": r["entries"], "payload_bytes": r["payload_bytes"]},
                              "e2e": r, "parity_bytes_checked": r["parity_bytes_checked"]}), flush=True)
        c.finish()
        return
    if c.world != args.gpus and not (c.world == 1 and args.gpus == 1):
        if c.world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    main = measure_workload(c, args, args.workload, full=True, dump_dir=args.dump_outputs)
    extra = {}
    if not args.kernel_only and not args.no_extras:
        if c.world > 1 and args.workload == "cfg3":
            c.barrier()
            if c.rank == 0:
                try:
                    extra["e2e_inprocess"] = inprocess_e2e(c, args)
                except SystemExit:
                    raise
                except Exception as exc:  # reported, never fatal for the headline line
                    extra["e2e_inprocess"] = {"error": repr(exc)[:200]}
            c.barrier()
        if c.world == 1:
            for w in ("cfg2", "cfg4"):
                if w != args.workload:
                    sub_args = argparse.Namespace(**vars(args))
                    # burst figure from a SHORT timed region (a cfg4 step moves 67 GB: 20 of them run into the board's
                    # power cap half way and the "burst" number becomes a mixture), then the sustained run
                    sub_args.steps = max(5, min(args.steps, 20 if w == "cfg2" else 5))
                    sub_args.warmup = 3  # every 10 ms launch before the timed ones eats into the board's power budget
                    r = measure_workload(c, sub_args, w, full=False, sustain_s=1.5, cooldown_s=1.5)
                    extra[w] = {k: r[k] for k in ("value", "ms_per_step", "kernel_ms", "parity_bytes_checked",
                                                  "roofline", "config", "gpu_launches", "clocks")}
                    extra[w]["steps"] = sub_args.steps
            if c.rank == 0:
                os.sched_setaffinity(0, c.all_cpus)  # the file pipelines use every host core
                import gc
                gc.collect()  # hand the 16 GiB pinned + 33 GiB HBM blocks torch still caches back before the file legs
                if hasattr(torch_mod()._C, "_host_emptyCache"):
                    torch_mod()._C._host_emptyCache()
                torch_mod().cuda.empty_cache()
                try:
                    extra["cfg5"] = measure_cfg5(c)
                except SystemExit:
                    raise
                except Exception as exc:  # reported, never fatal for the headline line
                    extra["cfg5"] = {"error": repr(exc)[:300]}
    if c.rank != 0:
        c.finish()
        return

    # -- CPU baseline on this box (N == 1 only): the unmodified reference on a bounded sample
    cpu = None
    if c.world == 1 and not args.kernel_only:
        import oracle
        os.sched_setaffinity(0, c.all_cpus)  # the CPU baseline uses every host core
        kind = "reference" if oracle.have_ref() else "port"
        sample = cpu_sample(global_descs(c.mb, args.workload), args.workload)
        cores = min(os.cpu_count() or 1, len(sample["parts"]))
        work = np.empty(sample["bytes"], dtype=np.uint8)
        cpu_fill_plain(sample, work)
        cpu_step(sample, work, cores, kind)
        secs = min(cpu_step(sample, work, cores, kind) for _ in range(3))
        cpu = {"value": sample["bytes"] / secs / 1e9, "unit": "GB/s", "cores": cores if kind == "reference" else 1,
               "kind": kind, "sample": sample["sample"] + ", best of 3"}

    line = {
        "metric": METRIC, "value": main["value"], "unit": "GB/s", "n_gpus": c.world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic (counter-based splitmix64 payload generated on the device; identical to tests/synth.py)",
        "config": main["config"],
        "parity_bytes_checked": main["parity_bytes_checked"],
        "roofline": main["roofline"], "cpu_baseline": cpu,
        "e2e": main.get("e2e"),
        "gpu_launches": main["gpu_launches"], "clocks": main["clocks"],
        "host": "rank pinned to its GPU's NUMA-local CPUs (NVML affinity)" if c.numa_pinned else "default CPU affinity",
        "per_rank": {"payload_bytes": main["payload_bytes_this_rank"], "entries": main["entries_this_rank"],
                     "kernel_ms": main["kernel_ms"]},
        "extra": extra,
    }
    print(json.dumps(line), flush=True)
    c.finish()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--kernel-only", action="store_true",
                    help="profiling aid: device-resident legs only (no sustained run, e2e, extras or CPU baseline)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra.cfg2 / extra.cfg4 / in-process blocks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32, a seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "cfg5"):
        ap.error("--dump-outputs needs the GPU arm and a cfg2 / cfg3 / cfg4 workload")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
