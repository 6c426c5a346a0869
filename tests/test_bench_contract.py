"""The bench.py JSON contract: reference arm on CPU here, the GPU arm on the B200 box."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMMON = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
          "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def run_bench(*args, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert COMMON <= set(d) and d["impl"] == "reference"
    assert d["unit"] == "GB/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["config"]["workload"] == "cfg3" and d["dtype"] == "u8" and d["scaling"] == "strong"
    assert d["config"]["payload_bytes"] == 16 << 30 and d["config"]["entries"] == 32
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone runs and prints the reference arm; the other ranks exit 0 without work."""
    env = dict(os.environ, RANK="3", LOCAL_RANK="3", WORLD_SIZE="8")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "8", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == "", out.stdout + out.stderr


def test_device_payload_is_the_synth_stream():
    """bench.py generates its plaintext where the buffer lives (torch int64 splitmix64); it must be the
    same counter-based stream the oracle side regenerates window by window (tests/synth.py)."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench
    import synth
    for off, n in [(0, 64), (3, 1001), (123457, 1 << 18), ((1 << 34) + 5, 4099), ((16 << 30) - 77, 77)]:
        out = torch.empty(n, dtype=torch.uint8)
        bench.device_payload(torch, out, off, slice_bytes=1 << 16)
        assert (out.numpy() == synth.payload(off, n)).all(), (off, n)


def test_parity_windows_cover_both_sides_of_every_cut():
    """Every rank checks the first and last 256 KiB of each piece of its shard, so both sides of every
    interior cut and part boundary are compared by one rank or the other, and at least 64 MiB per rank."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    import modulate_b200 as mb
    descs = bench.global_descs(mb, "cfg3")
    for world in (1, 2, 3, 8):
        covered_starts, covered_ends = set(), set()
        for rank in range(world):
            shard = mb.shard_descs(descs, rank, world) if world > 1 else descs
            wins = bench.parity_windows(shard, bench.PARITY_TARGET, np.random.default_rng(rank))
            assert sum(w[2] for w in wins) >= bench.PARITY_TARGET
            for i, pos, n in wins:
                assert 0 <= pos and pos + n <= int(shard[i]["len"])
                if pos == 0:
                    covered_starts.add(int(shard[i]["dst_off"]))
                if pos + n == int(shard[i]["len"]):
                    covered_ends.add(int(shard[i]["dst_off"]) + int(shard[i]["len"]))
        total = int(descs["len"].sum())
        cuts = {total * r // world & ~15 for r in range(1, world)} | {int(d["dst_off"]) for d in descs[1:]}
        assert cuts <= covered_starts and cuts <= covered_ends


@pytest.mark.gpu
def test_gpu_arm_line():
    """The headline line: BASELINE configs[2] (16 GiB multi-part set), parity checked in the run."""
    d = run_bench("--steps", "5", "--warmup", "3")
    assert COMMON | {"roofline", "clocks", "parity_bytes_checked", "extra"} <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["warmup"] == 3 and d["scaling"] == "strong"
    assert d["config"]["workload"] == "cfg3" and d["dtype"] == "u8" and d["data"].startswith("synthetic")
    assert d["config"]["payload_bytes"] == 16 << 30
    assert d["parity_bytes_checked"] >= 64 << 20
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["algorithmic_bytes_per_launch"] == 2 * d["config"]["payload_bytes"]
    assert 0.3 < r["frac"] < 1.25
    s = r["sustained"]
    assert s["seconds"] >= 3.0 and 0.3 < s["frac"] < 1.25 and s["clocks"]["samples"] > 10
    assert d["gpu_launches"] == 2 * d["steps"]          # HDR Cycle + one batched launch per step
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > d["config"]["payload_bytes"] and e["d2h_bytes_per_step"] > 0
    assert 0 < e["value"] < d["value"] and e["parity_bytes_checked"] > 0 and e["steps"] == d["steps"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] > 0
    assert d["clocks"]["sm_max_mhz"] and isinstance(d["clocks"]["reasons"], list)
    for w, entries in (("cfg2", 10_000), ("cfg4", 1_000_000)):
        x = d["extra"][w]
        assert x["config"]["workload"] == w and x["config"]["entries"] == entries
        assert x["parity_bytes_checked"] > 0 and 0.3 < x["roofline"]["frac"] < 1.25


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_steps_wrote(tmp_path):
    """--dump-outputs DIR: float32 files of at most 64 MB in all.  The gather workload (cfg2) writes a fresh
    destination every step, so every sampled byte must be the oracle's cipher of its entry; the HDR is Cycled
    in place 7 times (parity pass, restore, 3 warm-ups, 2 timed steps), so it holds ciphertext."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    import modulate_b200 as mb
    import oracle
    import synth
    run_bench("--workload", "cfg2", "--kernel-only", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert sorted(p.name for p in tmp_path.iterdir()) == ["hdr.npy", "payload.npy"]
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    got = np.load(tmp_path / "payload.npy")
    descs = bench.global_descs(mb, "cfg2")
    idx, pos, width = bench.dump_windows(descs, 1)
    want = np.concatenate([oracle.cycle_at(synth.payload(int(descs[i]["src_off"]) + p, n), int(descs[i]["key"]), p)
                           for i, p, n in zip(idx, pos, width)])
    assert got.dtype == np.float32 and got.size == int(width.sum()) >= 1 << 20
    assert np.array_equal(got, want.astype(np.float32))
    hdr = np.load(tmp_path / "hdr.npy")
    plain = synth.payload(1 << 40, bench.HDR_BYTES)
    assert hdr.dtype == np.float32 and np.array_equal(hdr[:4], plain[:4].astype(np.float32))
    assert np.array_equal(hdr[4:], oracle.cycle(plain[4:], synth.PS4_KEY).astype(np.float32))
