"""GPU parity: the CUDA path (through the C ABI) against the oracle and the committed golden
vectors.  Bar: bit-exact (byte / integer work).  Run on the B200 box with `-m gpu`."""
import hashlib

import numpy as np
import pytest

import kernel_model
import oracle
import synth
from gpuutil import DeviceBuffer, sync

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def gpu_cycle(mb, data: np.ndarray, key: int) -> np.ndarray:
    buf = DeviceBuffer.from_numpy(data)
    mb.cycle(buf.ptr, data.size, key)
    out = buf.download()
    buf.free()
    return out


# ---- CEncryptionCycler::Cycle ------------------------------------------------------------------

def test_golden_keystreams(mb, golden):
    for k, hexbytes in golden["keystream_first64"].items():
        got = gpu_cycle(mb, np.zeros(64, np.uint8), int(k, 16))
        assert got.tobytes().hex() == hexbytes, k


def test_golden_deep_bytes(mb, golden):
    """Bytes far down the stream, reached by the kernel's jump-ahead, match what the reference
    reached by stepping."""
    n = (1 << 30) + 1
    buf = DeviceBuffer(n)
    for k, table in golden["deep_bytes"].items():
        key = int(k, 16)
        mb.cycle_device(buf.ptr, buf.ptr, 0, key)  # no-op length 0 is legal
        zero = np.zeros(1 << 24, np.uint8)
        for o in range(0, n, zero.size):
            buf.upload(zero[:min(zero.size, n - o)], o)
        mb.cycle(buf.ptr, n, key)
        for pos, val in table.items():
            if pos.startswith("window"):
                assert buf.download(1 << 29, 32).tobytes().hex() == val
            else:
                assert int(buf.download(int(pos), 1)[0]) == val, (k, pos)
    buf.free()


def test_golden_roundtrips(mb, golden):
    for case in golden["roundtrip"]:
        plain = synth.payload(0, case["size"])
        key = int(case["key"], 16)
        enc = gpu_cycle(mb, plain, key)
        assert sha(enc) == case["cycled_sha256"], case
        assert (gpu_cycle(mb, enc, key) == plain).all()


def test_golden_unaligned_windows(mb, golden):
    big = synth.payload(0, 1 << 16)
    for case in golden["unaligned"]:
        buf = DeviceBuffer.from_numpy(big)
        mb.cycle(buf.ptr + case["start"], case["size"], int(case["key"], 16))
        assert sha(buf.download()) == case["buffer_sha256"], case
        buf.free()


@pytest.mark.parametrize("size", [1, 2, 15, 16, 17, 31, 32, 33, 255, 511, 512, 513, 4095, 4096, 4097,
                                  8191, 8193, 65536, 100_003, 1_000_003, (4 << 20) + 5])
def test_cycle_sizes_vs_oracle(mb, size):
    data = synth.payload(size, size)
    for key in (synth.PS4_KEY, 0, 0x80000000, 0x12345678):
        assert (gpu_cycle(mb, data, key) == oracle.cycle(data, key)).all(), (size, hex(key))


def test_cycle_all_edge_keys(mb):
    data = synth.payload(99, 70_001)
    for key in synth.EDGE_KEYS + [2, 16807, 0x7FFFFFFD, 0x80000001, 0xDEADBEEF]:
        assert (gpu_cycle(mb, data, key) == oracle.cycle(data, key)).all(), hex(key)


@pytest.mark.parametrize("n", [5000, 41_003])
def test_cycle_every_alignment_combination(mb, n):
    """src and dst at every byte alignment, out of place; guard bytes around dst must survive.  5000 bytes
    stay inside one (edge) tile; 41 003 bytes have interior tiles, which take the predicate-free copy of the
    loop in each of its word-shift variants."""
    src_np = synth.payload(0, n + 64)
    src = DeviceBuffer.from_numpy(src_np)
    key = synth.PS3_KEY
    for so in range(0, 17):
        want = oracle.cycle(src_np[so:so + n], key)
        for do in range(0, 17):
            dst = DeviceBuffer.from_numpy(np.full(n + 64, 0xA5, np.uint8))
            mb.cycle_device(src.ptr + so, dst.ptr + do, n, key)
            sync()
            got = dst.download()
            assert (got[do:do + n] == want).all(), (so, do)
            assert (got[:do] == 0xA5).all() and (got[do + n:] == 0xA5).all(), (so, do)
            dst.free()
    src.free()


def test_cycle_small_lengths_every_alignment(mb):
    src_np = synth.payload(7, 256)
    src = DeviceBuffer.from_numpy(src_np)
    for n in (1, 2, 3, 15, 16, 17, 31, 32, 33, 47, 48, 49):
        for so in (0, 1, 5, 15):
            want = oracle.cycle(src_np[so:so + n], 0xDEADBEEF)
            for do in (0, 1, 7, 8, 15):
                dst = DeviceBuffer.from_numpy(np.full(128, 0x5A, np.uint8))
                mb.cycle_device(src.ptr + so, dst.ptr + do, n, 0xDEADBEEF)
                sync()
                got = dst.download()
                assert (got[do:do + n] == want).all(), (n, so, do)
                assert (got[:do] == 0x5A).all() and (got[do + n:] == 0x5A).all(), (n, so, do)
                dst.free()
    src.free()


def test_cycle_host_pointer_paths(mb):
    """mod_cycle on host memory (pageable numpy, bytearray) stages through HBM in slices."""
    for size in (1, 4097, 65536, 1_000_003, (40 << 20) + 3):
        data = synth.payload(1, size)
        want = oracle.cycle(data, synth.PS4_KEY) if size <= (8 << 20) else None
        work = data.copy()
        mb.CEncryptionCycler().Cycle(work, size, synth.PS4_KEY)
        if want is not None:
            assert (work == want).all(), size
        else:  # sampled windows + involution for the large case
            for o in (0, (16 << 20) - 8, (32 << 20) - 3, size - 100):
                w = min(100, size - o)
                assert (work[o:o + w] == oracle.cycle_at(data[o:o + w], synth.PS4_KEY, o)).all(), o
        mb.CEncryptionCycler().Cycle(work, size, synth.PS4_KEY)
        assert (work == data).all()
    ba = bytearray(synth.payload(0, 1000).tobytes())
    mb.cycle(ba, None, 1)
    assert bytes(ba) == oracle.cycle(synth.payload(0, 1000), 1).tobytes()


def test_cycle_beyond_32bit_length_and_period(mb):
    """64-bit lengths: one stream of 4 GiB + 1 MiB keeps the keystream going past the reference's
    32-bit limit and past the period 2^31-2 (checked against closed-form windows)."""
    n = (4 << 30) + (1 << 20) + 5
    buf = DeviceBuffer(n)
    zero = np.zeros(64 << 20, np.uint8)
    for o in range(0, n, zero.size):
        buf.upload(zero[:min(zero.size, n - o)], o)
    key = 0x12345678
    mb.cycle(buf.ptr, n, key)
    period = (1 << 31) - 2
    for o in (0, (1 << 30) - 20, (1 << 30), period - 30, (1 << 31) + 11, (1 << 32) - 40, (1 << 32), n - 64):
        got = buf.download(o, 64)
        want = oracle.cycle_at(np.zeros(64, np.uint8), key, o)
        assert (got == want).all(), o
    # periodicity: byte i equals byte i + (2^31 - 2)
    assert (buf.download(1000, 4096) == buf.download(1000 + period, 4096)).all()
    buf.free()


def test_whole_archive_1gib_roundtrip_and_samples(mb):
    """BASELINE config 2 (i): 1 GiB image, one key; sampled windows against the oracle, then
    decrypt restores the plain image exactly (checksum of the whole buffer)."""
    n = 1 << 30
    buf = DeviceBuffer(n)
    buf.fill_payload(0)
    plain_sha = hashlib.sha256()
    for o in range(0, n, 64 << 20):
        plain_sha.update(buf.download(o, 64 << 20).tobytes())
    mb.cycle(buf.ptr, n, synth.PS4_KEY)
    rng = np.random.default_rng(9)
    for o in [0, n - 4096] + [int(x) for x in rng.integers(0, n - 4096, size=24)]:
        got = buf.download(o, 4096)
        assert (got == oracle.cycle_at(synth.payload(o, 4096), synth.PS4_KEY, o)).all(), o
    mb.cycle(buf.ptr, n, synth.PS4_KEY)
    back = hashlib.sha256()
    for o in range(0, n, 64 << 20):
        back.update(buf.download(o, 64 << 20).tobytes())
    assert back.hexdigest() == plain_sha.hexdigest()
    buf.free()


# ---- descriptor batches (CArk gather / scatter + per-entry keys) ---------------------------------

def _run_batch(mb, descs, src_np, dst_np):
    src = DeviceBuffer.from_numpy(src_np)
    dst = DeviceBuffer.from_numpy(dst_np)
    mb.cycle_batch(descs, src.ptr, dst.ptr, src_np.size, dst_np.size)
    out = dst.download()
    src.free()
    dst.free()
    return out


def test_batch_golden_fixture(mb, golden):
    b = golden["batch"]
    descs = mb.make_descs(b["src_off"], b["dst_off"], b["len"], np.array(b["key"], dtype=np.int64))
    src = synth.payload(0, b["src_bytes"])
    dst = np.full(b["dst_bytes"], b["dst_fill"], dtype=np.uint8)
    assert sha(_run_batch(mb, descs, src, dst)) == b["dst_sha256"]
    # host-pointer form of the same call
    host_dst = dst.copy()
    mb.cycle_batch(descs, src.copy(), host_dst)
    assert sha(host_dst) == b["dst_sha256"]


@pytest.mark.parametrize("seed", range(6))
def test_batch_random_vs_oracle(mb, seed):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(1, 400))
    max_len = [40, 600, 5000, 20000, 70000, 300000][seed]
    sizes = rng.integers(0, max_len, size=n).astype(np.int64)
    src_off = synth.packed_offsets(sizes) + int(rng.integers(0, 16))
    order = rng.permutation(n)
    dst_off = np.zeros(n, np.int64)
    run = int(rng.integers(0, 16))
    for i in order:
        dst_off[i] = run
        run += int(sizes[i]) + int(rng.integers(0, 3))
    src = synth.payload(seed, int(src_off[-1] + sizes[-1]) + 9)
    dst = np.full(run + 5, 0xC3, np.uint8)
    descs = mb.make_descs(src_off, dst_off, sizes, synth.entry_keys(n, seed=seed + 1))
    want = oracle.cycle_batch(descs, src, dst.copy())
    assert (_run_batch(mb, descs, src, dst) == want).all()


def test_batch_in_place_and_plan_reuse(mb):
    sizes = synth.entry_sizes_loguniform(300, 8 << 20, lo=64, hi=1 << 18, seed=3)
    off = synth.packed_offsets(sizes)
    keys = synth.entry_keys(len(sizes))
    descs = mb.make_descs(off, off, sizes, keys)
    plain = synth.payload(0, 8 << 20)
    want = oracle.cycle_batch(descs, plain, plain.copy())
    buf = DeviceBuffer.from_numpy(plain)
    plan = mb.Plan(descs, plain.size, plain.size)
    assert plan.payload_bytes == 8 << 20
    plan.run(buf.ptr, buf.ptr)
    sync()
    assert (buf.download() == want).all()
    plan.run(buf.ptr, buf.ptr)  # involution: the same plan decrypts
    sync()
    assert (buf.download() == plain).all()
    plan.close()
    buf.free()


def test_plan_records_come_from_a_block_pool(mb):
    """mod_plan_destroy hands the plan's HBM records to a per-device pool and the next mod_plan_create may reuse
    the block (cudaMalloc / cudaFree stay off the per-archive path).  Plans of shrinking, growing and equal sizes,
    created and destroyed in turn and two alive at once, must each produce the oracle's bytes; mod_shutdown
    releases the pool and the library comes back up afterwards."""
    from modulate_b200 import _abi
    rng = np.random.default_rng(77)
    src_np = synth.payload(3, 6 << 20)

    def case(n, max_len, seed):
        sizes = np.random.default_rng(seed).integers(1, max_len, size=n).astype(np.int64)
        scale = min(1.0, (5 << 20) / float(sizes.sum()))
        sizes = np.maximum(1, (sizes * scale).astype(np.int64))
        off = synth.packed_offsets(sizes) + 5
        return mb.make_descs(off, off - 5, sizes, synth.entry_keys(n, seed=seed))

    src = DeviceBuffer.from_numpy(src_np)
    held = None
    for i, (n, max_len) in enumerate([(4000, 3000), (50, 200000), (3000, 4000), (7, 900000), (4000, 3000), (1, 100)]):
        descs = case(n, max_len, 200 + i)
        dst_np = np.full(6 << 20, 0x3C, np.uint8)
        want = oracle.cycle_batch(descs, src_np, dst_np.copy())
        dst = DeviceBuffer.from_numpy(dst_np)
        plan = mb.Plan(descs, src_np.size, dst_np.size)
        plan.run(src.ptr, dst.ptr)
        sync()
        assert (dst.download() == want).all(), i
        dst.free()
        if held is not None:
            held.close()
        held = plan if i % 2 == 0 else None  # every other plan stays alive while the next one is built
        if held is None:
            plan.close()
    if held is not None:
        held.close()
    src.free()
    _abi.load().mod_shutdown()  # frees the pool with everything else; the next call re-creates the context
    data = synth.payload(9, 100_000)
    assert (gpu_cycle(mb, data, 0x1234567) == oracle.cycle(data, 0x1234567)).all()


def test_batch_identity_key_is_plain_copy(mb):
    """key == 0 (mod m) is the reference's plain extract: ExtractFiles' fwrite (CArk.cpp:494)."""
    sizes = np.array([1, 100, 4096, 70001, 33], np.int64)
    src_off = synth.packed_offsets(sizes) + 3
    dst_off = synth.packed_offsets(sizes)[::-1].copy()
    src = synth.payload(5, int(sizes.sum()) + 3)
    descs = mb.make_descs(src_off, np.array([0, 1, 101, 4197, 74198]), sizes, [0, 0x7FFFFFFF, 0, 0x7FFFFFFF, 0])
    out = _run_batch(mb, descs, src, np.zeros(int(sizes.sum()), np.uint8))
    want = np.concatenate([src[int(o):int(o) + int(l)] for o, l in zip(src_off, sizes)])
    assert (out == want).all()
    del dst_off


def test_batch_errors_are_loud(mb):
    src = DeviceBuffer(1024)
    dst = DeviceBuffer(1024)
    bad = mb.make_descs([1000], [0], [100], [1])
    with pytest.raises(mb.ModError) as ei:
        mb.cycle_batch(bad, src.ptr, dst.ptr, 1024, 1024)
    assert ei.value.code == -2
    bad = mb.make_descs([0], [1000], [100], [1])
    with pytest.raises(mb.ModError):
        mb.cycle_batch(bad, src.ptr, dst.ptr, 1024, 1024)
    plan = mb.Plan(mb.make_descs([0], [0], [100], [1]), 1024, 1024, dst_align=0)
    with pytest.raises(mb.ModError) as ei:
        plan.run(src.ptr, dst.ptr + 1)
    assert ei.value.code == -3
    plan.close()
    mb.cycle_batch(mb.make_descs([], [], [], []), src.ptr, dst.ptr, 1024, 1024)  # empty batch is legal
    src.free()
    dst.free()


def test_archive_10k_entries_extract(mb):
    """BASELINE config 2 (ii) at 1/8 scale for the full compare: 10 000 byte-packed entries with
    per-entry keys gathered out of a 128 MiB image in one launch; every byte against the oracle."""
    total = 128 << 20
    sizes = synth.entry_sizes_loguniform(10_000, total, lo=128, hi=1 << 17)
    src_off = synth.packed_offsets(sizes)
    descs = mb.make_descs(src_off, src_off, sizes, synth.entry_keys(len(sizes)))
    src_np = synth.payload(0, total)
    want = oracle.cycle_batch(descs, src_np, np.zeros(total, np.uint8))
    got = _run_batch(mb, descs, src_np, np.zeros(total, np.uint8))
    assert (got == want).all()


def test_many_small_entries(mb):
    """BASELINE config 4 shape (1-64 KiB entries, per-entry keys, one launch) at 20k entries:
    sampled entries, and every entry that holds a byte only the kernel's redo branch gets right
    (tests/kernel_model.py), against the oracle; every entry through the decrypt round trip."""
    rng = np.random.default_rng(4)
    n = 20_000
    sizes = rng.integers(1 << 10, (64 << 10) + 1, size=n).astype(np.int64)
    off = synth.packed_offsets(sizes)
    total = int(sizes.sum())
    keys = synth.entry_keys(n)
    descs = mb.make_descs(off, off, sizes, keys)
    buf = DeviceBuffer(total)
    buf.fill_payload(0)
    plan = mb.Plan(descs, total, total)
    plan.run(buf.ptr, buf.ptr)
    sync()
    sampled = [0, 1, 2, 3, 4, n - 1] + [int(x) for x in rng.integers(0, n, size=40)]
    redo = kernel_model.entries_with_trigger_bytes(list(zip(off.tolist(), off.tolist(), sizes.tolist(), keys.tolist())))
    assert len(redo) > 1000
    for i in sampled + [int(x) for x in redo]:
        o, l = int(off[i]), int(sizes[i])
        assert (buf.download(o, l) == oracle.cycle(synth.payload(o, l), int(keys[i]))).all(), i
    plan.run(buf.ptr, buf.ptr)
    sync()
    for o in range(0, total, 64 << 20):
        m = min(64 << 20, total - o)
        assert (buf.download(o, m) == synth.payload(o, m)).all()
    plan.close()
    buf.free()


def test_sharded_plans_equal_unsharded(mb):
    """Offset-range sharding emulated on one GPU: the 4 shards of a batch (large entries cut, tail
    pieces with jumped keys) run one after another give the unsharded result byte for byte."""
    sizes = np.array([3 << 20, 17, 40 << 20, 0, 999_999, 20 << 20, 5], np.int64)
    off = synth.packed_offsets(sizes) + 1
    total = int(off[-1] + sizes[-1])
    descs = mb.make_descs(off, off, sizes, synth.entry_keys(len(sizes), seed=77))
    src = DeviceBuffer(total)
    src.fill_payload(0)
    whole = DeviceBuffer(total)
    parts = DeviceBuffer(total)
    zero = np.zeros(total, np.uint8)
    whole.upload(zero)
    parts.upload(zero)
    mb.cycle_batch(descs, src.ptr, whole.ptr, total, total)
    for r in range(4):
        shard = mb.shard_descs(descs, r, 4)
        mb.cycle_batch(shard, src.ptr, parts.ptr, total, total)
    assert (whole.download() == parts.download()).all()
    # and a sampled oracle check of the unsharded result inside the biggest entry
    o = int(off[2]) + (33 << 20) + 7
    assert (whole.download(o, 1000) == oracle.cycle_at(synth.payload(o, 1000), int(descs[2]["key"]),
                                                       o - int(off[2]))).all()
    for b in (src, whole, parts):
        b.free()


@pytest.mark.parametrize("layout", ["packed", "shuffled", "holes"])
def test_batch_host_buffers_pipelined(mb, layout, monkeypatch):
    """mod_cycle_batch on HOST buffers: grouped H2D / kernel / D2H pipeline (small groups forced),
    the non-monotone fallback, and a destination with many holes (bytes between entries survive)."""
    monkeypatch.setenv("MOD_GROUP_BYTES", str(1 << 20))
    rng = np.random.default_rng(8)
    n = 600
    sizes = synth.entry_sizes_loguniform(n, 12 << 20, lo=16, hi=1 << 17, seed=5)
    src_off = synth.packed_offsets(sizes)
    if layout == "packed":
        dst_off = synth.packed_offsets((sizes + 15) & ~15)  # 16-byte aligned slots, monotone, padding < 16
    elif layout == "shuffled":
        order = rng.permutation(n)
        dst_off = np.zeros(n, np.int64)
        run = 3
        for i in order:
            dst_off[i] = run
            run += int(sizes[i])
        # present the descriptors in destination order so that source windows jump around
        src_off, sizes, dst_off = src_off[order], sizes[order], dst_off[order]
    else:
        dst_off = src_off * 2 + 7  # every entry followed by a hole
    keys = synth.entry_keys(n, seed=21)
    descs = mb.make_descs(src_off, dst_off, sizes, keys)
    src = synth.payload(3, int((src_off + sizes).max()))
    dst = np.full(int((dst_off + sizes).max()) + 9, 0x77, np.uint8)
    want = oracle.cycle_batch(descs, src, dst.copy())
    mb.cycle_batch(descs, src, dst)
    assert (dst == want).all()


@pytest.mark.parametrize("src_shift,dst_shift", [(0, 0), (16, 48), (5, 5), (3, 16), (128, 64)])
@pytest.mark.parametrize("in_place", [False, True])
def test_batch_host_copy_alignment(mb, src_shift, dst_shift, in_place, monkeypatch):
    """The host-pointer batch path widens uploads and splits downloads at 128-byte boundaries of the HOST
    addresses when the caller's buffers are 16-byte aligned, and keeps plain copies otherwise.  Byte-packed
    entries (groups start anywhere), caller buffers at several phases, guard bytes either side of dst."""
    monkeypatch.setenv("MOD_GROUP_BYTES", str(1 << 20))
    n = 300
    sizes = synth.entry_sizes_loguniform(n, 9 << 20, lo=1, hi=1 << 18, seed=31)
    src_off = synth.packed_offsets(sizes) + 77
    dst_off = src_off if in_place else synth.packed_offsets(sizes) + 1000
    descs = mb.make_descs(src_off, dst_off, sizes, synth.entry_keys(n, seed=33))
    total = int((src_off + sizes).max()) + 300
    base = np.zeros(total + 4096 + 256, np.uint8)
    a0 = (-base.ctypes.data) % 4096  # a page-aligned origin inside the array, then the requested phases
    src = base[a0 + src_shift:a0 + src_shift + total]
    src[:] = synth.payload(11, total)
    if in_place:
        dst = src
        want = oracle.cycle_batch(descs, src.copy(), src.copy())
    else:
        dbase = np.full(total + 4096 + 256 + 1200, 0x5E, np.uint8)
        d0 = (-dbase.ctypes.data) % 4096
        dst = dbase[d0 + dst_shift:d0 + dst_shift + total + 1200]
        want = oracle.cycle_batch(descs, src, dst.copy())
    mb.cycle_batch(descs, src, dst)
    assert (dst == want).all(), (src_shift, dst_shift, in_place)
    if not in_place:
        assert (dbase[:d0 + dst_shift] == 0x5E).all() and (dbase[d0 + dst_shift + total + 1200:] == 0x5E).all()


def test_config3_16gib_multipart_sharded(mb):
    """BASELINE config 3 at FULL size: a 16 GiB set = 32 parts x 512 MiB (kuMaxArkSize, CArk.cpp:19),
    one (offset, len, key) per part, cut into 8 offset-range shards whose boundaries fall INSIDE
    parts (forces jump-ahead).  The shards run one after another on this GPU, in place.  Checked by
    size-independent properties: sampled windows against the closed-form oracle (zero plaintext ->
    the buffer is the keystream), shard union == unsharded run on a sampled basis, and decrypt
    restores all-zero (full-buffer check)."""
    part = 512 << 20
    n_parts = 32
    total = part * n_parts
    keys = synth.entry_keys(n_parts, seed=303)
    off = np.arange(n_parts, dtype=np.int64) * part
    descs = mb.make_descs(off, off, np.full(n_parts, part, np.int64), keys)
    buf = DeviceBuffer(total)
    zero = np.zeros(256 << 20, np.uint8)
    for o in range(0, total, zero.size):
        buf.upload(zero, o)
    world = 8
    shard_payload = []
    for r in range(world):
        shard = mb.shard_descs(descs, r, world)
        shard_payload.append(int(shard["len"].sum()))
        mb.cycle_batch(shard, buf.ptr, buf.ptr, total, total)
    assert sum(shard_payload) == total and max(shard_payload) - min(shard_payload) <= 32
    # shard boundaries are inside parts: 16 GiB / 8 = 2 GiB = 4 parts exactly -> shift the check:
    # also cut in 7 to force interior cuts, on a scratch copy of two parts (below)
    rng = np.random.default_rng(12)
    probes = [0, part - 64, part, total - 4096, 5 * part + 12345] + [int(x) for x in rng.integers(0, total - 4096, size=40)]
    for o in probes:
        p = o // part
        n = min(4096, (p + 1) * part - o)
        want = oracle.cycle_at(np.zeros(n, np.uint8), int(keys[p]), o - p * part)
        assert (buf.download(o, n) == want).all(), o
    # decrypt with 7 shards (boundaries now fall inside parts) and verify all-zero everywhere
    for r in range(7):
        shard = mb.shard_descs(descs, r, 7)
        if r < 6:
            last = shard[-1]
            assert (int(last["src_off"]) + int(last["len"])) % part != 0  # cut inside a part
        mb.cycle_batch(shard, buf.ptr, buf.ptr, total, total)
    for o in range(0, total, zero.size):
        assert not buf.download(o, zero.size).any(), o
    buf.free()


def test_config4_one_million_small_entries(mb):
    """BASELINE config 4 at FULL size: 1 000 000 byte-packed entries of 1..64 KiB (about 32.5 GiB) with
    per-entry keys, ONE launch of the batched kernel, in place.  Sampled entries (incl. the five edge
    keys and the last entry) against the oracle; the same plan run again restores all-zero."""
    rng = np.random.default_rng(44)
    n = 1_000_000
    sizes = rng.integers(1 << 10, (64 << 10) + 1, size=n).astype(np.int64)
    off = synth.packed_offsets(sizes)
    total = int(sizes.sum())
    keys = synth.entry_keys(n, seed=404)
    descs = mb.make_descs(off, off, sizes, keys)
    buf = DeviceBuffer(total)
    zero = np.zeros(256 << 20, np.uint8)
    for o in range(0, total, zero.size):
        buf.upload(zero[:min(zero.size, total - o)], o)
    plan = mb.Plan(descs, total, total)
    assert plan.payload_bytes == total
    launches = mb.launch_count()
    plan.run(buf.ptr, buf.ptr)
    sync()
    assert mb.launch_count() - launches == 1  # one variable-length batched launch for the million entries
    for i in [0, 1, 2, 3, 4, n - 1, n // 2] + [int(x) for x in rng.integers(0, n, size=60)]:
        o, l = int(off[i]), int(sizes[i])
        assert (buf.download(o, l) == oracle.keystream(int(keys[i]), l)).all(), i
    plan.run(buf.ptr, buf.ptr)
    sync()
    for o in range(0, total, zero.size):
        m = min(zero.size, total - o)
        assert not buf.download(o, m).any(), o
    plan.close()
    buf.free()


def test_max_length_entry_4gib_minus_1(mb):
    """One descriptor at the reference's length limit (unsigned int: 2^32 - 1 bytes), destination
    misaligned by one byte so the entry needs 2^28 + 1 chunks: exercises the top of the tile /
    jump-table range.  Zero plaintext -> the output is the keystream; windows against the closed form."""
    n = (1 << 32) - 1
    key = 0x7FFFFFFE
    src = DeviceBuffer(n + 16)
    dst = DeviceBuffer(n + 32)
    zero = np.zeros(256 << 20, np.uint8)
    for o in range(0, n + 16, zero.size):
        src.upload(zero[:min(zero.size, n + 16 - o)], o)
    guard = np.full(32, 0xAB, np.uint8)
    dst.upload(guard[:1], 0)
    dst.upload(guard[:31], n + 1)
    descs = mb.make_descs([5], [1], [n], [key])
    mb.cycle_batch(descs, src.ptr, dst.ptr, n + 16, n + 32)
    for o in (0, 1, 15, 16, 8191, 8192, (1 << 31) - 3, (1 << 31) + 7, n - 8192 - 3, n - 64):
        w = min(64, n - o)
        assert (dst.download(1 + o, w) == oracle.cycle_at(np.zeros(w, np.uint8), key, o)).all(), o
    assert dst.download(0, 1)[0] == 0xAB and (dst.download(n + 1, 31) == 0xAB).all()
    src.free()
    dst.free()
