"""GPU parity over the cipher kernels' path matrix: one launch per (launch kind, run_tile path, redo trigger)
cell that tests/kernel_model.py finds reachable, built so that the model says the launch reaches that cell
(with a key that makes the chosen chunk take the redo branch).  Every byte of the destination buffer --
sentinel guards and the holes between entries included -- is compared with the oracle.

Contiguous calls reach partial chunks that do not take the slow path only where they cross a 1 GiB
piece boundary; those cases cycle one call of 1 GiB + a few KiB and compare every tile the model keeps
(the first two and last two of each piece) plus the guard bytes.

A "ghost" cell's trigger lies in a chunk beyond the entry, in a thread that also owns a valid chunk: no
stored byte depends on the trigger itself, so a ghost cell does not show that the redo runs.  It checks
what the redo does when it runs: its start states and that it stores nothing beyond the entry."""
import functools
import zlib

import numpy as np
import pytest

import kernel_model as km
import oracle
import synth
from gpuutil import DeviceBuffer, sync

pytestmark = pytest.mark.gpu

SENTINEL = 0xC5


@functools.lru_cache(maxsize=None)
def _cases():
    return {c.cell: c for c in km.cases()}


def _descs(mb, descs):
    so, do, ln, key = zip(*descs)
    return mb.make_descs(list(so), list(do), list(ln), [k & 0xFFFFFFFF for k in key])


@pytest.fixture(scope="module")
def piece_buffers():
    """Source, destination and in-place buffers for contiguous calls of more than one piece: the sources
    hold synth.payload(offset), so any window of them can be regenerated on the host."""
    n = km.MAX_PIECE + (64 << 10)
    bufs = [DeviceBuffer(n) for _ in range(3)]
    bufs[0].fill_payload(0)
    bufs[2].fill_payload(0)
    yield bufs
    for b in bufs:
        b.free()


def _check_pieces(mb, case, bufs):
    src, dst, inplace = bufs
    assert max(case.src_alloc, case.dst_alloc) <= src.nbytes
    (so, do, ln, key), = case.descs
    ranges = case.modelled_ranges()
    assert any(hi == km.MAX_PIECE for lo, hi in ranges)  # the tile that ends the first piece is checked
    p, q = case.src_ptr + so, case.dst_ptr + do
    if case.kind == "inline-inplace":
        assert p == q
        mb.cycle_device(inplace.ptr + p, inplace.ptr + p, ln, key)
        sync()
        bad = [lo for lo, hi in ranges if not (inplace.download(p + lo, hi - lo) ==
                                               oracle.cycle_at(synth.payload(p + lo, hi - lo), key, lo)).all()]
        guards_ok = (inplace.download(0, p) == synth.payload(0, p)).all() and \
            (inplace.download(p + ln, 48) == synth.payload(p + ln, 48)).all()
        mb.cycle_device(inplace.ptr + p, inplace.ptr + p, ln, key)  # restore the shared buffer before asserting
        sync()
        assert not bad and guards_ok, (case.cell, bad)
        assert all((inplace.download(p + lo, hi - lo) == synth.payload(p + lo, hi - lo)).all() for lo, hi in ranges)
        return
    dst.upload(np.full(q, SENTINEL, np.uint8))
    dst.upload(np.full(48, SENTINEL, np.uint8), q + ln)
    mb.cycle_device(src.ptr + p, dst.ptr + q, ln, key)
    sync()
    for lo, hi in ranges:
        assert (dst.download(q + lo, hi - lo) == oracle.cycle_at(synth.payload(p + lo, hi - lo), key, lo)).all(), \
            (case.cell, lo)
    assert (dst.download(0, q) == SENTINEL).all() and (dst.download(q + ln, 48) == SENTINEL).all(), case.cell


def _buffer(a: np.ndarray) -> DeviceBuffer:
    b = DeviceBuffer.from_numpy(a)
    assert b.ptr % 16 == 0  # the model's addresses are offsets from 16-byte aligned bases
    return b


@pytest.mark.parametrize("cell", sorted(km.reachable_cells()), ids=lambda c: "-".join(c).replace("/", "."))
def test_kernel_path_cell(mb, cell, monkeypatch, request):
    case = _cases()[cell]
    assert cell in case.cells()
    if case.force_general:
        monkeypatch.setenv("MOD_FORCE_GENERAL", "1")
    if case.kind.startswith("inline") and case.descs[0][2] > km.MAX_PIECE:
        _check_pieces(mb, case, request.getfixturevalue("piece_buffers"))
        return
    src_np = synth.payload(zlib.crc32(repr(cell).encode()) & 0xFFFFF, case.src_alloc)
    if case.kind.startswith("inline"):
        (so, do, ln, key), = case.descs
        enc = oracle.cycle(src_np[case.src_ptr + so:case.src_ptr + so + ln], key)
        if case.kind == "inline-inplace":
            buf = _buffer(src_np)
            want = src_np.copy()
            want[case.dst_ptr + do:case.dst_ptr + do + ln] = enc
            mb.cycle_device(buf.ptr + case.src_ptr, buf.ptr + case.dst_ptr, ln, key)
            sync()
            assert (buf.download() == want).all(), cell
            return
        src = _buffer(src_np)
        dst = _buffer(np.full(case.dst_alloc, SENTINEL, np.uint8))
        want = np.full(case.dst_alloc, SENTINEL, np.uint8)
        want[case.dst_ptr + do:case.dst_ptr + do + ln] = enc
        mb.cycle_device(src.ptr + case.src_ptr, dst.ptr + case.dst_ptr, ln, key)
        sync()
        assert (dst.download() == want).all(), cell
        return

    descs = _descs(mb, case.descs)
    first = km.plan_first_tiles(case.descs, case.dst_align)
    plan = mb.Plan(descs, case.src_bytes, case.dst_bytes, dst_align=case.dst_align)
    assert plan.num_tiles == first[-1]
    for e in range(len(case.descs)):
        assert plan.tile_range(e, e + 1) == (first[e], first[e + 1]), e
    src = _buffer(src_np)
    if case.kind == "window":
        t0, t1, ws_ptr, ws_off, ws_bytes, wd_ptr, wd_off, wd_bytes = case.win
        win_np = np.zeros(ws_ptr + ws_bytes, np.uint8)
        win_np[ws_ptr:] = src_np[case.src_ptr + ws_off:case.src_ptr + ws_off + ws_bytes]
        so, do, ln, key = case.descs[case.target]
        want = np.full(wd_ptr + wd_bytes + 16, SENTINEL, np.uint8)
        oracle.cycle_batch(_descs(mb, [(so - ws_off, do - wd_off, ln, key)]), win_np[ws_ptr:], want[wd_ptr:])
        s_win = _buffer(win_np)
        d_win = _buffer(np.full(want.size, SENTINEL, np.uint8))
        plan.run_window(t0, t1, s_win.ptr + ws_ptr, ws_off, ws_bytes, d_win.ptr + wd_ptr, wd_off, wd_bytes)
        sync()
        assert (d_win.download() == want).all(), cell
        plan.close()
        return
    want = np.full(case.dst_alloc, SENTINEL, np.uint8)
    oracle.cycle_batch(descs, src_np[case.src_ptr:], want[case.dst_ptr:])
    dst = _buffer(np.full(case.dst_alloc, SENTINEL, np.uint8))
    plan.run(src.ptr + case.src_ptr, dst.ptr + case.dst_ptr)
    sync()
    assert (dst.download() == want).all(), cell
    plan.close()
    # the same descriptors through mod_cycle_batch on device pointers (plans with dst_align = dst & 15)
    dst.upload(np.full(case.dst_alloc, SENTINEL, np.uint8))
    mb.cycle_batch(descs, src.ptr + case.src_ptr, dst.ptr + case.dst_ptr, case.src_bytes, case.dst_bytes)
    assert (dst.download() == want).all(), cell

