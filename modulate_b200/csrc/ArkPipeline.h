// ArkPipeline.h -- the slot-ring pipeline both directions of the CArk facade stream through:
// ExtractFiles (part files -> GPU gather + Cycle -> extracted files) and SaveArk (input files ->
// GPU Cycle -> part files).
//
// The pieces are cut into groups of about MOD_IO_GROUP_MIB; each group travels through one slot of a
// ring (pinned host buffers, HBM windows and a stream, on every GPU in use):
//   * reader threads run the FILL stage's tasks of the group into the slot's pinned input buffer;
//   * the calling thread only ENQUEUES, per group and never waiting: upload of the group's source range,
//     the batched kernel over the group's tiles of the archive-wide plan (mod_plan_run_window), download
//     -- on the slot's own stream, slots (and GPUs) taking groups in turn;
//   * writer threads wait for the slot's stream and run the DRAIN stage's tasks, then hand the slot back.
// Disk reads, PCIe both ways, the kernel and disk writes all overlap; pinned memory and HBM are
// O(slots), not O(archive).  The two directions differ only in their fill and drain stages.
#pragma once

#include <cstdint>
#include <functional>
#include <vector>

#include "../../include/modulate_b200.h"
#include "Error.h"

namespace arkpipe {

// Tracing aid: reports a pipeline operation that took longer than 50 ms (MOD_TRACE=1).
struct SlowOp {
    const char* mpWhat;
    double mdStart;
    explicit SlowOp(const char* lpWhat);
    ~SlowOp();
};

int HostThreads();

// Group size G: MOD_IO_GROUP_MIB, 32 MiB by default.
uint64_t GroupBytes();

// A stretch of one entry.  Entries larger than a group travel in pieces, each continuing the entry's
// keystream from the jumped key, so that a slot never has to hold more than about one group.
struct Piece {
    uint32_t file;        // index into the file table
    uint64_t fileOffset;  // where in the entry the piece starts
    uint32_t size;
};

// Append the pieces of an entry of luSize bytes that lies at luSrc in the source and at luDst in the
// destination, ciphered with liKey from its first byte: whole when luSize <= 1.5 G, else pieces of G
// with no tail shorter than G / 2.  One descriptor per piece goes to laDescs.
void CutEntry(uint32_t luFile, uint64_t luSize, uint64_t luSrc, uint64_t luDst, int32_t liKey, uint64_t luGroupBytes,
              std::vector<Piece>& laPieces, std::vector<mod_desc>& laDescs);

struct Group {
    size_t first, last;     // positions in the piece / descriptor lists
    uint64_t srcLo, srcHi;  // source range of the group's non-empty pieces (0, 0 if there are none)
    uint64_t dstLo, dstHi;  // destination range
};

// Consecutive pieces, added to a group until its destination span reaches luGroupBytes (at least one each).
std::vector<Group> GroupPieces(const std::vector<mod_desc>& laDescs, uint64_t luGroupBytes);

// A fill or drain stage: how many tasks group g has, and task t of group g.  The fill stage gets the
// slot's input buffer at the group's srcLo (the range keeps its offset & 15 phase, like on the device);
// the drain stage gets the group's output bytes at its dstLo.  A task reports failure as an eError.
struct Stage {
    std::function<int(size_t liGroup)> mTasks;
    std::function<eError(size_t liGroup, int liTask, unsigned char* lpBytes)> mRun;
};

// Run the groups through the slot ring: lpName ("extract", "build") names the pipeline in messages and
// in the MOD_TRACE summary.  With lbUseGpu every group with a non-empty destination goes through the GPU
// (one plan over laDescs, luSrcBytes / luDstBytes, per device: every visible GPU once luDstBytes reaches
// 256 MiB, MOD_DEVICES = bit mask restricting them, else the calling thread's); without it no device
// memory is allocated and the drain stage gets the bytes the fill stage read.  liReaders /
// liWriters are the default pool sizes (MOD_IO_READERS / MOD_IO_WRITERS override them).  Returns the
// first error of any stage, or eError_NoData after reporting that the GPU could not be set up.  Every
// queued task has finished when it returns.
eError RunPipeline(const char* lpName, const std::vector<mod_desc>& laDescs, const std::vector<Group>& laGroups,
                   uint64_t luSrcBytes, uint64_t luDstBytes, bool lbUseGpu, int liReaders, int liWriters, const Stage& lFill,
                   const Stage& lDrain);

}  // namespace arkpipe
