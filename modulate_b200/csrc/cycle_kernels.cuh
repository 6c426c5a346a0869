// cycle_kernels.cuh -- launch interface of the sm_100a keystream kernels (see cycle_kernels.cu).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace modk {

// Geometry of the work decomposition.  A "chunk" is one 16-byte, 16-byte-aligned piece of the
// DESTINATION address space; a "tile" is what one CTA processes before it retires: kUnroll rounds
// of kThreadsPerCta consecutive chunks, i.e. one contiguous 8 KiB span of one entry with the defaults.
#ifndef MODK_THREADS
#define MODK_THREADS 128
#endif
#ifndef MODK_UNROLL
#define MODK_UNROLL 4
#endif
constexpr int kThreadsPerCta = MODK_THREADS;
constexpr int kUnroll = MODK_UNROLL;                       // chunks in flight per thread
constexpr int kChunksPerTile = kThreadsPerCta * kUnroll;   // 512 chunks
constexpr uint32_t kTileBytes = 16u * kChunksPerTile;      // 8 KiB of destination per tile
constexpr int kMaxInlineDescs = 64;  // descriptors that travel in the kernel parameter block
static_assert(kChunksPerTile <= 2048, "TileRec::geom holds the chunk count in 12 bits");

// Device-side descriptor: mod_desc plus the index of the entry's first tile (32 bytes).
struct __align__(16) DevDesc {
    uint64_t src_off;
    uint64_t dst_off;
    uint32_t len;
    int32_t key;
    uint32_t first_tile;
    uint32_t neg_state;  // modlcg::key_to_neg_state(key), filled on the host (no division on the device)
};

// One record per tile, written once by the plan kernel and read (one 32-byte broadcast load) by
// the CTA that owns the tile: everything it needs to start streaming, so the hot kernel does no
// search, no division and no table walk.
struct __align__(16) TileRec {
    int64_t src_rel;   // source byte (relative to the src base) that pairs with byte 0 of the tile's chunk 0
    int64_t dst_rel;   // destination byte (relative to the dst base) of chunk 0; base + dst_rel is 16-byte aligned
    uint32_t state;    // negated LCG state just before byte 0 of chunk 0
    uint32_t geom;     // bits 0-11: chunks in the tile; 12-15: first valid byte of chunk 0; 16-20: valid bytes of the last chunk
    uint32_t entry;    // descriptor index (the search kernel's counts and matches)
    uint32_t rest;     // bytes of the entry after this tile: bounds the search kernel's halo
};

__host__ __device__ inline uint32_t pack_geom(uint32_t n_valid, uint32_t head, uint32_t tail)
{
    return n_valid | (head << 12) | (tail << 16);
}

struct InlineDescs {
    DevDesc d[kMaxInlineDescs];
};

struct BatchArgs {
    const uint8_t* src;
    uint8_t* dst;
    const TileRec* tiles;  // HBM tile records (nullptr in inline mode)
    uint32_t n_tiles;
    uint32_t tiles_per_entry;  // inline mode: entry = tile / tiles_per_entry
    // 16-byte granules of the source may be loaded whole only inside [src_lo16, src_hi16).
    uint64_t src_lo16;
    uint64_t src_hi16;
    uint32_t two = 2;  // the literal 2, kept opaque to ptxas (see low8_canonical_fma)
    // (src_off - dst_off) & 15 if it is the same for every entry of the launch, else -1: together with
    // the base pointers it tells the host whether the co-aligned kernel may be used
    int32_t uniform_delta = -1;
};

// Search launch (find_batch_kernel): one CTA per tile of a plan whose chunk grid is co-aligned with the
// source (built with dst_off == src_off and dst_align == source address & 15), nothing stored.
constexpr uint32_t kMaxPattern = 64;
constexpr int kHaloChunks = (int)((kMaxPattern - 1 + 15) / 16);  // chunks past a tile a match may reach into
struct FindArgs {
    const uint8_t* src;    // virtual base: src + TileRec::src_rel is 16-byte aligned
    const TileRec* tiles;
    const DevDesc* descs;  // the plan's descriptors: a match's position is relative to its entry's src_off
    uint32_t n_tiles;
    uint64_t src_lo16, src_hi16;  // as in BatchArgs
    uint32_t* counts;             // per descriptor, accumulated
    uint2* matches;               // {descriptor, position}: slots [0, cap) of the list
    unsigned long long* total;    // accumulated; also hands out list slots
    uint64_t cap;
    uint32_t len;        // pattern bytes, 1..kMaxPattern
    uint32_t head_word;  // first min(4, len) pattern bytes, little-endian
    uint32_t head_mask;  // which bytes of head_word take part (masked search: its first four mask bytes)
    uint32_t rep0, rep1; // pattern[a] and pattern[a + 1] (0 if len == 1) in every byte: the search filter
    uint32_t two = 2;
    uint8_t pattern[kMaxPattern];
    // Masked search only (find_batch_kernel<true>): byte t matches pattern byte k when ((t ^ pattern[k]) & mask[k])
    // == 0, pattern[k] already AND-ed with mask[k].  The filter tests the anchor pair (a, a + 1), the adjacent pair
    // with the most mask bits; the exact kernel's anchor is a = 0 and it reads none of these fields.
    uint32_t anchor;             // a
    uint32_t mrep0, mrep1;       // mask[a] and mask[a + 1] (0 if len == 1) in every byte
    uint8_t mask[kMaxPattern];
};

// Pattern-set search (find_set_kernel): the decipher stage of find_batch_kernel, then every start tested against
// an exact 2-byte filter and the candidates verified against the set.  The index is built on the host
// (mod_pattern_set_create) and lives in HBM; callers never see it.
constexpr uint32_t kMaxSetPatterns = 256;
struct __align__(16) SetPattern {  // read as one 16-byte load
    uint32_t id;    // position in the caller's list
    uint32_t len;
    uint32_t head;  // first min(4, len) bytes, little-endian
    uint32_t mask;  // which bytes of head take part
};
// A case-folded set (mod_pattern_set_create_nocase) holds upper-cased keys, bytes and length-1 entries, and its
// bitmap has a bit for every case variant of a pattern's first two bytes.
__host__ __device__ inline uint32_t fold_ascii(uint32_t b) { return b - 0x61u < 26u ? b - 0x20u : b; }
struct SetIndex {  // ~30 KB, one cudaMalloc
    uint32_t bitmap[65536 / 32];          // bit b0 | b1 << 8: some pattern starts with (b0, b1); length 1 sets (b0, *)
    uint16_t keys[kMaxSetPatterns];       // distinct 2-byte keys of the patterns of length >= 2, ascending
    uint16_t one[256];                    // 1 + id of the length-1 pattern b0, or 0
    uint16_t group[kMaxSetPatterns + 1];  // CSR: patterns [group[g], group[g + 1]) have keys[g]
    SetPattern pat[kMaxSetPatterns];      // patterns of length >= 2, sorted by key
    uint8_t bytes[kMaxSetPatterns][kMaxPattern];  // pat[r]'s bytes
};
static_assert(offsetof(SetIndex, pat) % 16 == 0 && offsetof(SetIndex, bitmap) == 0, "SetIndex: 16-byte loads");
struct FindSetArgs {
    const uint8_t* src;
    const TileRec* tiles;
    const DevDesc* descs;
    uint32_t n_tiles;
    uint64_t src_lo16, src_hi16;
    const SetIndex* set;
    uint32_t n_keys;                   // distinct keys of length >= 2
    uint32_t lmin, lmax;
    const uint32_t* owned;             // per descriptor: starts >= owned[i] are not reported (nullptr: all are)
    uint32_t* counts;                  // per descriptor, accumulated
    unsigned long long* pattern_counts;  // per pattern, accumulated
    uint32_t* matches;                 // {descriptor, position, pattern}: slots [0, cap) of the list
    unsigned long long* total;
    uint64_t cap;
    uint32_t two = 2;
};

// Number of tiles an entry of `len` bytes occupies when its first destination byte sits at
// (address & 15) == h0.
__host__ __device__ inline uint32_t tiles_for_entry(uint32_t h0, uint32_t len)
{
    if (len == 0)
        return 0;
    const uint64_t chunks = ((uint64_t)h0 + len + 15u) >> 4;
    return (uint32_t)((chunks + (uint32_t)kChunksPerTile - 1) / (uint32_t)kChunksPerTile);
}

cudaError_t upload_tables();  // jump tables -> __constant__ / global memory of the current device
cudaError_t launch_batch(const BatchArgs& args, cudaStream_t stream);
cudaError_t launch_batch_inline(const BatchArgs& args, const InlineDescs& descs, cudaStream_t stream);
// `masked`: find_batch_kernel<true> (FindArgs' mask fields); `fold`: find_set_kernel<true> (a case-folded set).
cudaError_t launch_find(const FindArgs& args, bool masked, cudaStream_t stream);
cudaError_t launch_find_set(const FindSetArgs& args, bool fold, cudaStream_t stream);
// Plan kernel: expands descriptors into per-tile records (binary search + jump-ahead per tile).
cudaError_t launch_build_tiles(const DevDesc* descs, uint32_t n_descs, uint32_t dst_align, TileRec* tiles,
                               uint32_t n_tiles, cudaStream_t stream);

}  // namespace modk
