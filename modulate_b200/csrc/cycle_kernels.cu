// cycle_kernels.cu -- hand-written sm_100a kernels for the Modulate keystream path.
//
// What the kernel computes (per descriptor {src_off, dst_off, len, key}):
//     dst[dst_off + i] = src[src_off + i] ^ low8(k0 * a^(i+1) mod m) ^ 0xFF,   0 <= i < len
// which is CEncryptionCycler::Cycle (reference CEncryptionCycler.cpp:4-14) applied to a copy of
// the entry -- the copy being CArk::ExtractFiles' gather (CArk.cpp:494) or CArk::BuildArk's
// scatter (CArk.cpp:807-811).  One variable-length batched kernel serves every caller; a
// contiguous Cycle() is the same kernel with a few descriptors passed in the parameter block.
//
// Decomposition (B200: HBM-bound byte work, co-limited by the integer pipes -- no tensor cores):
//   * destination space is cut into 16-byte aligned chunks and 8 KiB tiles (512 chunks of ONE entry);
//   * ONE CTA PER TILE, NO LOOP: the 128 threads of a CTA each take 4 chunks 2 KiB apart, issue all
//     their 128-bit loads at once, generate the keystream, store, and the CTA RETIRES.  CTAs are
//     scheduled in tile order, so GPU-wide the bytes in flight form one window that slides linearly
//     through the image -- the access pattern of the fastest plain copy on this part (6.8 TB/s,
//     profiles/r01_copy_skeleton_bench.txt pattern B), where round 1's persistent warp-strided tiles
//     topped out at 6.1 TB/s (profiles/r02_kernel.md has the A/B);
//   * the serial recurrence is broken by modular jump-ahead: the tile record carries the state just
//     before the tile's first chunk, each thread multiplies it by a^(16*chunk) from a 2 KiB table, and
//     inside a chunk the state is stepped 16 times with a lazily reduced Mersenne fold (IMAD.WIDE +
//     one add).  The chains of a thread's 4 chunks are generated as one basic block so they
//     interleave (ILP 4).  Low bytes are packed straight from the lazy states; the same PRMT that
//     packs them also gathers the states' top bytes, one LOP3 per 4 bytes accumulates those, and a
//     chunk is redone exactly only if one of its states had bit 31 set (~2^-17 per byte);
//   * entries are byte-packed (BuildArk leaves no padding), so source and destination are
//     generally misaligned with respect to each other: the source is read as aligned 16-byte
//     granules (each thread takes the two granules its chunk straddles; the second is an L1 hit on
//     its neighbour's first) and a funnel shift re-aligns them, the word part of the shift being
//     a template parameter so no register-select network is needed;
//   * the first / last chunk of an entry are partial: they go through the same loads and the same
//     keystream and differ only in the store (aligned 4-byte and single-byte stores of the bytes that
//     belong to the entry).  Only tiles whose granules would leave the source buffer (the first / last
//     16 bytes of the image) take a byte-granular path.
// Round 1's persistent grid, register ping-pong, bulk-async (cp.async.bulk + mbarrier) staging ring
// and L2 prefetch variants are in the git history; their numbers are in profiles/r01_tuning.md.
#include "cycle_kernels.cuh"
#include "lcg.h"

#include <algorithm>
#include <cstdlib>

namespace modk {

using modlcg::mulmod;
using modlcg::step_lazy;
using modlcg::low8_canonical;

// ---- tuning knobs (defaults chosen from the measurements in profiles/) ------------------------------
#ifndef MODK_CANON_FMA_MASK
#define MODK_CANON_FMA_MASK 0x5  // exact path: which of every 4 bytes canonicalise on the FMA pipe (IMAD.HI) vs ALU (LEA.HI)
#endif
#ifndef MODK_MIN_CTAS
#define MODK_MIN_CTAS 10         // GENERAL kernels (any source alignment): resident CTAs per SM (48 registers)
#endif
#ifndef MODK_MIN_CTAS_INLINE
#define MODK_MIN_CTAS_INLINE 8   // general CONTIGUOUS kernel (out-of-place Cycle between misaligned buffers): it also computes its
                                 // tile record, which does not fit 48 registers without spilling
#endif
#ifndef MODK_MIN_CTAS_COAL
#define MODK_MIN_CTAS_COAL 10    // CO-ALIGNED kernels (source and destination agree mod 16, e.g. in place): 48 registers
#endif
#ifndef MODK_STAGE
#define MODK_STAGE 1             // general kernels: 1 = the tile's source span is staged through shared memory by ONE
                                 // bulk-async copy per CTA (cp.async.bulk + mbarrier), 0 = two LDG.128 per chunk into registers
#endif
#ifndef MODK_EDGE_ROUNDS
#define MODK_EDGE_ROUNDS 1       // co-aligned kernels: a partly filled tile runs only the rounds (of 128 chunks) that hold chunks
#endif
#ifndef MODK_STAGE_SEQ
#define MODK_STAGE_SEQ 1         // general kernels: read the staged granules chunk by chunk inside the store loop: 8 registers of
                                 // granules live instead of 32, which is what lets them run at 10 CTAs/SM without spilling
#endif
#ifndef MODK_GENERAL_FULL
#define MODK_GENERAL_FULL 1      // general kernels: separate predicate-free code for interior tiles (doubles their code size)
#endif
#ifndef MODK_HOIST_POW
#define MODK_HOIST_POW 1         // batched kernel: request the jump factors before the tile record arrives
#endif
#ifndef MODK_REC_PREFETCH
#define MODK_REC_PREFETCH 2048   // batched kernel: L2 prefetch distance for tile records, in tiles (0 = off)
#endif

// tile index within an entry < 2^32 / kTileBytes + 1; split 10 bits low / rest high
constexpr int kTw0Size = 1024;
constexpr int kTw1Size = (int)(((1ull << 32) / kTileBytes) / kTw0Size + 2);

__constant__ uint32_t c_tw0[kTw0Size];  // a^(kTileBytes * j)
__constant__ uint32_t c_tw1[kTw1Size];  // a^(kTileBytes * 1024 * j)
__constant__ uint32_t c_ainv[16];       // a^(-h): rewinds the stream to the chunk grid origin
__device__ uint32_t g_chunk_pow2[kChunksPerTile];  // 2 * a^(16 * j), PRE-DOUBLED for the multiply (see jump_lazy); the index
                                                   // is thread-divergent, so the table lives in L1 rather than the constant bank

// st * a^(16 j) for a canonical st and y2 = 2 * a^(16 j) from g_chunk_pow2, LAZILY reduced: one IMAD.WIDE and one
// add, no canonical fold.  The result can be anything below 2^32; that is fine for the first step of a chain
// (step_lazy is exact for every 32-bit input: the product of s and 2a is even, so hi + (lo >> 1) == s*a mod m)
// and no output byte is ever taken from it.
__device__ __forceinline__ uint32_t jump_lazy(uint32_t st, uint32_t y2)
{
    const uint64_t p = (uint64_t)st * (uint64_t)y2;
    return (uint32_t)(p >> 32) + ((uint32_t)p >> 1);
}

// ---- 128-bit global accesses (explicit state space: the addresses are rebuilt from integers) ------

__device__ __forceinline__ uint4 ldg128(uint64_t addr)
{
    uint4 r;
    asm volatile("ld.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(addr));
    return r;
}

__device__ __forceinline__ void stg128(uint64_t addr, const uint4& v)
{
    asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}

#if MODK_STAGE
// ---- bulk-async staging: mbarrier + cp.async.bulk (SASS: UBLKCP / SYNCS) --------------------------------

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MODK_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MODK_DONE;\n"
        "bra MODK_WAIT;\n"
        "MODK_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}

// global -> shared bulk copy of `bytes` (multiple of 16, both addresses 16-byte aligned); completion
// is signalled on the mbarrier as transaction bytes
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, uint64_t src_gmem, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src_gmem), "r"(bytes), "r"(bar)
                 : "memory");
}

__device__ __forceinline__ uint4 lds128(uint32_t addr)
{
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
    return r;
}
#endif

// ---- per-chunk arithmetic -------------------------------------------------------------------

// low8_canonical on the FMA pipe: hi32(s * 2) + s == (s >> 31) + s.  `two` is the constant 2
// delivered through the kernel parameter block: with a literal, ptxas strength-reduces the
// multiply back into an ALU-pipe LEA.HI.
__device__ __forceinline__ uint32_t low8_canonical_fma(uint32_t s, uint32_t two)
{
    uint32_t r;
    asm("mad.hi.u32 %0, %1, %2, %1;" : "=r"(r) : "r"(s), "r"(two));
    return r;
}

// XOR the 16 bytes of `d` with the keystream that follows (negated) state `s`, the state just
// before the chunk's first byte -- exact for every state.  Per byte: IMAD.WIDE + LEA.HI (step) and
// a canonical low byte (LEA.HI on the ALU pipe or IMAD.HI on the FMA pipe, per MODK_CANON_FMA_MASK);
// per word: three PRMTs pack four keystream bytes and one LOP3 applies them.  Out of line: used for
// the ~1 chunk in 14 000 the speculative hot loop hands over, and by the byte-granular slow path.
__device__ __noinline__ uint4 cycle_chunk_exact(uint4 d, uint32_t s, const uint32_t two)
{
    uint32_t w[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        s = step_lazy(s);
        const uint32_t b0 = (MODK_CANON_FMA_MASK & 1) ? low8_canonical_fma(s, two) : low8_canonical(s);
        s = step_lazy(s);
        const uint32_t b1 = (MODK_CANON_FMA_MASK & 2) ? low8_canonical_fma(s, two) : low8_canonical(s);
        s = step_lazy(s);
        const uint32_t b2 = (MODK_CANON_FMA_MASK & 4) ? low8_canonical_fma(s, two) : low8_canonical(s);
        s = step_lazy(s);
        const uint32_t b3 = (MODK_CANON_FMA_MASK & 8) ? low8_canonical_fma(s, two) : low8_canonical(s);
        const uint32_t lo = __byte_perm(b0, b1, 0x0040);
        const uint32_t hi = __byte_perm(b2, b3, 0x0040);
        w[j] ^= __byte_perm(lo, hi, 0x5410);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// ---- partial chunks and the byte-granular slow path -------------------------------------------------

// Store bytes [lo, hi) of the 16-byte value `v` at the 16-byte aligned address `addr`: aligned words
// that lie wholly inside the range go out as one 4-byte store, the (at most six) others byte by byte.
// Out of line -- at most two chunks per entry come here.
__device__ __noinline__ void store_partial(uint64_t addr, uint4 v, uint32_t lo, uint32_t hi)
{
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (uint32_t k = 0; k < 4; ++k) {
        const uint32_t b0 = 4u * k;
        if (lo <= b0 && b0 + 4u <= hi) {
            asm volatile("st.global.u32 [%0], %1;" ::"l"(addr + b0), "r"(w[k]));
        } else {
#pragma unroll
            for (uint32_t b = b0; b < b0 + 4u; ++b)
                if (b >= lo && b < hi)
                    asm volatile("st.global.u8 [%0], %1;" ::"l"(addr + b), "r"((w[k] >> (8u * (b - b0))) & 0xFFu));
        }
    }
}

// One chunk without any whole-granule source access: only the source bytes that belong to the
// entry are touched.  For the tiles at the very ends of the source buffer.
__device__ __noinline__ void slow_chunk(uint64_t src_byte0, uint64_t dst_chunk, uint32_t lo, uint32_t hi, uint32_t s,
                                        uint32_t two)
{
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (uint32_t b = 0; b < 16; ++b) {
        if (b >= lo && b < hi) {
            uint32_t byte;
            asm volatile("ld.global.u8 %0, [%1];" : "=r"(byte) : "l"(src_byte0 + b));
            w[b >> 2] |= byte << (8u * (b & 3u));
        }
    }
    store_partial(dst_chunk, cycle_chunk_exact(make_uint4(w[0], w[1], w[2], w[3]), s, two), lo, hi);
}

// ---- one tile = one CTA ----------------------------------------------------------------------------

// Thread `idx0`'s share of a tile: chunks idx0 + u * kThreadsPerCta, u < U.  Every load is issued
// before anything consumes one; the U keystream chunks are generated as ONE basic block so that the
// independent 16-step chains interleave.
// kWs < 0: source and destination are co-aligned (one load per chunk).  kWs in 0..3: the chunk
// starts kWs words (+ `bs` / 8 bytes) into its first granule and straddles two.
// kStaged: the tile's source span has been requested into shared memory by one bulk-async copy
// (issued by thread 0 in run_tile); the granules are read from there AFTER the keystream has been
// generated, so no register holds a load in flight; they are read chunk by chunk inside the store loop
// (MODK_STAGE_SEQ), shared memory being close enough that nothing is gained by batching the reads.
// kFull: the tile is a whole 512 chunks and none of them is partial (every tile of a big entry but its first
// and last): no per-chunk predicates on loads or stores at all.
template <int kWs, int U, bool kStaged, bool kFull = false>
__device__ __forceinline__ void process_tile(const uint64_t src_tile, const uint64_t dst_tile, const uint32_t st,
                                             const uint32_t n_valid, const uint32_t head, const uint32_t tail,
                                             const uint32_t bs, const uint32_t idx0, const uint32_t (&pw)[U],
                                             const uint32_t two, const uint32_t stage, const uint32_t bar)
{
    constexpr uint32_t T = (uint32_t)kThreadsPerCta;
    uint4 own[U], nxt[U];
    const uint64_t sp = src_tile + 16ull * idx0;
    if (!kStaged) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            own[u] = make_uint4(0u, 0u, 0u, 0u);
            nxt[u] = make_uint4(0u, 0u, 0u, 0u);
            if (kFull || idx0 + (uint32_t)u * T < n_valid) {
                own[u] = ldg128(sp + 16ull * T * u);
                if (kWs >= 0)
                    nxt[u] = ldg128(sp + 16ull * T * u + 16ull);
            }
        }
    }

    uint32_t s[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
        s[u] = jump_lazy(st, pw[u]);  // state just before this thread's chunk of round u

    // A lazily reduced state t = hi + lo31 (hi <= 16807) is already canonical unless bit 31 is set,
    // which needs lo31 >= 2^31 - 16807: about 2^-17 per byte.  So the low bytes are packed straight
    // from the lazy states; the first-level PRMT also carries the two states' TOP bytes in its upper
    // half, and OR-ing those words (one LOP3 per 4 bytes) tells whether any state of the group had
    // bit 31 set -- only then are the chunks redone by the exact routine.
    uint32_t ks[U][4];
    uint32_t any = 0u;
#if !defined(MODK_EXPERIMENT_COPY_ONLY)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t b0 = step_lazy(s[u]);
            const uint32_t b1 = step_lazy(b0);
            const uint32_t b2 = step_lazy(b1);
            const uint32_t b3 = step_lazy(b2);
            s[u] = b3;
            const uint32_t lo = __byte_perm(b0, b1, 0x7340);  // {b0.0, b1.0, b0.3, b1.3}
            const uint32_t hi = __byte_perm(b2, b3, 0x7340);
            any |= lo | hi;
            ks[u][j] = __byte_perm(lo, hi, 0x5410);
        }
    }
#else
    // measurement aid (never shipped): no keystream at all -> the memory-system ceiling of this skeleton
#pragma unroll
    for (int u = 0; u < U; ++u)
        ks[u][0] = ks[u][1] = ks[u][2] = ks[u][3] = s[u] & two;
#endif
    const bool redo = (any & 0x80800000u) != 0u;

#if MODK_STAGE
    auto load_staged = [&](const int u) {  // chunk u's granules out of the shared-memory stage
        own[u] = make_uint4(0u, 0u, 0u, 0u);
        nxt[u] = make_uint4(0u, 0u, 0u, 0u);
        if (kFull || idx0 + (uint32_t)u * T < n_valid) {
            own[u] = lds128(stage + 16u * (idx0 + (uint32_t)u * T));
            if (kWs >= 0)
                nxt[u] = lds128(stage + 16u * (idx0 + (uint32_t)u * T) + 16u);
        }
    };
    if (kStaged) {
        mbar_wait(bar, 0u);  // the CTA's only use of the barrier: phase 0
#if !MODK_STAGE_SEQ
#pragma unroll
        for (int u = 0; u < U; ++u)
            load_staged(u);
#endif
    }
#else
    auto load_staged = [&](const int) {};
#endif

    const uint32_t f_lo = head ? 1u : 0u;
    const uint32_t f_hi = max(n_valid - (tail < 16u ? 1u : 0u), f_lo);
    const uint64_t dp = dst_tile + 16ull * idx0;
    auto source = [&](const int u) {  // the 16 source bytes that pair with chunk u, re-aligned
        uint4 data = own[u];
        if (kWs >= 0) {
            const uint32_t w[8] = {own[u].x, own[u].y, own[u].z, own[u].w, nxt[u].x, nxt[u].y, nxt[u].z, nxt[u].w};
            constexpr int k = kWs < 0 ? 0 : kWs;
            data.x = __funnelshift_r(w[k + 0], w[k + 1], bs);
            data.y = __funnelshift_r(w[k + 1], w[k + 2], bs);
            data.z = __funnelshift_r(w[k + 2], w[k + 3], bs);
            data.w = __funnelshift_r(w[k + 3], w[k + 4], bs);
        }
        return data;
    };
    auto emit = [&](const int u, const uint4& out) {
        const uint32_t idx = idx0 + (uint32_t)u * T;
        if (kFull || idx - f_lo < f_hi - f_lo)
            stg128(dp + 16ull * T * u, out);
        else if (idx < n_valid)
            store_partial(dp + 16ull * T * u, out, idx == 0u ? head : 0u, idx + 1u == n_valid ? tail : 16u);
    };
    if (__builtin_expect(redo, 0)) {
#if MODK_STAGE_SEQ
        if (kStaged) {
#pragma unroll
            for (int u = 0; u < U; ++u)
                load_staged(u);
        }
#endif
        // some state of this thread's chunks needed a canonical subtract (~1 thread in 3 600): redo all four
        // exactly, from start states recomputed here (nothing is kept live for this path)
#pragma unroll 1
        for (int u = 0; u < U; ++u) {
            const uint32_t idx = idx0 + (uint32_t)u * T;
            uint4 data = own[0];
#pragma unroll
            for (int v = 0; v < U; ++v)
                if (v == u)
                    data = source(v);
            const uint4 out = cycle_chunk_exact(data, jump_lazy(st, __ldg(&g_chunk_pow2[idx])), two);
#pragma unroll
            for (int v = 0; v < U; ++v)
                if (v == u)
                    emit(v, out);
        }
        return;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#if MODK_STAGE_SEQ
        if (kStaged)
            load_staged(u);  // one chunk at a time: 8 registers of granules live instead of 32
#endif
        const uint4 data = source(u);
        emit(u, make_uint4(data.x ^ ks[u][0], data.y ^ ks[u][1], data.z ^ ks[u][2], data.w ^ ks[u][3]));
    }
}

// kGeneral = false: the launch guarantees that source and destination agree mod 16 (in-place runs, co-aligned
// copies): one LDG.128 per chunk straight into registers, no re-alignment code in the kernel at all.
// kGeneral = true: any alignment; the tile's source span comes through shared memory (MODK_STAGE) or as two
// LDG.128 per chunk, and a funnel shift re-aligns it.
template <int U, bool kGeneral>
__device__ __forceinline__ void run_tile(const BatchArgs& a, const int64_t src_rel, const int64_t dst_rel,
                                         const uint32_t st, const uint32_t geom, const uint32_t idx0,
                                         const uint32_t (&pw)[U], const uint32_t stage, const uint32_t bar)
{
    const uint64_t dst_tile = (uint64_t)a.dst + (uint64_t)dst_rel;
    const uint64_t sv = (uint64_t)a.src + (uint64_t)src_rel;  // source address that pairs with chunk 0, byte 0
    const uint32_t shift = (uint32_t)sv & 15u;
    const uint64_t src_tile = sv - shift;
    constexpr uint32_t kFullGeom = (uint32_t)kChunksPerTile | (16u << 16);  // pack_geom(kChunksPerTile, 0, 16)
    if (!kGeneral && geom == kFullGeom && shift == 0u && src_tile >= a.src_lo16 && src_tile + kTileBytes <= a.src_hi16) {
        // CTA-uniform fast exit of the co-aligned flavour: an interior tile of a big entry, nothing to decode
        process_tile<-1, U, false, true>(src_tile, dst_tile, st, (uint32_t)kChunksPerTile, 0u, 16u, 0u, idx0, pw, a.two, stage, bar);
        return;
    }
    const uint32_t n_valid = geom & 0xFFFu, head = (geom >> 12) & 15u, tail = (geom >> 16) & 31u;

    // whole-granule loads are allowed only inside the source buffer (CTA-uniform test); a misaligned
    // tile in a co-aligned launch (the host never produces one) also lands here and stays correct
    const uint64_t src_end = src_tile + 16ull * (n_valid + (shift ? 1u : 0u));
    if (__builtin_expect(src_tile < a.src_lo16 || src_end > a.src_hi16 || (!kGeneral && shift != 0u), 0)) {
#pragma unroll 1
        for (int u = 0; u < U; ++u) {
            const uint32_t idx = idx0 + (uint32_t)u * (uint32_t)kThreadsPerCta;
            if (idx < n_valid)
                slow_chunk(sv + 16ull * idx, dst_tile + 16ull * idx, idx == 0u ? head : 0u,
                           idx + 1u == n_valid ? tail : 16u, jump_lazy(st, g_chunk_pow2[idx]), a.two);
        }
        return;
    }

    const uint32_t bs = (shift & 3u) * 8u;
    if (!kGeneral) {
#if MODK_EDGE_ROUNDS
        // A partly filled tile (the last tile of an entry, every tile of a small one) only runs the rounds that
        // hold chunks (CTA-uniform): with many small entries about half of every last tile is empty, and a
        // keystream generated for chunks that do not exist is instructions and power for nothing.
        if (U == 4 && n_valid <= 3u * (uint32_t)kThreadsPerCta) {
            if (n_valid <= (uint32_t)kThreadsPerCta) {
                const uint32_t p1[1] = {pw[0]};
                process_tile<-1, 1, false, false>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, p1, a.two, stage, bar);
            } else if (n_valid <= 2u * (uint32_t)kThreadsPerCta) {
                const uint32_t p2[2] = {pw[0], pw[1]};
                process_tile<-1, 2, false, false>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, p2, a.two, stage, bar);
            } else {
                const uint32_t p3[3] = {pw[0], pw[1], pw[2]};
                process_tile<-1, 3, false, false>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, p3, a.two, stage, bar);
            }
            return;
        }
#endif
        process_tile<-1, U, false, false>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar);
        return;
    }
    constexpr bool kStaged = MODK_STAGE != 0;
#if MODK_STAGE
    if (threadIdx.x == 0) {  // one bulk-async copy brings the tile's whole source span into shared memory
        const uint32_t bytes = 16u * (n_valid + (shift ? 1u : 0u));
        mbar_expect_tx(bar, bytes);
        bulk_g2s(stage, src_tile, bytes, bar);
    }
#endif
#if MODK_GENERAL_FULL
    if (geom == kFullGeom) {  // CTA-uniform: an interior tile of a big entry -- no per-chunk predicates
        switch (shift ? (int)(shift >> 2) : -1) {
        case -1: process_tile<-1, U, kStaged, true>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        case 0: process_tile<0, U, kStaged, true>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        case 1: process_tile<1, U, kStaged, true>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        case 2: process_tile<2, U, kStaged, true>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        default: process_tile<3, U, kStaged, true>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        }
        return;
    }
#endif
    if (shift == 0u) {
        process_tile<-1, U, kStaged>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar);
    } else {
        switch (shift >> 2) {
        case 0: process_tile<0, U, kStaged>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        case 1: process_tile<1, U, kStaged>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        case 2: process_tile<2, U, kStaged>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        default: process_tile<3, U, kStaged>(src_tile, dst_tile, st, n_valid, head, tail, bs, idx0, pw, a.two, stage, bar); break;
        }
    }
}

// (negated) state just before byte (kTileBytes * tin - h0) of an entry whose negated start state is n0:
//   n0 * a^(-h0) * a^(kTileBytes * tin)
__device__ __forceinline__ uint32_t tile_start_state(uint32_t n0, uint32_t h0, uint32_t tin)
{
    const uint32_t st = mulmod(n0, c_ainv[h0]);
    return mulmod(st, mulmod(c_tw0[tin & (uint32_t)(kTw0Size - 1)], c_tw1[tin / (uint32_t)kTw0Size]));
}

// Tile `tin` of the entry {src_off, dst_off, len}: where it starts, how many chunks it holds and
// which bytes of its first / last chunk belong to the entry.
__device__ __forceinline__ TileRec make_tile_rec(uint64_t src_off, uint64_t dst_off, uint32_t len, uint32_t n0,
                                                 uint32_t tin, uint32_t dst_align, uint32_t entry)
{
    const uint32_t h0 = (dst_align + (uint32_t)dst_off) & 15u;
    const uint64_t span = (uint64_t)h0 + len;  // bytes from the chunk grid origin to the entry end
    const uint32_t nchunks = (uint32_t)((span + 15u) >> 4);
    const uint32_t c_begin = tin * (uint32_t)kChunksPerTile;
    const uint32_t n_valid = min((uint32_t)kChunksPerTile, nchunks - c_begin);
    const bool last = c_begin + n_valid == nchunks;
    TileRec r;
    r.src_rel = (int64_t)src_off - (int64_t)h0 + 16ll * (int64_t)c_begin;
    r.dst_rel = (int64_t)dst_off - (int64_t)h0 + 16ll * (int64_t)c_begin;
    r.state = tile_start_state(n0, h0, tin);
    r.geom = pack_geom(n_valid, tin == 0u ? h0 : 0u, last ? (((uint32_t)span - 1u) & 15u) + 1u : 16u);
    r.entry = entry;
    r.rest = last ? 0u : (uint32_t)(span - 16ull * (c_begin + n_valid));
    return r;
}

// Shared-memory stage + its mbarrier (general kernels only): initialised by thread 0 while the tile
// record is still in flight; used for exactly one phase, the CTA then retires.
#if MODK_STAGE
#define MODK_STAGE_SETUP                                                                          \
    uint32_t stage = 0u, bar = 0u;                                                                \
    if (kGeneral) {                                                                               \
        __shared__ __align__(128) uint8_t s_stage[kTileBytes + 16];                               \
        __shared__ __align__(8) uint64_t s_bar;                                                   \
        stage = smem_u32(s_stage);                                                                \
        bar = smem_u32(&s_bar);                                                                   \
        if (threadIdx.x == 0)                                                                     \
            mbar_init(bar, 1u);                                                                   \
        __syncthreads();                                                                          \
    }
#else
#define MODK_STAGE_SETUP const uint32_t stage = 0u, bar = 0u;
#endif

// This thread's jump factors a^(16 * chunk): they depend on nothing but the thread index, so they are
// requested before (and fly together with) the tile record.
template <int U>
__device__ __forceinline__ void load_chunk_pows(uint32_t (&pw)[U], uint32_t idx0)
{
#pragma unroll
    for (int u = 0; u < U; ++u)
        pw[u] = __ldg(&g_chunk_pow2[idx0 + (uint32_t)u * (uint32_t)kThreadsPerCta]);
}

// Batched kernel: CTA b owns tile b (one 32-byte record, broadcast to the CTA) and retires.  A CTA
// lives for ~3 us, so the DRAM latency of its own record would be a large part of its life: every
// CTA therefore pulls the 128-byte line holding the records of the CTAs MODK_REC_PREFETCH tiles
// further on (about two waves of resident CTAs) into L2.
template <bool kGeneral>
__global__ void __launch_bounds__(kThreadsPerCta, kGeneral ? MODK_MIN_CTAS : MODK_MIN_CTAS_COAL)
cycle_batch_kernel(const BatchArgs a)
{
    MODK_STAGE_SETUP
    const uint4* p = reinterpret_cast<const uint4*>(a.tiles + blockIdx.x);
    uint32_t pw[kUnroll];
#if MODK_HOIST_POW
    load_chunk_pows<kUnroll>(pw, threadIdx.x);
#endif
    const uint4 lo = __ldg(p);
    const uint4 hi = __ldg(p + 1);
#if MODK_REC_PREFETCH
    if (threadIdx.x == 0 && a.n_tiles - blockIdx.x > (uint32_t)MODK_REC_PREFETCH) {
        const uint64_t ahead = (uint64_t)(a.tiles + blockIdx.x + MODK_REC_PREFETCH);
        if ((ahead & 127u) == 0u)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(ahead));
    }
#endif
    const int64_t src_rel = (int64_t)((uint64_t)lo.x | ((uint64_t)lo.y << 32));
    const int64_t dst_rel = (int64_t)((uint64_t)lo.z | ((uint64_t)lo.w << 32));
#if !MODK_HOIST_POW
    load_chunk_pows<kUnroll>(pw, threadIdx.x);
#endif
    run_tile<kUnroll, kGeneral>(a, src_rel, dst_rel, hi.x, hi.y, threadIdx.x, pw, stage, bar);
}

// Same kernel with the (few) descriptors in the parameter block: nothing to upload, nothing to
// allocate, so a contiguous Cycle() is a single asynchronous launch.  The tile record is computed
// from the constant-bank jump tables instead of being loaded.  (A short buffer such as the 384 KiB
// HDR is 48 CTAs that all run at once, each thread's 4 chains interleaved: one chain latency.)
template <bool kGeneral>
__global__ void __launch_bounds__(kThreadsPerCta, kGeneral ? MODK_MIN_CTAS_INLINE : MODK_MIN_CTAS_COAL)
cycle_inline_kernel(const BatchArgs a, const __grid_constant__ InlineDescs in)
{
    MODK_STAGE_SETUP
    uint32_t pw[kUnroll];
    load_chunk_pows<kUnroll>(pw, threadIdx.x);
    const uint32_t tile = blockIdx.x;
    const uint32_t e = tile / a.tiles_per_entry;
    const DevDesc& d = in.d[e];
    const TileRec r = make_tile_rec(d.src_off, d.dst_off, d.len, d.neg_state, tile - d.first_tile,
                                    (uint32_t)(uintptr_t)a.dst & 15u, e);
    run_tile<kUnroll, kGeneral>(a, r.src_rel, r.dst_rel, r.state, r.geom, threadIdx.x, pw, stage, bar);
}

// Plan kernel, one thread per tile: find the tile's entry (the last entry whose first_tile <= tile;
// entries with no tiles share their successor's first_tile and are skipped by taking the last) and
// write the tile record, jump-ahead state included.
__global__ void build_tiles_kernel(const DevDesc* __restrict__ descs, uint32_t n_descs, uint32_t dst_align,
                                   TileRec* __restrict__ tiles, uint32_t n_tiles)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles)
        return;
    uint32_t lo = 0, hi = n_descs;  // invariant: first_tile[lo] <= t < first_tile[hi] (hi == n: sentinel)
    while (hi - lo > 1) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (descs[mid].first_tile <= t)
            lo = mid;
        else
            hi = mid;
    }
    const DevDesc d = descs[lo];
    tiles[t] = make_tile_rec(d.src_off, d.dst_off, d.len, d.neg_state, t - d.first_tile, dst_align, lo);
}

// ---- search: decipher a tile into shared memory, match a pattern there, store nothing -------------------
//
// One CTA per tile of a plan whose chunk grid is co-aligned with the source, so every chunk is one LDG.128.
// The keystream is the batched kernel's: lazy states, speculative packing, and the thread's chunks redone
// exactly when one of their states had bit 31 set (the redo reloads its source: ~1 thread in 3 600).
// A match may start in the tile and end in the next L - 1 bytes of its entry, so a tile whose entry
// continues also deciphers that HALO (at most kHaloChunks chunks, exact, a constant jump from the tile
// state).  Every start position inside the tile is tested: a 2-byte SWAR filter, then a 4-byte masked word
// compare, then the remaining pattern bytes.  Matches are rare, so the atomics that count
// and list them are off the common path.
#ifndef MODK_MIN_CTAS_FIND
#define MODK_MIN_CTAS_FIND 10
#endif

__constant__ uint32_t c_halo_pow2[kHaloChunks];  // 2 * a^(16 * (kChunksPerTile + k)): halo chunk k's jump

__device__ __noinline__ void find_record(const FindArgs& f, uint32_t entry, int64_t src_rel, uint32_t p)
{
    const uint64_t src_off = __ldg(&f.descs[entry].src_off);
    atomicAdd(&f.counts[entry], 1u);
    const unsigned long long slot = atomicAdd(f.total, 1ull);
    if (slot < f.cap)
        f.matches[slot] = make_uint2(entry, (uint32_t)((uint64_t)(src_rel + (int64_t)p) - src_off));
}

// Bytes [lo, hi) of the 16 at `addr`, the others zero: for chunks whose granule may leave the source buffer.
__device__ __noinline__ uint4 load_bytes(uint64_t addr, uint32_t lo, uint32_t hi)
{
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (uint32_t b = 0; b < 16; ++b) {
        if (b >= lo && b < hi) {
            uint32_t byte;
            asm volatile("ld.global.u8 %0, [%1];" : "=r"(byte) : "l"(addr + b));
            w[b >> 2] |= byte << (8u * (b & 3u));
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// What a CTA knows about the tile it has deciphered: where the tile lies and which of its bytes are the entry's.
struct TileView {
    int64_t src_rel;   // the tile record's src_rel
    uint32_t entry;    // descriptor index
    uint32_t head;     // tile-local first byte of the entry
    uint32_t end;      // tile-local end of the entry's bytes in the tile
    uint32_t halo;     // entry bytes past the tile that were deciphered too
};

// The decipher stage of both search kernels: tile `rec` of a plan whose chunk grid lies on the source, deciphered
// into s_w (one LDG.128 per chunk, lazy states, speculative packing, the thread's chunks redone exactly from their
// source when one of their states had bit 31 set), plus up to `halo_max` entry bytes past the tile (exact, a
// constant jump from the tile state).  `pw` are the thread's chunk jump factors.  The caller synchronises the CTA
// before it reads s_w.
__device__ __forceinline__ TileView decipher_tile(const TileRec* rec, const uint8_t* src, uint64_t src_lo16, uint64_t src_hi16,
                                                  uint32_t halo_max, uint32_t two, const uint32_t (&pw)[kUnroll], uint32_t* s_w)
{
    constexpr int U = kUnroll;
    constexpr uint32_t T = (uint32_t)kThreadsPerCta;
    const uint32_t tid = threadIdx.x;
    const uint4* rp = reinterpret_cast<const uint4*>(rec);
    const uint4 lo = __ldg(rp);
    const uint4 hi = __ldg(rp + 1);
    const int64_t src_rel = (int64_t)((uint64_t)lo.x | ((uint64_t)lo.y << 32));
    const uint32_t st = hi.x, geom = hi.y, entry = hi.z;
    const uint32_t n_valid = geom & 0xFFFu, head = (geom >> 12) & 15u, tail = (geom >> 16) & 31u;
    const uint32_t end = 16u * (n_valid - 1u) + tail;  // tile-local end of the entry's bytes
    const uint32_t halo = min(hi.w, halo_max);         // entry bytes past the tile a match can reach
    const uint64_t src_tile = (uint64_t)src + (uint64_t)src_rel;
    const bool whole = src_tile >= src_lo16 && src_tile + 16ull * n_valid <= src_hi16;  // CTA-uniform

    auto load_chunk = [&](uint32_t idx) {
        return whole ? ldg128(src_tile + 16ull * idx)
                     : load_bytes(src_tile + 16ull * idx, idx == 0u ? head : 0u, idx + 1u == n_valid ? tail : 16u);
    };
    uint4 d[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const uint32_t idx = tid + (uint32_t)u * T;
        d[u] = make_uint4(0u, 0u, 0u, 0u);
        if (idx < n_valid)
            d[u] = load_chunk(idx);
    }
    // the halo: exact keystream, byte loads (it ends inside the entry, wherever the granule does)
    if (tid < (uint32_t)kHaloChunks && 16u * tid < halo) {
        const uint4 h = load_bytes(src_tile + 16ull * (n_valid + tid), 0u, min(16u, halo - 16u * tid));
        const uint4 o = cycle_chunk_exact(h, jump_lazy(st, c_halo_pow2[tid]), two);
        reinterpret_cast<uint4*>(s_w)[n_valid + tid] = o;
    }

    uint32_t s[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
        s[u] = jump_lazy(st, pw[u]);
    uint32_t any = 0u;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t b0 = step_lazy(s[u]);
            const uint32_t b1 = step_lazy(b0);
            const uint32_t b2 = step_lazy(b1);
            const uint32_t b3 = step_lazy(b2);
            s[u] = b3;
            const uint32_t l = __byte_perm(b0, b1, 0x7340);
            const uint32_t h = __byte_perm(b2, b3, 0x7340);
            any |= l | h;
            const uint32_t ks = __byte_perm(l, h, 0x5410);
            if (j == 0) d[u].x ^= ks;
            if (j == 1) d[u].y ^= ks;
            if (j == 2) d[u].z ^= ks;
            if (j == 3) d[u].w ^= ks;
        }
    }
    if (__builtin_expect((any & 0x80800000u) != 0u, 0)) {
        // some state needed a canonical subtract: redo this thread's chunks exactly from their source
#pragma unroll 1
        for (int u = 0; u < U; ++u) {
            const uint32_t idx = tid + (uint32_t)u * T;
            if (idx < n_valid)
                reinterpret_cast<uint4*>(s_w)[idx] =
                    cycle_chunk_exact(load_chunk(idx), jump_lazy(st, __ldg(&g_chunk_pow2[idx])), two);
        }
    } else {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t idx = tid + (uint32_t)u * T;
            if (idx < n_valid)
                reinterpret_cast<uint4*>(s_w)[idx] = d[u];
        }
    }
    return TileView{src_rel, entry, head, end, halo};
}

// The masked instantiation (kMasked) differs in the filter and the compare only.  Its filter tests the anchor pair
// (a, a + 1) -- the adjacent pattern bytes with the most mask bits, so that leading wildcards do not make every start
// a candidate -- with the same SWAR test on (bytes ^ rep) & mrep; its compare masks the head word and every byte.
//
// Shared slack.  The masked filter of word w reads words w + a/4 and w + a/4 + 1, bytes up to 4w + a + 7.  A word is
// tested only when 4w < p_end <= end + halo - L + 1, and a <= max(0, L - 2), halo <= min(rest, L - 1), so the
// farthest byte is end + halo + 5 <= kTileBytes + kMaxPattern + 4 for L >= 2 (and end + 6 for L = 1, where
// halo = 0).  s_w holds kTileBytes + 16 * kHaloChunks + 16 bytes.  Bytes past end + halo may be stale from an
// earlier layout of the array; only the filter reads them, the compare stays below p + L <= end + halo.
constexpr uint32_t kFindSlackWords = 4u;
static_assert(kTileBytes + kMaxPattern + 4u < kTileBytes + 16u * kHaloChunks + 4u * kFindSlackWords,
              "find_batch_kernel<true>: the masked filter reads past s_w");
template <bool kMasked>
__global__ void __launch_bounds__(kThreadsPerCta, MODK_MIN_CTAS_FIND) find_batch_kernel(const __grid_constant__ FindArgs f)
{
    constexpr uint32_t T = (uint32_t)kThreadsPerCta;
    // the tile, its halo, and slack for the filter's second word (the masked filter's words past the anchor)
    __shared__ __align__(16) uint32_t s_w[(kTileBytes + 16u * kHaloChunks) / 4u + kFindSlackWords];
    const uint32_t tid = threadIdx.x;
    uint32_t pw[kUnroll];
    load_chunk_pows<kUnroll>(pw, tid);
    const TileView v = decipher_tile(f.tiles + blockIdx.x, f.src, f.src_lo16, f.src_hi16, f.len - 1u, f.two, pw, s_w);
    const int64_t src_rel = v.src_rel;
    const uint32_t entry = v.entry, head = v.head, end = v.end, halo = v.halo;
    __syncthreads();

    // start positions [head, p_end): inside the tile's part of the entry, with room for the whole pattern
    const int32_t reach = (int32_t)(end + halo) - (int32_t)f.len + 1;
    const uint32_t p_end = (uint32_t)max(0, min((int32_t)end, reach));
    // Filter, 4 starts per word: a SWAR zero-byte test of (bytes ^ pattern[0]) AND-ed with the same test of the
    // next bytes ^ pattern[1] (L >= 2).  It flags every start whose first two bytes match (false positives only
    // above a matching byte), about 2 instructions per byte; the flagged starts are then compared exactly.
    const uint8_t* sb = reinterpret_cast<const uint8_t*>(s_w);
    const bool two_bytes = f.len > 1u;
    for (uint32_t w = (head >> 2) + tid; 4u * w < p_end; w += T) {
        const uint32_t x = s_w[w], y = s_w[w + 1u];
        uint32_t m;
        if constexpr (!kMasked) {
            const uint32_t v0 = x ^ f.rep0;
            m = (v0 - 0x01010101u) & ~v0;
            if (two_bytes) {
                const uint32_t v1 = __funnelshift_r(x, y, 8u) ^ f.rep1;
                m &= (v1 - 0x01010101u) & ~v1;
            }
        } else {
            // bytes p + a and p + a + 1 of starts p = 4w..4w+3; the clamped shift of a & 3 == 3 takes all of the second word
            const uint32_t wa = w + (f.anchor >> 2u), sh = 8u * (f.anchor & 3u);
            const uint32_t xa = s_w[wa], ya = s_w[wa + 1u];
            const uint32_t v0 = (__funnelshift_r(xa, ya, sh) ^ f.rep0) & f.mrep0;
            m = (v0 - 0x01010101u) & ~v0;
            if (two_bytes) {
                const uint32_t v1 = (__funnelshift_rc(xa, ya, sh + 8u) ^ f.rep1) & f.mrep1;
                m &= (v1 - 0x01010101u) & ~v1;
            }
        }
        if (__builtin_expect((m & 0x80808080u) == 0u, 1))
            continue;
#pragma unroll 1
        for (uint32_t o = 0; o < 4u; ++o) {
            const uint32_t p = 4u * w + o;
            if (((__funnelshift_r(x, y, 8u * o) ^ f.head_word) & f.head_mask) != 0u || p < head || p >= p_end)
                continue;
            bool hit = true;
            for (uint32_t k = 4u; k < f.len && hit; ++k)
                hit = kMasked ? ((sb[p + k] ^ f.pattern[k]) & f.mask[k]) == 0u : sb[p + k] == f.pattern[k];
            if (hit)
                find_record(f, entry, src_rel, p);
        }
    }
}

// ---- pattern-set search: the same decipher stage, an exact 2-byte filter, the set verified in HBM -----------------
//
// A persistent grid (every resident CTA slot of the device, each looping over tiles) so that the 8 KiB filter
// bitmap is loaded into shared memory once per CTA rather than once per 8 KiB tile.  Per tile the CTA deciphers
// the tile plus min(rest, Lmax - 1) halo bytes, then tests every start in [head, p_end) -- p_end from Lmin, the
// owned-start bound and the tile end -- against the bitmap bit of its first two bytes.  A start that passes is a
// candidate, and find_set_verify (out of line) checks each pattern that can start there, its end against the
// entry's.
#ifndef MODK_MIN_CTAS_FIND_SET
#define MODK_MIN_CTAS_FIND_SET 10
#endif

// Every pattern of the set that starts at tile-local p, whose first two bytes passed the filter: the length-1
// pattern of the first byte, then the patterns of the 2-byte key (binary search over the distinct keys), each
// checked against `lim` (where the deciphered entry bytes end), its head word and then its remaining bytes.
// `pos0` is the entry position of tile-local byte 0.  A folded set (kFold) holds upper-cased patterns, so the
// candidate's key, head word and bytes are folded before they are compared.
template <bool kFold>
__device__ __noinline__ void find_set_verify(const FindSetArgs& f, const uint8_t* sb, const uint16_t* s_keys, uint32_t p,
                                             uint32_t lim, uint32_t entry, int64_t pos0)
{
    auto at = [&](uint32_t i) -> uint32_t { return kFold ? fold_ascii(sb[i]) : sb[i]; };
    auto record = [&](uint32_t id) {
        atomicAdd(&f.counts[entry], 1u);
        atomicAdd(&f.pattern_counts[id], 1ull);
        const unsigned long long slot = atomicAdd(f.total, 1ull);
        if (slot < f.cap) {
            uint32_t* m = f.matches + 3ull * slot;
            m[0] = entry;
            m[1] = (uint32_t)(pos0 + (int64_t)p);
            m[2] = id;
        }
    };
    const uint32_t b0 = at(p), key = b0 | (at(p + 1) << 8);
    const uint32_t one = __ldg(&f.set->one[b0]);
    if (one)
        record(one - 1u);
    uint32_t lo = 0, hi = f.n_keys;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (s_keys[mid] < key)
            lo = mid + 1u;
        else
            hi = mid;
    }
    if (lo == f.n_keys || s_keys[lo] != key)
        return;
    const uint32_t word = b0 | (at(p + 1) << 8) | (at(p + 2) << 16) | (at(p + 3) << 24);
    const uint32_t r1 = __ldg(&f.set->group[lo + 1u]);
    for (uint32_t r = __ldg(&f.set->group[lo]); r < r1; ++r) {
        const uint4 sp = __ldg(reinterpret_cast<const uint4*>(&f.set->pat[r]));  // {id, len, head, mask}
        if (p + sp.y > lim || ((word ^ sp.z) & sp.w) != 0u)
            continue;
        bool hit = true;
        for (uint32_t k = 4u; k < sp.y && hit; ++k)
            hit = at(p + k) == __ldg(&f.set->bytes[r][k]);
        if (hit)
            record(sp.x);
    }
}

template <bool kFold>
__global__ void __launch_bounds__(kThreadsPerCta, MODK_MIN_CTAS_FIND_SET) find_set_kernel(const __grid_constant__ FindSetArgs f)
{
    constexpr uint32_t T = (uint32_t)kThreadsPerCta;
    __shared__ __align__(16) uint32_t s_w[(kTileBytes + 16u * kHaloChunks) / 4u + 4u];
    __shared__ __align__(16) uint32_t s_bm[65536u / 32u];
    __shared__ uint16_t s_keys[kMaxSetPatterns];
    const uint32_t tid = threadIdx.x;
    for (uint32_t i = tid; i < 65536u / 128u; i += T)
        reinterpret_cast<uint4*>(s_bm)[i] = __ldg(reinterpret_cast<const uint4*>(f.set->bitmap) + i);
    for (uint32_t i = tid; i < f.n_keys; i += T)
        s_keys[i] = __ldg(&f.set->keys[i]);
    uint32_t pw[kUnroll];
    load_chunk_pows<kUnroll>(pw, tid);
    const uint8_t* sb = reinterpret_cast<const uint8_t*>(s_w);
    for (uint32_t t = blockIdx.x; t < f.n_tiles; t += gridDim.x) {
        const TileView v = decipher_tile(f.tiles + t, f.src, f.src_lo16, f.src_hi16, f.lmax - 1u, f.two, pw, s_w);
        const int64_t pos0 = v.src_rel - (int64_t)__ldg(&f.descs[v.entry].src_off);
        const uint32_t lim = v.end + v.halo;  // every pattern must end here: the entry ends, or Lmax - 1 bytes on
        // starts [head, p_end): inside the tile, with room for the shortest pattern, below the owned bound
        int64_t p_end = min((int32_t)v.end, (int32_t)lim - (int32_t)f.lmin + 1);
        if (f.owned)
            p_end = min(p_end, (int64_t)__ldg(&f.owned[v.entry]) - pos0);
        const uint32_t pe = (uint32_t)max(p_end, (int64_t)0);
        __syncthreads();  // the tile (and, before the first, the bitmap and keys) are in shared memory
        for (uint32_t w = (v.head >> 2) + tid; 4u * w < pe; w += T) {
            const uint32_t x = s_w[w], y = s_w[w + 1u];
            auto bit = [&](uint32_t o) {  // the filter bit of start 4w + o, in bit 0
                const uint32_t key = __byte_perm(x, y, (o + 1u) << 4 | o) & 0xFFFFu;  // bytes p and p + 1
                return s_bm[key >> 5] >> (key & 31u);
            };
            if (__builtin_expect(((bit(0) | bit(1) | bit(2) | bit(3)) & 1u) == 0u, 1))
                continue;
#pragma unroll 1
            for (uint32_t o = 0; o < 4u; ++o) {
                const uint32_t p = 4u * w + o;
                if ((bit(o) & 1u) != 0u && p >= v.head && p < pe)
                    find_set_verify<kFold>(f, sb, s_keys, p, lim, v.entry, pos0);
            }
        }
        __syncthreads();  // the tile is no longer read: the next one may overwrite it
    }
}

// ---- host side --------------------------------------------------------------------------------------

cudaError_t upload_tables()
{
    static uint32_t h_tw0[kTw0Size], h_tw1[kTw1Size], h_ainv[16], h_chunk[kChunksPerTile], h_halo[kHaloChunks];
    static const bool built = []() {
        for (int j = 0; j < kTw0Size; ++j)
            h_tw0[j] = modlcg::pow_a((uint64_t)kTileBytes * (uint64_t)j);
        for (int j = 0; j < kTw1Size; ++j)
            h_tw1[j] = modlcg::pow_a((uint64_t)kTileBytes * (uint64_t)kTw0Size * (uint64_t)j);
        for (int h = 0; h < 16; ++h)
            h_ainv[h] = modlcg::pow_a_inv((uint64_t)h);
        for (int j = 0; j < kChunksPerTile; ++j)
            h_chunk[j] = 2u * modlcg::pow_a(16ull * (uint64_t)j);
        for (int k = 0; k < kHaloChunks; ++k)
            h_halo[k] = 2u * modlcg::pow_a(16ull * (uint64_t)(kChunksPerTile + k));
        return true;
    }();  // thread-safe: several device workers may call this at once
    (void)built;
    cudaError_t err;
    if ((err = cudaMemcpyToSymbol(c_tw0, h_tw0, sizeof(h_tw0))) != cudaSuccess) return err;
    if ((err = cudaMemcpyToSymbol(c_tw1, h_tw1, sizeof(h_tw1))) != cudaSuccess) return err;
    if ((err = cudaMemcpyToSymbol(c_ainv, h_ainv, sizeof(h_ainv))) != cudaSuccess) return err;
    if ((err = cudaMemcpyToSymbol(g_chunk_pow2, h_chunk, sizeof(h_chunk))) != cudaSuccess) return err;
    if ((err = cudaMemcpyToSymbol(c_halo_pow2, h_halo, sizeof(h_halo))) != cudaSuccess) return err;
    return cudaSuccess;
}

constexpr uint32_t kMaxGrid = 0x7FFFFFFFu;  // gridDim.x limit

// Every tile of the launch has source and destination co-aligned mod 16: all entries share one
// (src_off - dst_off) mod 16 and the two base pointers make up for it.
static bool coaligned(const BatchArgs& a)
{
    if (a.uniform_delta < 0 || getenv("MOD_FORCE_GENERAL") != nullptr)  // (the variable is a test / tuning aid)
        return false;
    return (((uintptr_t)a.src - (uintptr_t)a.dst + (uintptr_t)a.uniform_delta) & 15u) == 0u;
}

cudaError_t launch_batch(const BatchArgs& args, cudaStream_t stream)
{
    for (uint32_t t0 = 0; t0 < args.n_tiles;) {
        const uint32_t n = args.n_tiles - t0 < kMaxGrid ? args.n_tiles - t0 : kMaxGrid;
        BatchArgs a = args;
        a.tiles = args.tiles + t0;
        a.n_tiles = n;
        if (coaligned(args))
            cycle_batch_kernel<false><<<n, kThreadsPerCta, 0, stream>>>(a);
        else
            cycle_batch_kernel<true><<<n, kThreadsPerCta, 0, stream>>>(a);
        const cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess)
            return err;
        t0 += n;
    }
    return cudaSuccess;
}

cudaError_t launch_batch_inline(const BatchArgs& args, const InlineDescs& descs, cudaStream_t stream)
{
    if (args.n_tiles == 0)
        return cudaSuccess;
    if (coaligned(args))
        cycle_inline_kernel<false><<<args.n_tiles, kThreadsPerCta, 0, stream>>>(args, descs);
    else
        cycle_inline_kernel<true><<<args.n_tiles, kThreadsPerCta, 0, stream>>>(args, descs);
    return cudaGetLastError();
}

cudaError_t launch_find(const FindArgs& args, bool masked, cudaStream_t stream)
{
    for (uint32_t t0 = 0; t0 < args.n_tiles;) {
        const uint32_t n = args.n_tiles - t0 < kMaxGrid ? args.n_tiles - t0 : kMaxGrid;
        FindArgs a = args;
        a.tiles = args.tiles + t0;
        a.n_tiles = n;
        if (masked)
            find_batch_kernel<true><<<n, kThreadsPerCta, 0, stream>>>(a);
        else
            find_batch_kernel<false><<<n, kThreadsPerCta, 0, stream>>>(a);
        const cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess)
            return err;
        t0 += n;
    }
    return cudaSuccess;
}

cudaError_t launch_find_set(const FindSetArgs& args, bool fold, cudaStream_t stream)
{
    if (args.n_tiles == 0)
        return cudaSuccess;
    void (*kernel)(const FindSetArgs) = fold ? find_set_kernel<true> : find_set_kernel<false>;
    int dev = 0, sms = 0, per_sm = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err == cudaSuccess)
        err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (err == cudaSuccess)
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreadsPerCta, 0);
    if (err != cudaSuccess)
        return err;
    const uint32_t grid = (uint32_t)std::max(1, sms * per_sm);
    kernel<<<std::min(grid, args.n_tiles), kThreadsPerCta, 0, stream>>>(args);
    return cudaGetLastError();
}

cudaError_t launch_build_tiles(const DevDesc* descs, uint32_t n_descs, uint32_t dst_align, TileRec* tiles,
                               uint32_t n_tiles, cudaStream_t stream)
{
    if (n_tiles == 0)
        return cudaSuccess;
    const unsigned threads = 256;
    build_tiles_kernel<<<(n_tiles + threads - 1) / threads, threads, 0, stream>>>(descs, n_descs, dst_align,
                                                                                 tiles, n_tiles);
    return cudaGetLastError();
}

}  // namespace modk
