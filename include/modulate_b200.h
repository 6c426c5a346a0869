/*
 * modulate_b200.h -- C ABI of the B200-native keystream / archive data-movement path.
 *
 * This is the drop-in boundary for the one data-parallel hot path of AdamClixby/Modulate:
 *   - CEncryptionCycler::Cycle            (reference CEncryptionCycler.h:6, CEncryptionCycler.cpp:4-25)
 *   - CArk::ExtractFiles' gather          (reference CArk.cpp:494, by mi64Offset / miSize)
 *   - CArk::BuildArk's scatter            (reference CArk.cpp:807-811)
 *   - the three Cycle call sites          (CArk.cpp:338-339, CArk.cpp:1135-1136, Modulate.cpp:485-486)
 *
 * The reference has no FFI layer (it is one statically linked C++ program), so the entry
 * points below are what a binding for this path would bind: plain pointers and sizes, no
 * C++ or torch types.  The C++ facade classes with the reference's own signatures
 * (modulate_b200/csrc/CEncryptionCycler.h, CArk.h) forward to these functions; see
 * INTEGRATION.md for the two-line change a maintainer of the reference would make.
 *
 * Conventions
 *   - Every function that can fail returns int: 0 (MOD_OK) on success, a negative MOD_ERR_*
 *     otherwise; mod_last_error() returns a thread-local human-readable message.
 *   - There is NO CPU fallback.  If no CUDA device / driver is usable, compute entry points
 *     return MOD_ERR_CUDA and the C++ facade aborts loudly (the reference's Cycle is void).
 *   - Every visible GPU has its own context inside the library (streams, HBM workspaces, jump
 *     tables); nothing is torn down when a thread switches devices.  Single-device entry points
 *     work on the calling thread's current CUDA device (mod_init(d) sets it); the *_sharded entry
 *     points split one call over several GPUs inside ONE process (one host thread + stream set per
 *     device, SURVEY.md section 8(e)).  One process per GPU with the work split by mod_shard_descs
 *     / mod_shard_range works equally well -- shards are independent, so no collective is needed.
 *   - "stream" parameters are a cudaStream_t passed as void* (NULL = the legacy default stream).
 *     Functions taking a stream are asynchronous; the others return after the result is visible
 *     to the caller, which preserves Cycle's in-place contract.
 */
#ifndef MODULATE_B200_H
#define MODULATE_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOD_OK 0
#define MOD_ERR_CUDA (-1)      /* CUDA runtime / driver error (message holds cudaGetErrorString) */
#define MOD_ERR_ARG (-2)       /* invalid argument (null pointer, descriptor outside its buffer, ...) */
#define MOD_ERR_ALIGN (-3)     /* plan was built for a different dst alignment (dst & 15) */
#define MOD_ERR_NOMEM (-4)     /* host or device allocation failed */

#define MOD_ABI_VERSION 2

/* One archive entry / stream piece: copy `len` bytes from src+src_off to dst+dst_off while XORing
 * them with the keystream of CEncryptionCycler::Cycle(., len, key), the stream restarting at the
 * entry's first byte.  Device form of CArk::sFileDefinition {mi64Offset, miSize} (CArk.h:55-69)
 * plus a per-entry key.  key == 0 (mod 2^31-1) is the identity keystream, i.e. the reference's
 * plain fwrite/fread copy.  `len` is 32-bit like the reference's `unsigned int liDataSize`. */
typedef struct mod_desc {
    uint64_t src_off;
    uint64_t dst_off;
    uint32_t len;
    int32_t key;
} mod_desc;

typedef struct mod_plan mod_plan; /* opaque: descriptors + tile map resident in HBM */

/* ---- library / device management --------------------------------------------------------- */

int mod_abi_version(void);
/* Number of CUDA devices visible, or a negative MOD_ERR_* . */
int mod_device_count(void);
/* Bind the calling process to `device` (-1 = keep the current device), create the internal
 * streams and upload the jump tables.  Idempotent.  Called implicitly by the compute entry points. */
int mod_init(int device);
/* The CUDA device the calling thread is bound to, or a negative MOD_ERR_*. */
int mod_current_device(void);
/* 1 if `p` points into device (or managed) memory, 0 if it is a host pointer. */
int mod_is_device_pointer(const void* p);
void mod_shutdown(void);
const char* mod_last_error(void);
/* Kernels this library has launched in this process (all streams): bench.py's gpu_launches. */
uint64_t mod_launch_count(void);

/* ---- memory helpers ---------------------------------------------------------------------- */

void* mod_host_alloc(uint64_t bytes); /* pinned (page-locked, portable across devices) host memory; NULL on failure */
int mod_host_free(void* p);
void* mod_device_alloc(uint64_t bytes); /* HBM; NULL on failure */
int mod_device_free(void* p);
int mod_memcpy_h2d(void* d_dst, const void* h_src, uint64_t bytes, void* stream);
int mod_memcpy_d2h(void* h_dst, const void* d_src, uint64_t bytes, void* stream);
int mod_stream_sync(void* stream);
void* mod_stream_create(void); /* non-blocking stream on the current device; NULL on failure */
int mod_stream_destroy(void* stream);

/* ---- CEncryptionCycler::Cycle ------------------------------------------------------------ */

/* Exact semantics of CEncryptionCycler::Cycle (CEncryptionCycler.cpp:4-14) on `len` bytes at `data`,
 * in place, synchronous.  `data` may be a host pointer (pageable or pinned: staged through HBM in
 * pipelined slices, H2D / kernel / D2H overlapped) or a device pointer (cycled in HBM).  `len` is
 * 64-bit: streams longer than the reference's 32-bit length continue the same keystream
 * (period 2^31-2). */
int mod_cycle(void* data, uint64_t len, int32_t key);

/* mod_cycle on a HOST buffer split by offset range over several GPUs of this process: device g of
 * the G selected ones ciphers bytes mod_shard_range(len, g, G) starting from the jumped key
 * (mod_key_jump), each on its own host thread and stream set; returns when every range is back in
 * `data`.  `dev_mask` bit d selects CUDA device d; 0 = every visible device.  Lifts the reference's
 * single-threaded, 32-bit-length Cycle (CEncryptionCycler.h:6) to a whole node. */
int mod_cycle_sharded(void* data, uint64_t len, int32_t key, uint64_t dev_mask);

/* Device-resident, asynchronous on `stream`.  d_src == d_dst is the in-place form; otherwise the
 * ranges must not overlap.  No alignment requirement on either pointer. */
int mod_cycle_device(const void* d_src, void* d_dst, uint64_t len, int32_t key, void* stream);

/* Key k' such that Cycle(., ., k') emits the keystream of Cycle(., ., key) from byte `pos` on:
 * the O(log pos) modular jump-ahead used for offset-range sharding.  Pure host arithmetic. */
int32_t mod_key_jump(int32_t key, uint64_t pos);

/* ---- descriptor batches: CArk extract (gather) / build (scatter) / per-entry keys ----------- */

/* Validate `n` host descriptors against the two buffer sizes, upload them, and build the per-tile
 * records in HBM (the device form of the file table CArk::Load builds, CArk.cpp:401-408).  `dst_align` is (address of dst) & 15 for the buffer the plan will be
 * run on (0 for anything from mod_device_alloc / cudaMalloc).  Entries whose dst ranges overlap
 * give unspecified results (the reference never produces them). */
int mod_plan_create(const mod_desc* descs, uint64_t n, uint64_t src_bytes, uint64_t dst_bytes,
                    uint32_t dst_align, mod_plan** out);
/* Waits for the device (launches that still read the plan's records), then hands the records' HBM block back to
 * a small per-device pool that the next mod_plan_create draws from -- cudaMalloc / cudaFree are not on the
 * per-archive path.  mod_shutdown releases the pool. */
int mod_plan_destroy(mod_plan* plan);
uint64_t mod_plan_payload_bytes(const mod_plan* plan); /* sum of len */
uint64_t mod_plan_num_tiles(const mod_plan* plan);

/* One launch of the variable-length batched kernel over every descriptor of the plan: replaces the
 * per-entry loops of CArk::ExtractFiles (CArk.cpp:435-501, payload move :494) and CArk::BuildArk
 * (CArk.cpp:784-822, payload move :807-811), with one CEncryptionCycler::Cycle per entry folded in.
 * Asynchronous on `stream`.  d_src == d_dst with src_off == dst_off is the in-place form. */
int mod_plan_run(const mod_plan* plan, const void* d_src, void* d_dst, void* stream);

/* Tiles [*tile_begin, *tile_end) of the plan that belong to descriptors [entry_begin, entry_end). */
int mod_plan_tile_range(const mod_plan* plan, uint64_t entry_begin, uint64_t entry_end, uint64_t* tile_begin,
                        uint64_t* tile_end);

/* Run tiles [tile_begin, tile_end) of the plan with only a WINDOW of each buffer resident: bytes
 * [src_win_off, +src_win_bytes) of the plan's source space live at d_src_win and bytes
 * [dst_win_off, +dst_win_bytes) of its destination space at d_dst_win ((d_dst_win - dst_win_off) & 15
 * must equal the plan's dst_align).  Every byte the tile range touches must lie inside the windows
 * (checked on the host).  This is what lets a caller stream an archive through a ring of slot
 * buffers with ONE plan -- CArk::ExtractFiles / BuildArk do (the reference holds the whole image in
 * one allocation, CArk.cpp:738, :780).  Asynchronous on `stream`. */
int mod_plan_run_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                        uint64_t src_win_off, uint64_t src_win_bytes, void* d_dst_win, uint64_t dst_win_off,
                        uint64_t dst_win_bytes, void* stream);

/* Convenience: plan + run + destroy, synchronous.  `src` / `dst` are both host pointers (staged
 * through HBM in groups of entries, upload / kernel / download overlapped) or both device pointers.
 * In both forms bytes of dst that no descriptor covers keep their value. */
int mod_cycle_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes,
                    void* dst, uint64_t dst_bytes);

/* mod_cycle_batch on HOST buffers split over several GPUs of this process: the descriptor list is
 * cut into equal-payload shards (mod_shard_descs) and each selected device streams its shard on its
 * own host thread and stream set.  `dev_mask` as for mod_cycle_sharded. */
int mod_cycle_batch_sharded(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes,
                            void* dst, uint64_t dst_bytes, uint64_t dev_mask);

/* ---- search: which entries contain a byte pattern ------------------------------------------ */

/* One match: `pos` is where the pattern starts inside descriptor `desc`'s deciphered bytes. */
typedef struct mod_match {
    uint32_t desc;
    uint32_t pos;
} mod_match;

/* Search every descriptor of `plan` for the `len`-byte pattern (1 <= len <= 64, else MOD_ERR_ARG).  A
 * descriptor's bytes are src[src_off, +len) after Cycle(., len, key) -- what mod_plan_run would write for
 * it -- and every start i with i + pattern_len <= len whose bytes equal the pattern is a match, overlapping
 * matches included; a match never spans two descriptors.  The plan must have been built with dst_off ==
 * src_off for every descriptor and dst_align == d_src & 15 (the chunk grid then lies on the source, and
 * nothing is written but the results).  Results ACCUMULATE, so the caller zeroes them first:
 * d_counts[i] += matches in descriptor i (uint32_t per descriptor of the plan); *d_total += all matches;
 * each match takes slot (*d_total before it) of d_matches and is stored only if that slot is below `cap`.
 * The list order is unspecified; the counts are exact however many matches the list drops.
 * Asynchronous on `stream`; all four result pointers are device memory. */
int mod_plan_find(const mod_plan* plan, const void* d_src, const uint8_t* pattern, uint32_t len, uint32_t* d_counts,
                  mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream);

/* mod_plan_find over tiles [tile_begin, tile_end) with only a window of the source resident (bytes
 * [src_win_off, +src_win_bytes) of the plan's source space at d_src_win; (d_src_win - src_win_off) & 15
 * must equal the plan's dst_align).  Every byte the tiles read, the up to len - 1 bytes past a tile that a
 * match starting in it may cover included, must lie inside the window (checked on the host).  This is the
 * slot-ring form CArk::FindInFiles streams an archive through.  Asynchronous on `stream`. */
int mod_plan_find_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                         uint64_t src_win_off, uint64_t src_win_bytes, const uint8_t* pattern, uint32_t len,
                         uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream);

/* Plan + find + destroy, synchronous: `d_src` must be device memory (MOD_ERR_ARG otherwise).  The HOST
 * outputs get the per-descriptor counts (n entries), the total, and min(total, cap) matches sorted by
 * (desc, pos); which matches a truncated list keeps is unspecified.  Only src_off, len and key of the
 * descriptors are used. */
int mod_find_batch(const mod_desc* descs, uint64_t n, const void* d_src, uint64_t src_bytes, const uint8_t* pattern,
                   uint32_t len, uint32_t* counts_out, mod_match* matches_out, uint64_t cap, uint64_t* total_out);

/* ---- masked search: wildcard bytes and nibbles, ASCII case folding --------------------------- */

/* mod_plan_find with a mask byte per pattern byte: byte t matches pattern byte k when
 * ((t ^ pattern[k]) & mask[k]) == 0.  mask 0xFF is an exact byte, 0x00 any byte, 0xF0 / 0x0F leave one nibble
 * free, and 0xDF with pattern[k] in 'A'..'Z' matches that letter in either case.  The results, their accumulation
 * and the cap are mod_plan_find's.  MOD_ERR_ARG for a null mask, len outside 1..64 and an all-zero mask.  An
 * all-0xFF mask runs the exact search.  Asynchronous on `stream`. */
int mod_plan_find_masked(const mod_plan* plan, const void* d_src, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                         uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream);

/* mod_plan_find_window with a mask, as mod_plan_find_masked. */
int mod_plan_find_masked_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                                uint64_t src_win_off, uint64_t src_win_bytes, const uint8_t* pattern, const uint8_t* mask,
                                uint32_t len, uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total,
                                void* stream);

/* mod_find_batch with a mask, as mod_plan_find_masked. */
int mod_find_masked_batch(const mod_desc* descs, uint64_t n, const void* d_src, uint64_t src_bytes, const uint8_t* pattern,
                          const uint8_t* mask, uint32_t len, uint32_t* counts_out, mod_match* matches_out, uint64_t cap,
                          uint64_t* total_out);

/* ---- search for a set of patterns in one pass ------------------------------------------------ */

typedef struct mod_pattern_set mod_pattern_set; /* opaque: the set's filter and index, resident in HBM */

/* One match of a set: pattern `pattern` (its position in the list the set was created from) starts at `pos`
 * inside descriptor `desc`'s deciphered bytes. */
typedef struct mod_set_match {
    uint32_t desc;
    uint32_t pos;
    uint32_t pattern;
} mod_set_match;

/* Build a set of `n` patterns (1 <= n <= 256) on the calling thread's current device: pattern j is lens[j] bytes
 * (1..64) of `bytes`, the patterns concatenated in list order.  Lengths may differ; the same pattern twice is
 * refused.  Every invalid input is MOD_ERR_ARG, checked on the host.  Synchronous. */
int mod_pattern_set_create(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out);
int mod_pattern_set_destroy(mod_pattern_set* set);

/* mod_pattern_set_create for a case-insensitive search: ASCII letters 'A'..'Z' match 'a'..'z' and back, every other
 * byte only itself.  Two patterns that are equal ignoring case are refused.  The set is searched with
 * mod_plan_find_set / _window like any other. */
int mod_pattern_set_create_nocase(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out);

/* mod_plan_find for every pattern of `set` in one pass over the source.  A match is a pair (pattern j, start p)
 * with p + len_j <= len whose bytes equal pattern j: overlapping matches count, and so do matches of different
 * patterns at one start.  `d_owned` (device, one uint32 per descriptor, or NULL): starts p >= d_owned[i] of
 * descriptor i are not reported -- what lets pieces of one entry overlap by Lmax - 1 bytes and still report each
 * match once.  Results ACCUMULATE into caller-zeroed device memory: d_counts[i] (uint32) += matches in descriptor
 * i; d_pattern_counts[j] (uint64) += matches of pattern j; *d_total += all matches; each match takes slot
 * (*d_total before it) of d_matches and is stored only if that slot is below `cap`.  The list order is
 * unspecified; the counts are exact however many matches the list drops.  The set must live on the plan's
 * device (MOD_ERR_ARG otherwise); the plan must lie on the source grid as for mod_plan_find (MOD_ERR_ALIGN).
 * Asynchronous on `stream`. */
int mod_plan_find_set(const mod_plan* plan, const void* d_src, const mod_pattern_set* set, const uint32_t* d_owned,
                      uint32_t* d_counts, uint64_t* d_pattern_counts, mod_set_match* d_matches, uint64_t cap,
                      uint64_t* d_total, void* stream);

/* mod_plan_find_set over tiles [tile_begin, tile_end) with only a window of the source resident, as
 * mod_plan_find_window with Lmax (the set's longest pattern) in place of the pattern length. */
int mod_plan_find_set_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                             uint64_t src_win_off, uint64_t src_win_bytes, const mod_pattern_set* set,
                             const uint32_t* d_owned, uint32_t* d_counts, uint64_t* d_pattern_counts,
                             mod_set_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream);

/* Set + plan + find + destroy, synchronous: `d_src` must be device memory.  The HOST outputs get the counts per
 * descriptor (n) and per pattern (n_patterns), the total, and min(total, cap) matches sorted by
 * (desc, pos, pattern). */
int mod_find_set_batch(const mod_desc* descs, uint64_t n, const void* d_src, uint64_t src_bytes, const uint8_t* bytes,
                       const uint32_t* lens, uint32_t n_patterns, uint32_t* counts_out, uint64_t* pattern_counts_out,
                       mod_set_match* matches_out, uint64_t cap, uint64_t* total_out);

/* ---- offset-range sharding (host logic, no GPU needed) -------------------------------------- */

/* (No reference counterpart: the reference is single-threaded, SURVEY.md section 8(e).)
 * Byte range [*begin, *end) of a `total`-byte stream owned by `rank` of `world`: equal shares
 * rounded to 16-byte boundaries (the last rank takes the remainder). */
int mod_shard_range(uint64_t total, int rank, int world, uint64_t* begin, uint64_t* end);

/* Split a descriptor list into `world` shards of (nearly) equal payload bytes and write rank's
 * shard to `out` (capacity out_cap; pass out == NULL to query the count).  An entry that straddles
 * a shard boundary is cut at a 16-byte-aligned position inside the entry and the second piece gets
 * the jumped key (mod_key_jump), so the union of all shards is byte-identical to the unsharded
 * batch.  Returns the number of descriptors in rank's shard, or a negative MOD_ERR_*. */
int64_t mod_shard_descs(const mod_desc* descs, uint64_t n, int rank, int world, mod_desc* out,
                        uint64_t out_cap);

/* How the host-pointer batch path (mod_cycle_batch on host buffers) cuts a descriptor list into pipeline
 * groups of ~group_bytes of payload: group boundaries fall on destination addresses with
 * (dst_phase + dst_off) % modulus == 0 INSIDE entries (modulus a power of two >= 16; the library uses 128 and
 * the low bits of the caller's dst pointer, because pinned <-> HBM copies only run at full speed between
 * 128-byte aligned addresses); a piece that starts `pos` bytes into its entry carries the jumped key.
 * Writes the pieces to `out` and, per piece, whether a group ends after it to `closes` (capacity out_cap each;
 * pass out == NULL to query the count).  Returns the number of pieces, or a negative MOD_ERR_*.  Host logic, no
 * GPU needed (exposed so the cut can be tested and reproduced). */
int64_t mod_group_descs(const mod_desc* descs, uint64_t n, uint64_t group_bytes, uint64_t dst_phase, uint64_t modulus,
                        mod_desc* out, uint8_t* closes, uint64_t out_cap);

#ifdef __cplusplus
}
#endif

#endif /* MODULATE_B200_H */
