// mod_abi.cu -- the C ABI declared in include/modulate_b200.h: per-device contexts, pinned / HBM
// memory helpers, CEncryptionCycler::Cycle on host or device buffers, descriptor plans for CArk's
// extract / build data movement, the in-process multi-GPU entry points and the host-side shard
// planner.  No CPU compute path exists here: every byte of keystream is produced by the kernels in
// cycle_kernels.cu.
#include "../../include/modulate_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <mutex>
#include <memory>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "batch_cut.h"
#include "cycle_kernels.cuh"
#include "lcg.h"

namespace {

#ifndef MOD_PIPE_SLOTS
#define MOD_PIPE_SLOTS 4
#endif
constexpr int kPipeSlots = MOD_PIPE_SLOTS;  // slices / groups in flight on the host-pointer paths
constexpr uint64_t kMaxPiece = 1ull << 30;  // a contiguous stream is cut into <= 1 GiB pieces
constexpr int kMaxDevices = 64;
constexpr uint64_t kCopyAlign = 128;        // pinned <-> HBM copies run ~13 % faster between 128-byte aligned addresses

thread_local std::string tl_error = "";
std::atomic<uint64_t> g_launches{0};

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    tl_error = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return fail(MOD_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

// No C++ exception may cross the extern "C" boundary (a C caller would std::terminate).
#define MOD_ABI_BEGIN try {
#define MOD_ABI_END(name)                                                                       \
    }                                                                                           \
    catch (const std::bad_alloc&) { return fail(MOD_ERR_NOMEM, name ": out of host memory"); }  \
    catch (const std::exception& ex__) { return fail(MOD_ERR_ARG, name ": %s", ex__.what()); }  \
    catch (...) { return fail(MOD_ERR_ARG, name ": unknown exception"); }

// Everything the library owns on ONE GPU.  Contexts of different devices are independent: binding
// another device never tears one down, and the sharded entry points drive several at once.
struct DeviceCtx {
    int device = -1;
    std::atomic<bool> ready{false};
    std::mutex mu;  // the host-pointer paths share the workspaces below: one call at a time per device
    cudaStream_t pipe_stream[kPipeSlots] = {};
    cudaEvent_t plan_ready = nullptr;
    // grow-only HBM workspaces: slices of mod_cycle, source / destination windows of mod_cycle_batch
    void* slice_buf[kPipeSlots] = {};
    uint64_t slice_bytes[kPipeSlots] = {};
    void* slot_src[kPipeSlots] = {};
    uint64_t slot_src_bytes[kPipeSlots] = {};
    void* slot_dst[kPipeSlots] = {};
    uint64_t slot_dst_bytes[kPipeSlots] = {};
    // plan scratch of the host-pointer batch path: pinned staging for descriptors, HBM descriptors + tiles
    void* h_descs = nullptr;
    uint64_t h_descs_bytes = 0;
    void* ws_descs = nullptr;
    uint64_t ws_descs_bytes = 0;
    void* ws_tiles = nullptr;
    uint64_t ws_tiles_bytes = 0;
    // HBM blocks handed back by destroyed plans, kept for the next plan: cudaMalloc / cudaFree are device-wide
    // synchronisation points that were seen to stall for 0.1-1 s inside a process that holds many other
    // allocations, which is more than moving a whole archive costs
    struct Block {
        void* p;
        uint64_t bytes;
    };
    std::mutex pool_mu;
    std::vector<Block> pool;
};
constexpr size_t kPoolBlocks = 8;
constexpr uint64_t kPoolMaxBlockBytes = 256ull << 20;

DeviceCtx g_dev[kMaxDevices];
std::mutex g_init_mu;

double now_ms()
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

uint64_t env_u64(const char* name, uint64_t dflt)
{
    const char* v = getenv(name);
    if (!v || !*v)
        return dflt;
    return strtoull(v, nullptr, 10);
}

// Switch the calling thread to `device` for the lifetime of the guard.
class DeviceGuard {
public:
    int enter(int device)
    {
        CUDA_TRY(cudaGetDevice(&prev_));
        if (prev_ != device) {
            CUDA_TRY(cudaSetDevice(device));
            active_ = true;
        }
        return MOD_OK;
    }
    ~DeviceGuard()
    {
        if (active_)
            cudaSetDevice(prev_);
    }

private:
    int prev_ = -1;
    bool active_ = false;
};

void release_ctx(DeviceCtx& c)  // current device == c.device
{
    auto drop = [](void*& p, uint64_t& n) {
        if (p)
            cudaFree(p);
        p = nullptr;
        n = 0;
    };
    for (int i = 0; i < kPipeSlots; ++i) {
        drop(c.slice_buf[i], c.slice_bytes[i]);
        drop(c.slot_src[i], c.slot_src_bytes[i]);
        drop(c.slot_dst[i], c.slot_dst_bytes[i]);
    }
    drop(c.ws_descs, c.ws_descs_bytes);
    drop(c.ws_tiles, c.ws_tiles_bytes);
    {
        std::lock_guard<std::mutex> lock(c.pool_mu);
        for (DeviceCtx::Block& b : c.pool)
            cudaFree(b.p);
        c.pool.clear();
    }
    if (c.h_descs)
        cudaFreeHost(c.h_descs);
    c.h_descs = nullptr;
    c.h_descs_bytes = 0;
    if (c.plan_ready)
        cudaEventDestroy(c.plan_ready);
    c.plan_ready = nullptr;
    for (int i = 0; i < kPipeSlots; ++i) {
        if (c.pipe_stream[i])
            cudaStreamDestroy(c.pipe_stream[i]);
        c.pipe_stream[i] = nullptr;
    }
    c.ready.store(false, std::memory_order_release);
}

// Bind (device >= 0) or keep (device < 0) the calling thread's CUDA device and return its context,
// preparing it on first use: jump tables, pipeline streams.
int acquire(int device, DeviceCtx** out)
{
    int count = 0;
    CUDA_TRY(cudaGetDeviceCount(&count));
    if (count <= 0)
        return fail(MOD_ERR_CUDA, "no CUDA device visible: this library has no CPU fallback");
    if (device >= 0) {
        if (device >= count || device >= kMaxDevices)
            return fail(MOD_ERR_ARG, "device %d out of range (%d visible)", device, count);
        CUDA_TRY(cudaSetDevice(device));
    }
    int cur = 0;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur >= kMaxDevices)
        return fail(MOD_ERR_ARG, "device %d beyond the supported %d", cur, kMaxDevices);
    DeviceCtx& c = g_dev[cur];
    if (!c.ready.load(std::memory_order_acquire)) {
        std::lock_guard<std::mutex> lock(g_init_mu);
        if (!c.ready.load(std::memory_order_relaxed)) {
            c.device = cur;
            const double t_ctx = now_ms();
            CUDA_TRY(modk::upload_tables());
            if (env_u64("MOD_TRACE", 0) != 0)
                fprintf(stderr, "[mod] device %d: context + module load + jump tables: %.1f ms\n", cur, now_ms() - t_ctx);
            for (int i = 0; i < kPipeSlots; ++i)
                if (!c.pipe_stream[i])
                    CUDA_TRY(cudaStreamCreateWithFlags(&c.pipe_stream[i], cudaStreamNonBlocking));
            if (!c.plan_ready)
                CUDA_TRY(cudaEventCreateWithFlags(&c.plan_ready, cudaEventDisableTiming));
            c.ready.store(true, std::memory_order_release);
        }
    }
    *out = &c;
    return MOD_OK;
}

// Wait for everything the host-pointer paths have in flight on this device: called on every exit
// of those paths, error exits included, because the copies reference the CALLER's buffers.
cudaError_t drain(DeviceCtx& c)
{
    cudaError_t first = cudaSuccess;
    for (int k = 0; k < kPipeSlots; ++k) {
        const cudaError_t e = cudaStreamSynchronize(c.pipe_stream[k]);
        if (first == cudaSuccess)
            first = e;
    }
    return first;
}

bool pointer_device(const void* p, int* device)
{
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    if (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) {
        *device = attr.device;
        return true;
    }
    return false;
}

int grow(void** buf, uint64_t* have, uint64_t need)
{
    if (*have >= need)
        return MOD_OK;
    if (*buf) {
        CUDA_TRY(cudaFree(*buf));
        *buf = nullptr;
        *have = 0;
    }
    need = (need + 255) & ~255ull;
    cudaError_t e = cudaMalloc(buf, need);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *buf = nullptr;
        return fail(MOD_ERR_NOMEM, "cudaMalloc(%llu) failed: %s", (unsigned long long)need, cudaGetErrorString(e));
    }
    *have = need;
    return MOD_OK;
}

int grow_pinned(void** buf, uint64_t* have, uint64_t need)
{
    if (*have >= need)
        return MOD_OK;
    if (*buf) {
        CUDA_TRY(cudaFreeHost(*buf));
        *buf = nullptr;
        *have = 0;
    }
    need = (need + 4095) & ~4095ull;
    cudaError_t e = cudaHostAlloc(buf, need, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *buf = nullptr;
        return fail(MOD_ERR_NOMEM, "cudaHostAlloc(%llu) failed: %s", (unsigned long long)need, cudaGetErrorString(e));
    }
    *have = need;
    return MOD_OK;
}

// Plan scratch from the device's block pool (current device == c.device).  A cached block serves a request
// it is not more than 4x too large for; *got receives the block's real size for pool_free.
cudaError_t pool_alloc(DeviceCtx& c, uint64_t bytes, void** out, uint64_t* got)
{
    bytes = std::max<uint64_t>(256, (bytes + 255) & ~255ull);
    {
        std::lock_guard<std::mutex> lock(c.pool_mu);
        size_t best = c.pool.size();
        for (size_t i = 0; i < c.pool.size(); ++i)
            if (c.pool[i].bytes >= bytes && c.pool[i].bytes / 4 <= bytes && (best == c.pool.size() || c.pool[i].bytes < c.pool[best].bytes))
                best = i;
        if (best != c.pool.size()) {
            *out = c.pool[best].p;
            *got = c.pool[best].bytes;
            c.pool.erase(c.pool.begin() + (long)best);
            return cudaSuccess;
        }
    }
    *got = bytes;
    return cudaMalloc(out, bytes);
}

void pool_free(DeviceCtx& c, void* p, uint64_t bytes)
{
    if (!p)
        return;
    if (bytes <= kPoolMaxBlockBytes && c.ready.load(std::memory_order_acquire)) {
        std::lock_guard<std::mutex> lock(c.pool_mu);
        if (c.pool.size() >= kPoolBlocks) {  // full: the smallest cached block makes room if this one is larger
            size_t smallest = 0;
            for (size_t i = 1; i < c.pool.size(); ++i)
                if (c.pool[i].bytes < c.pool[smallest].bytes)
                    smallest = i;
            if (c.pool[smallest].bytes < bytes) {
                cudaFree(c.pool[smallest].p);
                c.pool[smallest] = DeviceCtx::Block{p, bytes};
                return;
            }
        } else {
            c.pool.push_back(DeviceCtx::Block{p, bytes});
            return;
        }
    }
    cudaFree(p);
}

// One launch (or a few, beyond 64 pieces) of the batched kernel over a contiguous stream.
int launch_contiguous(const uint8_t* d_src, uint8_t* d_dst, uint64_t len, int32_t key, cudaStream_t stream)
{
    if (len == 0)
        return MOD_OK;
    const uint32_t h0 = (uint32_t)((uintptr_t)d_dst & 15u);
    const uint64_t piece = kMaxPiece;
    const uint64_t src_lo16 = ((uint64_t)(uintptr_t)d_src + 15u) & ~15ull;
    const uint64_t src_hi16 = ((uint64_t)(uintptr_t)d_src + len) & ~15ull;
    const uint32_t tpe = modk::tiles_for_entry(h0, (uint32_t)piece);
    uint64_t done = 0;
    const uint32_t k0 = modlcg::key_residue(key);
    while (done < len) {
        modk::InlineDescs in;
        modk::BatchArgs args;
        uint32_t n = 0, tiles = 0;
        const uint64_t group_base = done;
        while (done < len && n < (uint32_t)modk::kMaxInlineDescs) {
            const uint64_t this_len = std::min(piece, len - done);
            modk::DevDesc& d = in.d[n];
            d.src_off = done - group_base;
            d.dst_off = done - group_base;
            d.len = (uint32_t)this_len;
            d.key = (int32_t)modlcg::mulmod(k0, modlcg::pow_a(done));
            d.first_tile = n * tpe;
            d.neg_state = modlcg::key_to_neg_state(d.key);
            tiles = n * tpe + modk::tiles_for_entry(h0, (uint32_t)this_len);
            done += this_len;
            ++n;
        }
        args.src = d_src + group_base;
        args.dst = d_dst + group_base;
        args.tiles = nullptr;
        args.n_tiles = tiles;
        args.tiles_per_entry = tpe;
        args.src_lo16 = src_lo16;
        args.src_hi16 = src_hi16;
        args.uniform_delta = 0;  // src_off == dst_off for every piece
        CUDA_TRY(modk::launch_batch_inline(args, in, stream));
        g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    return MOD_OK;
}

// CEncryptionCycler::Cycle on a HOST buffer: slices travel H2D -> kernel -> D2H on kPipeSlots streams
// so that the upload of slice i+1, the kernel of slice i and the download of slice i-1 overlap.
int cycle_host(DeviceCtx& c, uint8_t* host, uint64_t len, int32_t key)
{
    std::lock_guard<std::mutex> lock(c.mu);
    uint64_t slice = env_u64("MOD_SLICE_BYTES", 16ull << 20);
    slice = std::max<uint64_t>(4096, slice & ~4095ull);
    if (len < slice * 2)  // small buffers: still use several slots so both directions overlap
        slice = std::max<uint64_t>(4096, ((len / kPipeSlots) + 4095) & ~4095ull);
    const int slots = (int)std::min<uint64_t>(kPipeSlots, (len + slice - 1) / slice);
    for (int i = 0; i < slots; ++i) {
        const int rc = grow(&c.slice_buf[i], &c.slice_bytes[i], slice);
        if (rc != MOD_OK)
            return rc;
    }
    const uint32_t k0 = modlcg::key_residue(key);
    int rc = MOD_OK;
    cudaError_t e = cudaSuccess;
    uint64_t pos = 0;
    // a long buffer that does not start on a 128-byte boundary gets a short first slice, so that every other
    // slice is copied between 128-byte aligned addresses (see kCopyAlign)
    const uint64_t head = len >= 4 * slice ? ((kCopyAlign - ((uintptr_t)host & (kCopyAlign - 1))) & (kCopyAlign - 1)) : 0;
    for (uint64_t i = 0; pos < len && rc == MOD_OK && e == cudaSuccess; ++i) {
        const int slot = (int)(i % kPipeSlots);
        const uint64_t n = i == 0 && head ? head : std::min(slice, len - pos);
        cudaStream_t s = c.pipe_stream[slot];
        uint8_t* d = (uint8_t*)c.slice_buf[slot];
        e = cudaMemcpyAsync(d, host + pos, n, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess)
            break;
        rc = launch_contiguous(d, d, n, (int32_t)modlcg::mulmod(k0, modlcg::pow_a(pos)), s);
        if (rc != MOD_OK)
            break;
        e = cudaMemcpyAsync(host + pos, d, n, cudaMemcpyDeviceToHost, s);
        pos += n;
    }
    const cudaError_t ed = drain(c);  // also on failure: the copies in flight touch the caller's buffer
    if (rc != MOD_OK)
        return rc;
    if (e == cudaSuccess)
        e = ed;
    if (e != cudaSuccess)
        return fail(MOD_ERR_CUDA, "mod_cycle: %s", cudaGetErrorString(e));
    return MOD_OK;
}

int validate_descs(const char* who, const mod_desc* descs, uint64_t n, uint64_t src_bytes, uint64_t dst_bytes)
{
    for (uint64_t i = 0; i < n; ++i) {
        const mod_desc& d = descs[i];
        if (d.src_off > src_bytes || (uint64_t)d.len > src_bytes - d.src_off)
            return fail(MOD_ERR_ARG, "%s: descriptor %llu: source range [%llu, +%u) leaves the %llu-byte buffer", who,
                        (unsigned long long)i, (unsigned long long)d.src_off, d.len, (unsigned long long)src_bytes);
        if (d.dst_off > dst_bytes || (uint64_t)d.len > dst_bytes - d.dst_off)
            return fail(MOD_ERR_ARG, "%s: descriptor %llu: destination range [%llu, +%u) leaves the %llu-byte buffer", who,
                        (unsigned long long)i, (unsigned long long)d.dst_off, d.len, (unsigned long long)dst_bytes);
    }
    return MOD_OK;
}

// (src_off - dst_off) & 15 when every non-empty descriptor agrees on it, else -1.
int32_t uniform_delta_of(const mod_desc* descs, uint64_t n)
{
    int32_t delta = -1;
    for (uint64_t i = 0; i < n; ++i) {
        if (!descs[i].len)
            continue;
        const int32_t d = (int32_t)((descs[i].src_off - descs[i].dst_off) & 15u);
        if (delta < 0)
            delta = d;
        else if (delta != d)
            return -1;
    }
    return delta;
}

// Expand (already validated) descriptors into device descriptors with their first-tile prefix.
int expand_descs(const mod_desc* descs, uint64_t n, uint32_t dst_align, modk::DevDesc* out, uint64_t* tiles_out,
                 uint64_t* payload_out)
{
    uint64_t tiles = 0, payload = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const mod_desc& d = descs[i];
        modk::DevDesc& o = out[i];
        o.src_off = d.src_off;
        o.dst_off = d.dst_off;
        o.len = d.len;
        o.key = d.key;
        o.first_tile = (uint32_t)tiles;
        o.neg_state = modlcg::key_to_neg_state(d.key);
        tiles += modk::tiles_for_entry((uint32_t)((dst_align + d.dst_off) & 15u), d.len);
        payload += d.len;
        if (tiles >= 0xFFFFFFFFull)
            return fail(MOD_ERR_ARG, "batch too large (tile count overflows 32 bits)");
    }
    *tiles_out = tiles;
    *payload_out = payload;
    return MOD_OK;
}

// ---- mod_cycle_batch on HOST buffers -------------------------------------------------------------------
//
// The entries are streamed in GROUPS of consecutive descriptors (~MOD_GROUP_BYTES of payload each;
// entries larger than that are first cut into pieces with jumped keys).  One plan (descriptors ->
// tile records) is built for the whole call, asynchronously on pipe stream 0.  Group g then uploads
// the source WINDOW its entries span into slot g % kPipeSlots, runs the batched kernel over its tile
// sub-range against the slot's two window buffers, and downloads the destination runs it covers --
// so the upload of one group, the kernel of another and the download of a third overlap, and HBM
// use is O(slots x group), not O(archive).  Only bytes covered by descriptors are written back, so
// untouched bytes of dst survive exactly like with the reference's per-entry fwrite / fread.
struct Group {
    uint64_t e0, e1;      // descriptor range
    uint32_t t0, t1;      // tile range
    uint64_t s_lo, s_hi;  // source window
    uint64_t d_lo, d_hi;  // destination window
};

int batch_host(DeviceCtx& c, const mod_desc* user_descs, uint64_t user_n, const uint8_t* src, uint64_t src_bytes,
               uint8_t* dst, uint64_t dst_bytes)
{
    const bool trace = env_u64("MOD_TRACE", 0) != 0;
    const double t_begin = now_ms();
    int rc = validate_descs("mod_cycle_batch", user_descs, user_n, src_bytes, dst_bytes);
    if (rc != MOD_OK)
        return rc;

    // the descriptor list is cut into groups of ~group_bytes of payload whose boundaries fall on aligned
    // destination addresses INSIDE entries (batch_cut.h); pieces continue their entry's keystream through
    // jumped keys.  The alignment is that of the host address when the caller's buffers allow aligned copies.
    const uint64_t group_bytes = std::max<uint64_t>(1 << 20, env_u64("MOD_GROUP_BYTES", 16ull << 20)) & ~(kCopyAlign - 1);
    const bool align_copies = (((uintptr_t)src | (uintptr_t)dst) & 15u) == 0u && env_u64("MOD_ALIGN_COPIES", 1) != 0;
    modcut::Cut cut;
    modcut::cut_into_groups(user_descs, user_n, group_bytes, align_copies ? (uint64_t)((uintptr_t)dst & (kCopyAlign - 1)) : 0,
                            align_copies ? kCopyAlign : 16, cut);
    const mod_desc* descs = cut.pieces.data();
    const uint64_t n = cut.pieces.size();
    if (n >= 0xFFFFFFFFull)
        return fail(MOD_ERR_ARG, "mod_cycle_batch: too many descriptors (%llu)", (unsigned long long)n);

    std::lock_guard<std::mutex> lock(c.mu);
    if ((rc = grow_pinned(&c.h_descs, &c.h_descs_bytes, n * sizeof(modk::DevDesc))) != MOD_OK)
        return rc;
    uint64_t plan_tiles = 0, plan_payload = 0;
    if ((rc = expand_descs(descs, n, 0, (modk::DevDesc*)c.h_descs, &plan_tiles, &plan_payload)) != MOD_OK)
        return rc;
    if (plan_tiles == 0)
        return MOD_OK;
    if ((rc = grow(&c.ws_descs, &c.ws_descs_bytes, n * sizeof(modk::DevDesc))) != MOD_OK)
        return rc;
    if ((rc = grow(&c.ws_tiles, &c.ws_tiles_bytes, plan_tiles * sizeof(modk::TileRec))) != MOD_OK)
        return rc;

    // groups of consecutive descriptors and the windows they span
    std::vector<Group> groups;
    auto whole = [&]() {
        Group all{0, n, 0, (uint32_t)plan_tiles, UINT64_MAX, 0, UINT64_MAX, 0};
        for (uint64_t i = 0; i < n; ++i) {
            if (!descs[i].len)
                continue;
            all.s_lo = std::min(all.s_lo, descs[i].src_off);
            all.s_hi = std::max(all.s_hi, descs[i].src_off + descs[i].len);
            all.d_lo = std::min(all.d_lo, descs[i].dst_off);
            all.d_hi = std::max(all.d_hi, descs[i].dst_off + descs[i].len);
        }
        groups.assign(1, all);
    };
    {
        Group g{0, 0, 0, 0, UINT64_MAX, 0, UINT64_MAX, 0};
        uint32_t tile = 0;
        for (uint64_t i = 0; i < n; ++i) {
            const mod_desc& d = descs[i];
            if (d.len) {
                g.s_lo = std::min(g.s_lo, d.src_off);
                g.s_hi = std::max(g.s_hi, d.src_off + d.len);
                g.d_lo = std::min(g.d_lo, d.dst_off);
                g.d_hi = std::max(g.d_hi, d.dst_off + d.len);
            }
            tile += modk::tiles_for_entry((uint32_t)(d.dst_off & 15u), d.len);
            if (cut.closes[i]) {
                g.e1 = i + 1;
                g.t1 = tile;
                if (g.t1 > g.t0)
                    groups.push_back(g);
                g = Group{i + 1, 0, tile, 0, UINT64_MAX, 0, UINT64_MAX, 0};
            }
        }
    }
    // If the entries are not laid out in order the windows overlap heavily and per-group copies would
    // move the buffers many times: one group over the full extents then.
    {
        uint64_t s_sum = 0, d_sum = 0;
        for (const Group& g : groups) {
            s_sum += g.s_hi - g.s_lo;
            d_sum += g.d_hi - g.d_lo;
        }
        if (s_sum > src_bytes + src_bytes / 4 + (1 << 20) || d_sum > dst_bytes + dst_bytes / 4 + (1 << 20))
            whole();
    }

    // Destination runs (maximal intervals downloaded with one copy) per group.  Two entries that are
    // neighbours in the GLOBAL destination order and less than 16 bytes apart (alignment padding) are
    // bridged into one run; the host bytes of such a gap are saved first and put back after the
    // download, so every byte not covered by a descriptor keeps its value.  A batch whose destination
    // is full of larger holes (more than 64 runs in a group) is handled exactly but without
    // pipelining: its whole destination extent makes a round trip through HBM.
    std::vector<uint32_t> rank(n, 0);   // position of each non-empty entry in global dst order
    std::vector<uint8_t> bridge_after;  // by rank: the gap to the next entry may be bridged
    {
        std::vector<uint32_t> order;
        order.reserve(n);
        bool monotone = true;
        uint64_t last = 0;
        for (uint64_t i = 0; i < n; ++i) {
            if (!descs[i].len)
                continue;
            if (descs[i].dst_off < last)
                monotone = false;
            last = descs[i].dst_off;
            order.push_back((uint32_t)i);
        }
        if (!monotone)
            std::sort(order.begin(), order.end(),
                      [&](uint32_t a, uint32_t b) { return descs[a].dst_off < descs[b].dst_off; });
        bridge_after.assign(order.size(), 0);
        for (size_t r = 0; r < order.size(); ++r) {
            rank[order[r]] = (uint32_t)r;
            if (r + 1 < order.size()) {
                const uint64_t end = descs[order[r]].dst_off + descs[order[r]].len;
                const uint64_t nxt = descs[order[r + 1]].dst_off;
                bridge_after[r] = (nxt >= end && nxt - end < 16) ? 1 : 0;
            }
        }
    }
    struct Gap {
        uint64_t off;
        uint32_t len;
        uint8_t bytes[15];
    };
    std::vector<Gap> gaps;
    std::vector<uint32_t> members;
    auto merged_runs = [&](const Group& g, std::vector<std::pair<uint64_t, uint64_t>>& runs, bool save_gaps) {
        runs.clear();
        members.clear();
        for (uint64_t i = g.e0; i < g.e1; ++i)
            if (descs[i].len)
                members.push_back((uint32_t)i);
        std::sort(members.begin(), members.end(), [&](uint32_t a, uint32_t b) { return rank[a] < rank[b]; });
        uint32_t prev_rank = 0;
        for (uint32_t idx : members) {
            const uint64_t b0 = descs[idx].dst_off, b1 = b0 + descs[idx].len;
            const bool adjacent = !runs.empty() && rank[idx] == prev_rank + 1;
            if (adjacent && b0 <= runs.back().second) {
                runs.back().second = std::max(runs.back().second, b1);
            } else if (adjacent && bridge_after[prev_rank] && b0 - runs.back().second < 16) {
                if (save_gaps && b0 > runs.back().second) {
                    Gap gap;
                    gap.off = runs.back().second;
                    gap.len = (uint32_t)(b0 - runs.back().second);
                    std::memcpy(gap.bytes, dst + gap.off, gap.len);
                    gaps.push_back(gap);
                }
                runs.back().second = b1;
            } else {
                runs.emplace_back(b0, b1);
            }
            prev_rank = rank[idx];
        }
    };
    std::vector<std::pair<uint64_t, uint64_t>> runs;
    bool holes = false;
    for (const Group& g : groups) {
        merged_runs(g, runs, false);
        if (runs.size() > 64) {
            holes = true;
            break;
        }
    }
    if (holes)
        whole();

    // slot buffers: the source window keeps its (offset & 15) phase and the destination window starts
    // at a 16-byte boundary of the destination space, so host co-alignment survives on the device.
    // Beyond that, pinned <-> HBM copies only run at full speed when both addresses are 128-byte aligned
    // (tools/copy_align_probe.py: 47 GB/s each way against 41 at any smaller phase), and groups of
    // byte-packed entries start anywhere: with 16-byte aligned caller buffers a window therefore sits at the
    // phase (host address & 127) in its slot, uploads are widened to 128-byte boundaries of the host address
    // (a few source bytes more) and downloads are split into an aligned body and up to two short ends.
    const bool split_downloads = env_u64("MOD_SPLIT_DOWNLOADS", 1) != 0;
    const int slots = (int)std::min<size_t>(kPipeSlots, groups.size());
    {
        uint64_t s_need = 0, d_need = 0;
        for (const Group& g : groups) {
            s_need = std::max<uint64_t>(s_need, (g.s_lo & 15u) + (g.s_hi - g.s_lo) + 3 * kCopyAlign);
            d_need = std::max<uint64_t>(d_need, g.d_hi - (g.d_lo & ~15ull) + kCopyAlign);
        }
        for (int k = 0; k < slots; ++k) {
            if ((rc = grow(&c.slot_src[k], &c.slot_src_bytes[k], s_need)) != MOD_OK)
                return rc;
            if ((rc = grow(&c.slot_dst[k], &c.slot_dst_bytes[k], d_need)) != MOD_OK)
                return rc;
        }
    }

    cudaError_t e = cudaMemcpyAsync(c.ws_descs, c.h_descs, n * sizeof(modk::DevDesc), cudaMemcpyHostToDevice, c.pipe_stream[0]);
    if (e == cudaSuccess) {
        e = modk::launch_build_tiles((const modk::DevDesc*)c.ws_descs, (uint32_t)n, 0, (modk::TileRec*)c.ws_tiles,
                                     (uint32_t)plan_tiles, c.pipe_stream[0]);
        g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    if (e == cudaSuccess)
        e = cudaEventRecord(c.plan_ready, c.pipe_stream[0]);
    const modk::TileRec* d_tiles = (const modk::TileRec*)c.ws_tiles;
    const int32_t uniform_delta = uniform_delta_of(descs, n);
    const double t_plan = now_ms();

    // test hook (tests/test_gpu_multidev.py): pretend the runtime failed at this group, with earlier
    // groups still in flight, to exercise the drain-before-return path
    const uint64_t fail_group = env_u64("MOD_TEST_FAIL_GROUP", UINT64_MAX);
    for (size_t gi = 0; gi < groups.size() && e == cudaSuccess; ++gi) {
        if (gi == fail_group) {
            e = cudaErrorUnknown;
            break;
        }
        const Group& g = groups[gi];
        const int k = (int)(gi % (size_t)slots);
        cudaStream_t s = c.pipe_stream[k];
        const uint64_t d_lo16 = g.d_lo & ~15ull;
        // uploaded source bytes [up_lo, up_hi) >= [s_lo, s_hi); address of source byte s_lo / destination byte d_lo16
        uint64_t up_lo = g.s_lo, up_hi = g.s_hi;
        uint8_t* win_src = (uint8_t*)c.slot_src[k] + (g.s_lo & 15u);
        uint8_t* win_dst = (uint8_t*)c.slot_dst[k];
        if (align_copies) {
            up_lo -= std::min<uint64_t>(g.s_lo, (uintptr_t)(src + g.s_lo) & (kCopyAlign - 1));
            up_hi = std::min<uint64_t>(src_bytes, g.s_hi + ((kCopyAlign - ((uintptr_t)(src + g.s_hi) & (kCopyAlign - 1))) & (kCopyAlign - 1)));
            win_src = (uint8_t*)c.slot_src[k] + ((uintptr_t)(src + up_lo) & (kCopyAlign - 1)) + (g.s_lo - up_lo);
            win_dst = (uint8_t*)c.slot_dst[k] + ((uintptr_t)(dst + d_lo16) & (kCopyAlign - 1));
        }
        e = cudaMemcpyAsync(win_src - (g.s_lo - up_lo), src + up_lo, up_hi - up_lo, cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess && holes)
            e = cudaMemcpyAsync(win_dst, dst + d_lo16, g.d_hi - d_lo16, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess)
            break;
        if (!holes)
            merged_runs(g, runs, true);
        if (gi > 0 && gi < (size_t)slots) {  // first use of this stream: the plan must be complete
            e = cudaStreamWaitEvent(s, c.plan_ready, 0);
            if (e != cudaSuccess)
                break;
        }
        modk::BatchArgs args;
        args.src = win_src - g.s_lo;  // virtual bases: base + offset lands inside the window
        args.dst = win_dst - d_lo16;
        args.tiles = d_tiles + g.t0;
        args.n_tiles = g.t1 - g.t0;
        args.tiles_per_entry = 0;
        args.src_lo16 = ((uint64_t)(uintptr_t)(win_src - (g.s_lo - up_lo)) + 15u) & ~15ull;
        args.src_hi16 = ((uint64_t)(uintptr_t)(win_src + (up_hi - g.s_lo))) & ~15ull;
        args.uniform_delta = uniform_delta;
        e = modk::launch_batch(args, s);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (e != cudaSuccess)
            break;
        if (holes) {
            e = cudaMemcpyAsync(dst + d_lo16, win_dst, g.d_hi - d_lo16, cudaMemcpyDeviceToHost, s);
        } else {
            for (const auto& r : runs) {
                // cut points: the run's ends and, for a long run, the 128-byte boundaries just inside them
                uint64_t cut[4] = {r.first, r.first, r.second, r.second};
                if (align_copies && split_downloads && r.second - r.first >= (64u << 10)) {
                    cut[1] = r.first + ((kCopyAlign - ((uintptr_t)(dst + r.first) & (kCopyAlign - 1))) & (kCopyAlign - 1));
                    cut[2] = r.second - ((uintptr_t)(dst + r.second) & (kCopyAlign - 1));
                }
                for (int q = 0; q < 3 && e == cudaSuccess; ++q)
                    if (cut[q + 1] > cut[q])
                        e = cudaMemcpyAsync(dst + cut[q], win_dst + (cut[q] - d_lo16), cut[q + 1] - cut[q],
                                            cudaMemcpyDeviceToHost, s);
                if (e != cudaSuccess)
                    break;
            }
        }
    }
    const double t_enq = now_ms();
    const cudaError_t ed = drain(c);  // also on failure: the copies in flight touch the caller's buffers
    if (e == cudaSuccess)
        e = ed;
    if (e == cudaSuccess)
        for (const Gap& gap : gaps)  // put the padding bytes the bridged downloads ran over back
            std::memcpy(dst + gap.off, gap.bytes, gap.len);
    if (trace)
        fprintf(stderr, "[mod] cycle_batch dev %d: plan %.2f ms, enqueue %zu groups %.2f ms, drain %.2f ms\n", c.device,
                t_plan - t_begin, groups.size(), t_enq - t_plan, now_ms() - t_enq);
    if (e != cudaSuccess)
        return fail(MOD_ERR_CUDA, "mod_cycle_batch: %s", cudaGetErrorString(e));
    return MOD_OK;
}

// ---- in-process multi-GPU: one host thread + stream set per selected device --------------------------------

int selected_devices(uint64_t dev_mask, std::vector<int>& out)
{
    int count = 0;
    CUDA_TRY(cudaGetDeviceCount(&count));
    if (count <= 0)
        return fail(MOD_ERR_CUDA, "no CUDA device visible: this library has no CPU fallback");
    for (int d = 0; d < count && d < kMaxDevices; ++d)
        if (dev_mask == 0 || ((dev_mask >> d) & 1ull))
            out.push_back(d);
    if (out.empty())
        return fail(MOD_ERR_ARG, "dev_mask 0x%llx selects none of the %d visible devices", (unsigned long long)dev_mask, count);
    return MOD_OK;
}

// fn(rank, world, ctx) runs once per selected device, each on its own host thread bound to that
// device; the first failure (by rank) is reported with its message.
template <class F>
int for_each_device(uint64_t dev_mask, F fn)
{
    std::vector<int> devs;
    int rc = selected_devices(dev_mask, devs);
    if (rc != MOD_OK)
        return rc;
    const int world = (int)devs.size();
    std::vector<int> rcs((size_t)world, MOD_OK);
    std::vector<std::string> errs((size_t)world);
    auto body = [&](int r) {
        try {
            DeviceCtx* c = nullptr;
            int my = acquire(devs[(size_t)r], &c);
            if (my == MOD_OK)
                my = fn(r, world, *c);
            rcs[(size_t)r] = my;
        } catch (const std::bad_alloc&) {
            rcs[(size_t)r] = fail(MOD_ERR_NOMEM, "out of host memory");
        } catch (...) {
            rcs[(size_t)r] = fail(MOD_ERR_ARG, "unexpected exception");
        }
        if (rcs[(size_t)r] != MOD_OK)
            errs[(size_t)r] = tl_error;
    };
    if (world == 1) {  // on the calling thread; acquire() binds the device, so put the caller's back afterwards
        int prev = 0;
        CUDA_TRY(cudaGetDevice(&prev));
        body(0);
        cudaSetDevice(prev);
    } else {
        std::vector<std::thread> threads;
        threads.reserve((size_t)world);
        for (int r = 0; r < world; ++r)
            threads.emplace_back(body, r);
        for (std::thread& t : threads)
            t.join();
    }
    for (int r = 0; r < world; ++r) {
        if (rcs[(size_t)r] != MOD_OK) {
            tl_error = "device " + std::to_string(devs[(size_t)r]) + ": " + errs[(size_t)r];
            return rcs[(size_t)r];
        }
    }
    return MOD_OK;
}

}  // namespace

struct mod_plan {
    int device = -1;
    uint64_t n = 0;
    uint64_t src_bytes = 0;
    uint64_t dst_bytes = 0;
    uint32_t dst_align = 0;
    uint64_t payload = 0;
    uint32_t n_tiles = 0;
    int32_t uniform_delta = -1;  // (src_off - dst_off) & 15 if all entries agree: selects the co-aligned kernel
    modk::TileRec* d_tiles = nullptr;
    uint64_t d_tiles_bytes = 0;         // size of the pool block behind d_tiles
    modk::DevDesc* d_descs = nullptr;   // the descriptors in HBM: the search kernel reads a match's src_off there
    uint64_t d_descs_bytes = 0;
    std::vector<mod_desc> descs;        // host copy: window validation, tile ranges
    std::vector<uint32_t> first_tile;   // n + 1 entries
};

struct mod_pattern_set {
    int device = -1;
    modk::SetIndex* d_index = nullptr;  // filter bitmap and index, built on the host
    uint32_t n = 0;
    uint32_t n_keys = 0;  // distinct 2-byte keys of the patterns of length >= 2
    uint32_t lmin = 0, lmax = 0;
    bool fold = false;    // mod_pattern_set_create_nocase: upper-cased patterns, searched with find_set_kernel<true>
};

extern "C" {

int mod_abi_version(void) { return MOD_ABI_VERSION; }

const char* mod_last_error(void) { return tl_error.c_str(); }

uint64_t mod_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int mod_device_count(void)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(MOD_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    return count;
}

int mod_init(int device)
{
    DeviceCtx* c = nullptr;
    return acquire(device, &c);
}

int mod_current_device(void)
{
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    return cur;
}

int mod_is_device_pointer(const void* p)
{
    int dev = -1;
    return pointer_device(p, &dev) ? 1 : 0;
}

void mod_shutdown(void)
{
    std::lock_guard<std::mutex> init_lock(g_init_mu);
    int prev = -1;
    cudaGetDevice(&prev);
    for (int d = 0; d < kMaxDevices; ++d) {
        DeviceCtx& c = g_dev[d];
        if (!c.ready.load(std::memory_order_acquire))
            continue;
        std::lock_guard<std::mutex> lock(c.mu);
        if (cudaSetDevice(d) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        cudaDeviceSynchronize();
        release_ctx(c);
    }
    if (prev >= 0)
        cudaSetDevice(prev);
}

/* ---- memory helpers ------------------------------------------------------------------------ */

void* mod_host_alloc(uint64_t bytes)
{
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        fail(MOD_ERR_NOMEM, "cudaHostAlloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e));
        return nullptr;
    }
    return p;
}

int mod_host_free(void* p)
{
    if (!p)
        return MOD_OK;
    CUDA_TRY(cudaFreeHost(p));
    return MOD_OK;
}

void* mod_device_alloc(uint64_t bytes)
{
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        fail(MOD_ERR_NOMEM, "cudaMalloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e));
        return nullptr;
    }
    return p;
}

int mod_device_free(void* p)
{
    if (!p)
        return MOD_OK;
    CUDA_TRY(cudaFree(p));
    return MOD_OK;
}

int mod_memcpy_h2d(void* d_dst, const void* h_src, uint64_t bytes, void* stream)
{
    CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return MOD_OK;
}

int mod_memcpy_d2h(void* h_dst, const void* d_src, uint64_t bytes, void* stream)
{
    CUDA_TRY(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return MOD_OK;
}

int mod_stream_sync(void* stream)
{
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return MOD_OK;
}

void* mod_stream_create(void)
{
    DeviceCtx* c = nullptr;
    if (acquire(-1, &c) != MOD_OK)
        return nullptr;
    cudaStream_t s = nullptr;
    cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        cudaGetLastError();
        fail(MOD_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        return nullptr;
    }
    return (void*)s;
}

int mod_stream_destroy(void* stream)
{
    if (!stream)
        return MOD_OK;
    CUDA_TRY(cudaStreamDestroy((cudaStream_t)stream));
    return MOD_OK;
}

/* ---- CEncryptionCycler::Cycle ---------------------------------------------------------------- */

int32_t mod_key_jump(int32_t key, uint64_t pos)
{
    return (int32_t)modlcg::mulmod(modlcg::key_residue(key), modlcg::pow_a(pos));
}

int mod_cycle_device(const void* d_src, void* d_dst, uint64_t len, int32_t key, void* stream)
{
    if (len == 0)
        return MOD_OK;
    if (!d_src || !d_dst)
        return fail(MOD_ERR_ARG, "mod_cycle_device: null pointer");
    DeviceCtx* c = nullptr;
    int rc = acquire(-1, &c);
    if (rc != MOD_OK)
        return rc;
    return launch_contiguous((const uint8_t*)d_src, (uint8_t*)d_dst, len, key, (cudaStream_t)stream);
}

int mod_cycle(void* data, uint64_t len, int32_t key)
{
    MOD_ABI_BEGIN
    if (len == 0)
        return MOD_OK;
    if (!data)
        return fail(MOD_ERR_ARG, "mod_cycle: null pointer");
    int ptr_dev = -1;
    if (pointer_device(data, &ptr_dev)) {  // resident buffer: cycle it where it lives
        DeviceGuard guard;
        int rc = guard.enter(ptr_dev);
        if (rc != MOD_OK)
            return rc;
        DeviceCtx* c = nullptr;
        if ((rc = acquire(-1, &c)) != MOD_OK)
            return rc;
        if ((rc = launch_contiguous((const uint8_t*)data, (uint8_t*)data, len, key, nullptr)) != MOD_OK)
            return rc;
        CUDA_TRY(cudaStreamSynchronize(nullptr));
        return MOD_OK;
    }
    DeviceCtx* c = nullptr;
    int rc = acquire(-1, &c);
    if (rc != MOD_OK)
        return rc;
    return cycle_host(*c, (uint8_t*)data, len, key);
    MOD_ABI_END("mod_cycle")
}

int mod_cycle_sharded(void* data, uint64_t len, int32_t key, uint64_t dev_mask)
{
    MOD_ABI_BEGIN
    if (len == 0)
        return MOD_OK;
    if (!data)
        return fail(MOD_ERR_ARG, "mod_cycle_sharded: null pointer");
    int ptr_dev = -1;
    if (pointer_device(data, &ptr_dev))
        return fail(MOD_ERR_ARG, "mod_cycle_sharded: `data` must be a host buffer (a device buffer lives on one GPU: use mod_cycle)");
    uint8_t* host = (uint8_t*)data;
    return for_each_device(dev_mask, [=](int rank, int world, DeviceCtx& c) -> int {
        uint64_t b = 0, e = 0;
        int rc = mod_shard_range(len, rank, world, &b, &e);
        if (rc != MOD_OK || e <= b)
            return rc;
        return cycle_host(c, host + b, e - b, mod_key_jump(key, b));
    });
    MOD_ABI_END("mod_cycle_sharded")
}

/* ---- descriptor plans -------------------------------------------------------------------------- */

int mod_plan_create(const mod_desc* descs, uint64_t n, uint64_t src_bytes, uint64_t dst_bytes,
                    uint32_t dst_align, mod_plan** out)
{
    MOD_ABI_BEGIN
    if (!out)
        return fail(MOD_ERR_ARG, "mod_plan_create: out is null");
    *out = nullptr;
    if (n && !descs)
        return fail(MOD_ERR_ARG, "mod_plan_create: descs is null");
    if (n >= 0xFFFFFFFFull)
        return fail(MOD_ERR_ARG, "mod_plan_create: too many descriptors (%llu)", (unsigned long long)n);
    if (dst_align > 15)
        return fail(MOD_ERR_ARG, "mod_plan_create: dst_align must be < 16");
    DeviceCtx* c = nullptr;
    int rc = acquire(-1, &c);
    if (rc != MOD_OK)
        return rc;
    if ((rc = validate_descs("mod_plan_create", descs, n, src_bytes, dst_bytes)) != MOD_OK)
        return rc;

    std::vector<modk::DevDesc> host(n);
    uint64_t tiles = 0, payload = 0;
    if ((rc = expand_descs(descs, n, dst_align, host.data(), &tiles, &payload)) != MOD_OK)
        return rc;

    mod_plan* p = new mod_plan();
    p->device = c->device;
    p->n = n;
    p->src_bytes = src_bytes;
    p->dst_bytes = dst_bytes;
    p->dst_align = dst_align;
    p->payload = payload;
    p->n_tiles = (uint32_t)tiles;
    p->uniform_delta = uniform_delta_of(descs, n);
    auto cleanup = [&]() {
        pool_free(*c, p->d_descs, p->d_descs_bytes);
        pool_free(*c, p->d_tiles, p->d_tiles_bytes);
        delete p;
    };
    try {
        p->descs.assign(descs, descs + n);
        p->first_tile.resize(n + 1);
        for (uint64_t i = 0; i < n; ++i)
            p->first_tile[i] = host[i].first_tile;
        p->first_tile[n] = (uint32_t)tiles;
    } catch (...) {
        cleanup();
        throw;
    }
    if (n && tiles) {
        cudaError_t e = pool_alloc(*c, n * sizeof(modk::DevDesc), (void**)&p->d_descs, &p->d_descs_bytes);
        if (e == cudaSuccess)
            e = pool_alloc(*c, tiles * sizeof(modk::TileRec), (void**)&p->d_tiles, &p->d_tiles_bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            cleanup();
            return fail(MOD_ERR_NOMEM, "mod_plan_create: cudaMalloc failed: %s", cudaGetErrorString(e));
        }
        e = cudaMemcpy(p->d_descs, host.data(), n * sizeof(modk::DevDesc), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) {
            e = modk::launch_build_tiles(p->d_descs, (uint32_t)n, dst_align, p->d_tiles, p->n_tiles, nullptr);
            g_launches.fetch_add(1, std::memory_order_relaxed);
        }
        if (e == cudaSuccess)
            e = cudaStreamSynchronize(nullptr);
        if (e != cudaSuccess) {
            cleanup();
            return fail(MOD_ERR_CUDA, "mod_plan_create: %s", cudaGetErrorString(e));
        }
    }
    *out = p;
    return MOD_OK;
    MOD_ABI_END("mod_plan_create")
}

int mod_plan_destroy(mod_plan* plan)
{
    if (!plan)
        return MOD_OK;
    if (plan->d_tiles || plan->d_descs) {
        DeviceGuard guard;
        guard.enter(plan->device);
        cudaDeviceSynchronize();  // launches that still read the records finish first (what cudaFree used to guarantee)
        for (auto blk : {std::make_pair((void*)plan->d_tiles, plan->d_tiles_bytes), std::make_pair((void*)plan->d_descs, plan->d_descs_bytes)}) {
            if (plan->device >= 0 && plan->device < kMaxDevices)
                pool_free(g_dev[plan->device], blk.first, blk.second);  // back to the device's block pool
            else if (blk.first)
                cudaFree(blk.first);
        }
    }
    delete plan;
    return MOD_OK;
}

uint64_t mod_plan_payload_bytes(const mod_plan* plan) { return plan ? plan->payload : 0; }
uint64_t mod_plan_num_tiles(const mod_plan* plan) { return plan ? plan->n_tiles : 0; }

int mod_plan_tile_range(const mod_plan* plan, uint64_t entry_begin, uint64_t entry_end, uint64_t* tile_begin,
                        uint64_t* tile_end)
{
    if (!plan || !tile_begin || !tile_end)
        return fail(MOD_ERR_ARG, "mod_plan_tile_range: null argument");
    if (entry_begin > entry_end || entry_end > plan->n)
        return fail(MOD_ERR_ARG, "mod_plan_tile_range: entries [%llu, %llu) outside the plan's %llu",
                    (unsigned long long)entry_begin, (unsigned long long)entry_end, (unsigned long long)plan->n);
    *tile_begin = plan->first_tile[entry_begin];
    *tile_end = plan->first_tile[entry_end];
    return MOD_OK;
}

static int plan_check_device(const mod_plan* plan, const char* who)
{
    int cur = -1;
    CUDA_TRY(cudaGetDevice(&cur));
    if (cur != plan->device)
        return fail(MOD_ERR_ARG, "%s: the plan lives on device %d but the calling thread is bound to device %d", who,
                    plan->device, cur);
    return MOD_OK;
}

int mod_plan_run(const mod_plan* plan, const void* d_src, void* d_dst, void* stream)
{
    if (!plan)
        return fail(MOD_ERR_ARG, "mod_plan_run: null plan");
    if (plan->n_tiles == 0)
        return MOD_OK;
    if (!d_src || !d_dst)
        return fail(MOD_ERR_ARG, "mod_plan_run: null buffer");
    if (((uintptr_t)d_dst & 15u) != plan->dst_align)
        return fail(MOD_ERR_ALIGN, "mod_plan_run: dst & 15 is %u but the plan was built for %u",
                    (unsigned)((uintptr_t)d_dst & 15u), plan->dst_align);
    int rc = plan_check_device(plan, "mod_plan_run");
    if (rc != MOD_OK)
        return rc;
    modk::BatchArgs args;
    args.src = (const uint8_t*)d_src;
    args.dst = (uint8_t*)d_dst;
    args.tiles = plan->d_tiles;
    args.n_tiles = plan->n_tiles;
    args.tiles_per_entry = 0;
    args.src_lo16 = ((uint64_t)(uintptr_t)d_src + 15u) & ~15ull;
    args.src_hi16 = ((uint64_t)(uintptr_t)d_src + plan->src_bytes) & ~15ull;
    args.uniform_delta = plan->uniform_delta;
    CUDA_TRY(modk::launch_batch(args, (cudaStream_t)stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MOD_OK;
}

int mod_plan_run_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                        uint64_t src_win_off, uint64_t src_win_bytes, void* d_dst_win, uint64_t dst_win_off,
                        uint64_t dst_win_bytes, void* stream)
{
    if (!plan)
        return fail(MOD_ERR_ARG, "mod_plan_run_window: null plan");
    if (tile_begin > tile_end || tile_end > plan->n_tiles)
        return fail(MOD_ERR_ARG, "mod_plan_run_window: tiles [%llu, %llu) outside the plan's %u",
                    (unsigned long long)tile_begin, (unsigned long long)tile_end, plan->n_tiles);
    if (tile_begin == tile_end)
        return MOD_OK;
    if (!d_src_win || !d_dst_win)
        return fail(MOD_ERR_ARG, "mod_plan_run_window: null buffer");
    if ((((uintptr_t)d_dst_win - dst_win_off) & 15u) != plan->dst_align)
        return fail(MOD_ERR_ALIGN, "mod_plan_run_window: (d_dst_win - dst_win_off) & 15 is %u but the plan was built for %u",
                    (unsigned)(((uintptr_t)d_dst_win - dst_win_off) & 15u), plan->dst_align);
    int rc = plan_check_device(plan, "mod_plan_run_window");
    if (rc != MOD_OK)
        return rc;
    // every byte the tile range touches must lie inside the two windows
    const uint32_t* ft = plan->first_tile.data();
    uint64_t e = (uint64_t)(std::upper_bound(ft, ft + plan->n + 1, (uint32_t)tile_begin) - ft) - 1;
    for (; e < plan->n && ft[e] < tile_end; ++e) {
        const mod_desc& d = plan->descs[e];
        if (ft[e + 1] == ft[e])
            continue;  // empty entry
        const uint32_t h0 = (uint32_t)((plan->dst_align + d.dst_off) & 15u);
        const uint64_t ta = std::max<uint64_t>(tile_begin, ft[e]) - ft[e], tb = std::min<uint64_t>(tile_end, ft[e + 1]) - ft[e];
        const uint64_t b0 = ta == 0 ? 0 : ta * modk::kTileBytes - h0;
        const uint64_t b1 = std::min<uint64_t>(d.len, tb * modk::kTileBytes - h0);
        if (d.src_off + b0 < src_win_off || d.src_off + b1 > src_win_off + src_win_bytes)
            return fail(MOD_ERR_ARG, "mod_plan_run_window: entry %llu reads outside the source window", (unsigned long long)e);
        if (d.dst_off + b0 < dst_win_off || d.dst_off + b1 > dst_win_off + dst_win_bytes)
            return fail(MOD_ERR_ARG, "mod_plan_run_window: entry %llu writes outside the destination window", (unsigned long long)e);
    }
    modk::BatchArgs args;
    args.src = (const uint8_t*)d_src_win - src_win_off;  // virtual bases: base + offset lands inside the window
    args.dst = (uint8_t*)d_dst_win - dst_win_off;
    args.tiles = plan->d_tiles + tile_begin;
    args.n_tiles = (uint32_t)(tile_end - tile_begin);
    args.tiles_per_entry = 0;
    args.src_lo16 = ((uint64_t)(uintptr_t)d_src_win + 15u) & ~15ull;
    args.src_hi16 = ((uint64_t)(uintptr_t)d_src_win + src_win_bytes) & ~15ull;
    args.uniform_delta = plan->uniform_delta;
    CUDA_TRY(modk::launch_batch(args, (cudaStream_t)stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MOD_OK;
}

// Checks shared by every search launch: the result buffers, the chunk grid on the source, the device.  `src_base`
// is the virtual base (source byte 0 of the plan's space).
static int find_check(const char* who, const mod_plan* plan, const uint8_t* src_base, const void* d_counts, const void* d_total,
                      uint64_t cap, const void* d_matches)
{
    if (!d_counts || !d_total || (cap && !d_matches))
        return fail(MOD_ERR_ARG, "%s: null result buffer", who);
    // the search kernels need the chunk grid on the source: src_off - dst_off == delta for every entry and
    // base + delta - dst_align == 0 (mod 16)
    if (plan->uniform_delta < 0 || (((uintptr_t)src_base + (uintptr_t)plan->uniform_delta - plan->dst_align) & 15u) != 0u)
        return fail(MOD_ERR_ALIGN, "%s: the plan's chunk grid does not lie on the source (build it with dst_off == src_off "
                    "and dst_align == source address & 15)", who);
    return plan_check_device(plan, who);
}

// Checks shared by the windowed searches: the tile range, the buffer, and that every byte the tiles read -- the up
// to `halo` bytes past a tile that a match starting in it may cover included -- lies inside the window.
static int find_window_check(const char* who, const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                             uint64_t src_win_off, uint64_t src_win_bytes, uint32_t halo)
{
    if (tile_begin > tile_end || tile_end > plan->n_tiles)
        return fail(MOD_ERR_ARG, "%s: tiles [%llu, %llu) outside the plan's %u", who, (unsigned long long)tile_begin,
                    (unsigned long long)tile_end, plan->n_tiles);
    if (tile_begin < tile_end && !d_src_win)
        return fail(MOD_ERR_ARG, "%s: null buffer", who);
    const uint32_t* ft = plan->first_tile.data();
    uint64_t e = tile_begin < tile_end ? (uint64_t)(std::upper_bound(ft, ft + plan->n + 1, (uint32_t)tile_begin) - ft) - 1 : plan->n;
    for (; e < plan->n && ft[e] < tile_end; ++e) {
        const mod_desc& d = plan->descs[e];
        if (ft[e + 1] == ft[e])
            continue;  // empty entry
        const uint32_t h0 = (uint32_t)((plan->dst_align + d.dst_off) & 15u);
        const uint64_t ta = std::max<uint64_t>(tile_begin, ft[e]) - ft[e], tb = std::min<uint64_t>(tile_end, ft[e + 1]) - ft[e];
        const uint64_t b0 = ta == 0 ? 0 : ta * modk::kTileBytes - h0;
        const uint64_t b1 = std::min<uint64_t>(d.len, tb * modk::kTileBytes - h0 + halo);
        if (d.src_off + b0 < src_win_off || d.src_off + b1 > src_win_off + src_win_bytes)
            return fail(MOD_ERR_ARG, "%s: entry %llu reads outside the source window", who, (unsigned long long)e);
    }
    return MOD_OK;
}

// The mask checks of the masked searches: a mask with a byte to anchor on, `len` within 1..kMaxPattern.
static int masked_check(const char* who, const uint8_t* pattern, const uint8_t* mask, uint32_t len)
{
    if (!pattern || !mask || len == 0 || len > modk::kMaxPattern)
        return fail(MOD_ERR_ARG, "%s: the pattern and its mask must be 1 to %u bytes", who, modk::kMaxPattern);
    for (uint32_t k = 0; k < len; ++k)
        if (mask[k])
            return MOD_OK;
    return fail(MOD_ERR_ARG, "%s: the mask is all zero (no byte to anchor on)", who);
}

// The anchor of a masked pattern: the adjacent pair (a, a + 1) with the most mask bits, the first of equals (0 if
// len == 1).
static uint32_t find_anchor(const uint8_t* mask, uint32_t len)
{
    uint32_t a = 0;
    int best = -1;
    for (uint32_t k = 0; k + 1 < len; ++k) {
        const int bits = __builtin_popcount(mask[k]) + __builtin_popcount(mask[k + 1]);
        if (bits > best) {
            best = bits;
            a = k;
        }
    }
    return a;
}

// The launch shared by mod_plan_find*, mod_plan_find_masked*; [lo16, hi16) are the granules that may be loaded whole.
// `mask` (len bytes, checked by masked_check) or nullptr: the exact search.  An all-0xFF mask is the exact search too.
static int plan_find_launch(const char* who, const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end,
                            const uint8_t* src_base, uint64_t lo16, uint64_t hi16, const uint8_t* pattern, const uint8_t* mask,
                            uint32_t len, uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream)
{
    if (!pattern || len == 0 || len > modk::kMaxPattern)
        return fail(MOD_ERR_ARG, "%s: the pattern must be 1 to %u bytes", who, modk::kMaxPattern);
    if (tile_begin == tile_end)
        return MOD_OK;
    int rc = find_check(who, plan, src_base, d_counts, d_total, cap, d_matches);
    if (rc != MOD_OK)
        return rc;
    uint8_t v[modk::kMaxPattern];
    if (mask) {
        bool exact = true;
        for (uint32_t k = 0; k < len; ++k) {
            v[k] = pattern[k] & mask[k];
            exact = exact && mask[k] == 0xFFu;
        }
        pattern = v;
        if (exact)
            mask = nullptr;
    }
    modk::FindArgs f;
    f.src = src_base;
    f.tiles = plan->d_tiles + tile_begin;
    f.descs = plan->d_descs;
    f.n_tiles = (uint32_t)(tile_end - tile_begin);
    f.src_lo16 = lo16;
    f.src_hi16 = hi16;
    f.counts = d_counts;
    f.matches = (uint2*)d_matches;
    f.total = (unsigned long long*)d_total;
    f.cap = cap;
    f.len = len;
    f.head_word = 0;
    f.head_mask = 0;
    for (uint32_t k = 0; k < 4 && k < len; ++k) {
        f.head_word |= (uint32_t)pattern[k] << (8 * k);
        f.head_mask |= 0xFFu << (8 * k);
    }
    f.rep0 = 0x01010101u * pattern[0];
    f.rep1 = len > 1 ? 0x01010101u * pattern[1] : 0u;
    std::memset(f.pattern, 0, sizeof(f.pattern));
    std::memcpy(f.pattern, pattern, len);
    f.anchor = 0;
    f.mrep0 = f.mrep1 = 0;
    std::memset(f.mask, 0, sizeof(f.mask));
    if (mask) {
        const uint32_t a = find_anchor(mask, len);
        f.anchor = a;
        f.head_mask = 0;
        for (uint32_t k = 0; k < 4 && k < len; ++k)
            f.head_mask |= (uint32_t)mask[k] << (8 * k);
        f.rep0 = 0x01010101u * pattern[a];
        f.mrep0 = 0x01010101u * mask[a];
        f.rep1 = len > 1 ? 0x01010101u * pattern[a + 1] : 0u;
        f.mrep1 = len > 1 ? 0x01010101u * mask[a + 1] : 0u;
        std::memcpy(f.mask, mask, len);
    }
    CUDA_TRY(modk::launch_find(f, mask != nullptr, (cudaStream_t)stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MOD_OK;
}

int mod_plan_find(const mod_plan* plan, const void* d_src, const uint8_t* pattern, uint32_t len, uint32_t* d_counts,
                  mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream)
{
    if (!plan)
        return fail(MOD_ERR_ARG, "mod_plan_find: null plan");
    if (!d_src && plan->n_tiles)
        return fail(MOD_ERR_ARG, "mod_plan_find: null buffer");
    return plan_find_launch("mod_plan_find", plan, 0, plan->n_tiles, (const uint8_t*)d_src,
                            ((uint64_t)(uintptr_t)d_src + 15u) & ~15ull, ((uint64_t)(uintptr_t)d_src + plan->src_bytes) & ~15ull,
                            pattern, nullptr, len, d_counts, d_matches, cap, d_total, stream);
}

// The body of mod_plan_find_window and mod_plan_find_masked_window (mask: nullptr for the exact search).
static int plan_find_window(const char* who, const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                            uint64_t src_win_off, uint64_t src_win_bytes, const uint8_t* pattern, const uint8_t* mask,
                            uint32_t len, uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream)
{
    int rc = find_window_check(who, plan, tile_begin, tile_end, d_src_win, src_win_off, src_win_bytes, len - 1);
    if (rc != MOD_OK)
        return rc;
    return plan_find_launch(who, plan, tile_begin, tile_end, (const uint8_t*)d_src_win - src_win_off,
                            ((uint64_t)(uintptr_t)d_src_win + 15u) & ~15ull,
                            ((uint64_t)(uintptr_t)d_src_win + src_win_bytes) & ~15ull, pattern, mask, len, d_counts, d_matches,
                            cap, d_total, stream);
}

int mod_plan_find_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                         uint64_t src_win_off, uint64_t src_win_bytes, const uint8_t* pattern, uint32_t len,
                         uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream)
{
    if (!plan)
        return fail(MOD_ERR_ARG, "mod_plan_find_window: null plan");
    if (!pattern || len == 0 || len > modk::kMaxPattern)
        return fail(MOD_ERR_ARG, "mod_plan_find_window: the pattern must be 1 to %u bytes", modk::kMaxPattern);
    return plan_find_window("mod_plan_find_window", plan, tile_begin, tile_end, d_src_win, src_win_off, src_win_bytes, pattern,
                            nullptr, len, d_counts, d_matches, cap, d_total, stream);
}

int mod_plan_find_masked(const mod_plan* plan, const void* d_src, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                         uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream)
{
    if (!plan)
        return fail(MOD_ERR_ARG, "mod_plan_find_masked: null plan");
    if (!d_src && plan->n_tiles)
        return fail(MOD_ERR_ARG, "mod_plan_find_masked: null buffer");
    const int rc = masked_check("mod_plan_find_masked", pattern, mask, len);
    if (rc != MOD_OK)
        return rc;
    return plan_find_launch("mod_plan_find_masked", plan, 0, plan->n_tiles, (const uint8_t*)d_src,
                            ((uint64_t)(uintptr_t)d_src + 15u) & ~15ull, ((uint64_t)(uintptr_t)d_src + plan->src_bytes) & ~15ull,
                            pattern, mask, len, d_counts, d_matches, cap, d_total, stream);
}

int mod_plan_find_masked_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                                uint64_t src_win_off, uint64_t src_win_bytes, const uint8_t* pattern, const uint8_t* mask,
                                uint32_t len, uint32_t* d_counts, mod_match* d_matches, uint64_t cap, uint64_t* d_total,
                                void* stream)
{
    if (!plan)
        return fail(MOD_ERR_ARG, "mod_plan_find_masked_window: null plan");
    const int rc = masked_check("mod_plan_find_masked_window", pattern, mask, len);
    if (rc != MOD_OK)
        return rc;
    return plan_find_window("mod_plan_find_masked_window", plan, tile_begin, tile_end, d_src_win, src_win_off, src_win_bytes,
                            pattern, mask, len, d_counts, d_matches, cap, d_total, stream);
}

// Plan + one search launch + destroy, synchronous: the body of mod_find_batch and mod_find_set_batch.  One device
// allocation holds the total, the counts per descriptor, `aux_bytes` of counts per pattern and a list of `cap`
// records of `rec` bytes; `launch(plan, d_counts, d_aux, d_list, d_total)` enqueues the search on the legacy
// stream.  Everything comes back but the list order, which the caller sorts.
extern "C++" {  // a template cannot have C linkage
template <class Launch>
static int find_batch_run(const char* who, const mod_desc* descs, uint64_t n, const void* d_src, uint64_t src_bytes,
                          uint32_t* counts_out, void* aux_out, uint64_t aux_bytes, void* matches_out, uint64_t rec,
                          uint64_t cap, uint64_t* total_out, Launch launch)
{
    if ((n && (!descs || !counts_out)) || !total_out || (cap && !matches_out) || (aux_bytes && !aux_out))
        return fail(MOD_ERR_ARG, "%s: null argument", who);
    int src_dev = -1;
    if (!d_src || !pointer_device(d_src, &src_dev))
        return fail(MOD_ERR_ARG, "%s: d_src must be device memory (stream host data with CArk::FindInFiles)", who);
    DeviceGuard guard;
    int rc = guard.enter(src_dev);
    if (rc != MOD_OK)
        return rc;
    std::vector<mod_desc> own(descs, descs + n);
    for (mod_desc& d : own)
        d.dst_off = d.src_off;
    mod_plan* plan = nullptr;
    if ((rc = mod_plan_create(own.data(), n, src_bytes, src_bytes, (uint32_t)((uintptr_t)d_src & 15u), &plan)) != MOD_OK)
        return rc;
    // one allocation: total, counts, counts per pattern, list
    const uint64_t counts_at = 16, aux_at = (counts_at + 4 * n + 15) & ~15ull, list_at = (aux_at + aux_bytes + 15) & ~15ull,
                   bytes = list_at + rec * cap;
    uint8_t* d_out = nullptr;
    cudaError_t e = cudaMalloc((void**)&d_out, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        mod_plan_destroy(plan);
        return fail(MOD_ERR_NOMEM, "%s: cudaMalloc(%llu): %s", who, (unsigned long long)bytes, cudaGetErrorString(e));
    }
    e = cudaMemsetAsync(d_out, 0, list_at, nullptr);
    if (e == cudaSuccess)
        rc = launch(plan, (uint32_t*)(d_out + counts_at), d_out + aux_at, d_out + list_at, (uint64_t*)d_out);
    uint64_t total = 0;
    if (e == cudaSuccess && rc == MOD_OK)
        e = cudaMemcpyAsync(&total, d_out, 8, cudaMemcpyDeviceToHost, nullptr);
    if (e == cudaSuccess && rc == MOD_OK && n)
        e = cudaMemcpyAsync(counts_out, d_out + counts_at, 4 * n, cudaMemcpyDeviceToHost, nullptr);
    if (e == cudaSuccess && rc == MOD_OK && aux_bytes)
        e = cudaMemcpyAsync(aux_out, d_out + aux_at, aux_bytes, cudaMemcpyDeviceToHost, nullptr);
    if (e == cudaSuccess && rc == MOD_OK)
        e = cudaStreamSynchronize(nullptr);
    const uint64_t kept = std::min(total, cap);
    if (e == cudaSuccess && rc == MOD_OK && kept)
        e = cudaMemcpyAsync(matches_out, d_out + list_at, rec * kept, cudaMemcpyDeviceToHost, nullptr);
    if (e == cudaSuccess && rc == MOD_OK)
        e = cudaStreamSynchronize(nullptr);
    cudaFree(d_out);
    mod_plan_destroy(plan);
    if (rc != MOD_OK)
        return rc;
    CUDA_TRY(e);
    *total_out = total;
    return MOD_OK;
}
}

int mod_find_batch(const mod_desc* descs, uint64_t n, const void* d_src, uint64_t src_bytes, const uint8_t* pattern,
                   uint32_t len, uint32_t* counts_out, mod_match* matches_out, uint64_t cap, uint64_t* total_out)
{
    MOD_ABI_BEGIN
    if (!pattern || len == 0 || len > modk::kMaxPattern)
        return fail(MOD_ERR_ARG, "mod_find_batch: the pattern must be 1 to %u bytes", modk::kMaxPattern);
    const int rc = find_batch_run("mod_find_batch", descs, n, d_src, src_bytes, counts_out, nullptr, 0, matches_out, 8, cap,
                                  total_out, [&](mod_plan* plan, uint32_t* d_counts, uint8_t*, uint8_t* d_list, uint64_t* d_total) {
                                      return mod_plan_find(plan, d_src, pattern, len, d_counts, (mod_match*)d_list, cap, d_total,
                                                           nullptr);
                                  });
    if (rc != MOD_OK)
        return rc;
    std::sort(matches_out, matches_out + std::min(*total_out, cap),
              [](const mod_match& a, const mod_match& b) { return a.desc != b.desc ? a.desc < b.desc : a.pos < b.pos; });
    return MOD_OK;
    MOD_ABI_END("mod_find_batch")
}

int mod_find_masked_batch(const mod_desc* descs, uint64_t n, const void* d_src, uint64_t src_bytes, const uint8_t* pattern,
                          const uint8_t* mask, uint32_t len, uint32_t* counts_out, mod_match* matches_out, uint64_t cap,
                          uint64_t* total_out)
{
    MOD_ABI_BEGIN
    int rc = masked_check("mod_find_masked_batch", pattern, mask, len);
    if (rc != MOD_OK)
        return rc;
    rc = find_batch_run("mod_find_masked_batch", descs, n, d_src, src_bytes, counts_out, nullptr, 0, matches_out, 8, cap,
                        total_out, [&](mod_plan* plan, uint32_t* d_counts, uint8_t*, uint8_t* d_list, uint64_t* d_total) {
                            return mod_plan_find_masked(plan, d_src, pattern, mask, len, d_counts, (mod_match*)d_list, cap,
                                                        d_total, nullptr);
                        });
    if (rc != MOD_OK)
        return rc;
    std::sort(matches_out, matches_out + std::min(*total_out, cap),
              [](const mod_match& a, const mod_match& b) { return a.desc != b.desc ? a.desc < b.desc : a.pos < b.pos; });
    return MOD_OK;
    MOD_ABI_END("mod_find_masked_batch")
}

/* ---- pattern sets ------------------------------------------------------------------------------ */

// The body of mod_pattern_set_create and mod_pattern_set_create_nocase.  A folded set (`fold`) keeps every pattern
// upper-cased (modk::fold_ascii) and sets the filter bit of every case variant of its first two bytes.
static int pattern_set_create(const char* who, const uint8_t* bytes, const uint32_t* lens, uint32_t n, bool fold,
                              mod_pattern_set** out)
{
    if (!out)
        return fail(MOD_ERR_ARG, "%s: out is null", who);
    *out = nullptr;
    if (!bytes || !lens || n == 0 || n > modk::kMaxSetPatterns)
        return fail(MOD_ERR_ARG, "%s: a set holds 1 to %u patterns", who, modk::kMaxSetPatterns);
    std::vector<std::string> pats(n);
    uint64_t at = 0;
    for (uint32_t j = 0; j < n; ++j) {
        if (lens[j] == 0 || lens[j] > modk::kMaxPattern)
            return fail(MOD_ERR_ARG, "%s: pattern %u is %u bytes, not 1 to %u", who, j, lens[j], modk::kMaxPattern);
        pats[j].assign((const char*)bytes + at, lens[j]);
        at += lens[j];
        if (fold)
            for (char& ch : pats[j])
                ch = (char)modk::fold_ascii((uint8_t)ch);
    }
    std::vector<uint32_t> order(n);
    for (uint32_t j = 0; j < n; ++j)
        order[j] = j;
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return pats[a] != pats[b] ? pats[a] < pats[b] : a < b; });
    for (uint32_t j = 1; j < n; ++j)
        if (pats[order[j]] == pats[order[j - 1]])
            return fail(MOD_ERR_ARG, fold ? "%s: patterns %u and %u are the same ignoring case" : "%s: patterns %u and %u are the same",
                        who, order[j - 1], order[j]);

    // the index: filter bits, the length-1 table, and the longer patterns sorted by their 2-byte key
    std::unique_ptr<modk::SetIndex> idx(new modk::SetIndex());
    std::memset(idx.get(), 0, sizeof(modk::SetIndex));
    auto key_of = [&](uint32_t j) { return (uint32_t)(uint8_t)pats[j][0] | ((uint32_t)(uint8_t)pats[j][1] << 8); };
    std::vector<uint32_t> longer;
    uint32_t lmin = modk::kMaxPattern, lmax = 1;
    for (uint32_t j = 0; j < n; ++j) {
        lmin = std::min(lmin, lens[j]);
        lmax = std::max(lmax, lens[j]);
        const uint32_t b0 = (uint8_t)pats[j][0];
        // the case variants of a folded byte: itself, and its lower case if it is a letter
        const uint32_t v0 = fold && b0 - 0x41u < 26u ? b0 | 0x20u : b0;
        if (lens[j] == 1) {
            idx->one[b0] = (uint16_t)(j + 1);
            for (uint32_t b1 = 0; b1 < 256; ++b1) {
                idx->bitmap[(b0 | b1 << 8) >> 5] |= 1u << ((b0 | b1 << 8) & 31u);
                idx->bitmap[(v0 | b1 << 8) >> 5] |= 1u << ((v0 | b1 << 8) & 31u);
            }
        } else {
            const uint32_t b1 = (uint8_t)pats[j][1], v1 = fold && b1 - 0x41u < 26u ? b1 | 0x20u : b1;
            for (uint32_t k : {b0 | b1 << 8, v0 | b1 << 8, b0 | v1 << 8, v0 | v1 << 8})
                idx->bitmap[k >> 5] |= 1u << (k & 31u);
            longer.push_back(j);
        }
    }
    std::sort(longer.begin(), longer.end(), [&](uint32_t a, uint32_t b) { return key_of(a) != key_of(b) ? key_of(a) < key_of(b) : a < b; });
    uint32_t n_keys = 0;
    for (uint32_t r = 0; r < longer.size(); ++r) {
        const uint32_t j = longer[r];
        if (r == 0 || key_of(j) != key_of(longer[r - 1])) {
            idx->keys[n_keys] = (uint16_t)key_of(j);
            idx->group[n_keys++] = (uint16_t)r;
        }
        modk::SetPattern& sp = idx->pat[r];
        sp.id = j;
        sp.len = lens[j];
        for (uint32_t k = 0; k < 4 && k < lens[j]; ++k) {
            sp.head |= (uint32_t)(uint8_t)pats[j][k] << (8 * k);
            sp.mask |= 0xFFu << (8 * k);
        }
        std::memcpy(idx->bytes[r], pats[j].data(), lens[j]);
    }
    idx->group[n_keys] = (uint16_t)longer.size();

    DeviceCtx* c = nullptr;
    int rc = acquire(-1, &c);
    if (rc != MOD_OK)
        return rc;
    modk::SetIndex* d_idx = nullptr;
    CUDA_TRY(cudaMalloc((void**)&d_idx, sizeof(modk::SetIndex)));
    cudaError_t e = cudaMemcpyAsync(d_idx, idx.get(), sizeof(modk::SetIndex), cudaMemcpyHostToDevice, nullptr);
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(nullptr);
    if (e != cudaSuccess) {
        cudaFree(d_idx);
        return fail(MOD_ERR_CUDA, "%s: %s", who, cudaGetErrorString(e));
    }
    mod_pattern_set* set = new mod_pattern_set();
    set->device = c->device;
    set->d_index = d_idx;
    set->n = n;
    set->n_keys = n_keys;
    set->lmin = lmin;
    set->lmax = lmax;
    set->fold = fold;
    *out = set;
    return MOD_OK;
}

int mod_pattern_set_create(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out)
{
    MOD_ABI_BEGIN
    return pattern_set_create("mod_pattern_set_create", bytes, lens, n, false, out);
    MOD_ABI_END("mod_pattern_set_create")
}

int mod_pattern_set_create_nocase(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out)
{
    MOD_ABI_BEGIN
    return pattern_set_create("mod_pattern_set_create_nocase", bytes, lens, n, true, out);
    MOD_ABI_END("mod_pattern_set_create_nocase")
}

int mod_pattern_set_destroy(mod_pattern_set* set)
{
    if (!set)
        return MOD_OK;
    if (set->d_index) {
        DeviceGuard guard;
        guard.enter(set->device);
        cudaDeviceSynchronize();  // launches that still read the index finish first
        cudaFree(set->d_index);
    }
    delete set;
    return MOD_OK;
}

// The launch shared by mod_plan_find_set and mod_plan_find_set_window.
static int plan_find_set_launch(const char* who, const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end,
                                const uint8_t* src_base, uint64_t lo16, uint64_t hi16, const mod_pattern_set* set,
                                const uint32_t* d_owned, uint32_t* d_counts, uint64_t* d_pattern_counts,
                                mod_set_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream)
{
    if (tile_begin == tile_end)
        return MOD_OK;
    if (!d_pattern_counts)
        return fail(MOD_ERR_ARG, "%s: null result buffer", who);
    int rc = find_check(who, plan, src_base, d_counts, d_total, cap, d_matches);
    if (rc != MOD_OK)
        return rc;
    if (set->device != plan->device)
        return fail(MOD_ERR_ARG, "%s: the pattern set lives on device %d but the plan on device %d", who, set->device, plan->device);
    modk::FindSetArgs f;
    f.src = src_base;
    f.tiles = plan->d_tiles + tile_begin;
    f.descs = plan->d_descs;
    f.n_tiles = (uint32_t)(tile_end - tile_begin);
    f.src_lo16 = lo16;
    f.src_hi16 = hi16;
    f.set = set->d_index;
    f.n_keys = set->n_keys;
    f.lmin = set->lmin;
    f.lmax = set->lmax;
    f.owned = d_owned;
    f.counts = d_counts;
    f.pattern_counts = (unsigned long long*)d_pattern_counts;
    f.matches = (uint32_t*)d_matches;
    f.total = (unsigned long long*)d_total;
    f.cap = cap;
    CUDA_TRY(modk::launch_find_set(f, set->fold, (cudaStream_t)stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MOD_OK;
}

int mod_plan_find_set(const mod_plan* plan, const void* d_src, const mod_pattern_set* set, const uint32_t* d_owned,
                      uint32_t* d_counts, uint64_t* d_pattern_counts, mod_set_match* d_matches, uint64_t cap,
                      uint64_t* d_total, void* stream)
{
    if (!plan || !set)
        return fail(MOD_ERR_ARG, "mod_plan_find_set: null plan or pattern set");
    if (!d_src && plan->n_tiles)
        return fail(MOD_ERR_ARG, "mod_plan_find_set: null buffer");
    return plan_find_set_launch("mod_plan_find_set", plan, 0, plan->n_tiles, (const uint8_t*)d_src,
                                ((uint64_t)(uintptr_t)d_src + 15u) & ~15ull,
                                ((uint64_t)(uintptr_t)d_src + plan->src_bytes) & ~15ull, set, d_owned, d_counts,
                                d_pattern_counts, d_matches, cap, d_total, stream);
}

int mod_plan_find_set_window(const mod_plan* plan, uint64_t tile_begin, uint64_t tile_end, const void* d_src_win,
                             uint64_t src_win_off, uint64_t src_win_bytes, const mod_pattern_set* set,
                             const uint32_t* d_owned, uint32_t* d_counts, uint64_t* d_pattern_counts,
                             mod_set_match* d_matches, uint64_t cap, uint64_t* d_total, void* stream)
{
    if (!plan || !set)
        return fail(MOD_ERR_ARG, "mod_plan_find_set_window: null plan or pattern set");
    int rc = find_window_check("mod_plan_find_set_window", plan, tile_begin, tile_end, d_src_win, src_win_off, src_win_bytes,
                               set->lmax - 1);
    if (rc != MOD_OK)
        return rc;
    return plan_find_set_launch("mod_plan_find_set_window", plan, tile_begin, tile_end, (const uint8_t*)d_src_win - src_win_off,
                                ((uint64_t)(uintptr_t)d_src_win + 15u) & ~15ull,
                                ((uint64_t)(uintptr_t)d_src_win + src_win_bytes) & ~15ull, set, d_owned, d_counts,
                                d_pattern_counts, d_matches, cap, d_total, stream);
}

int mod_find_set_batch(const mod_desc* descs, uint64_t n, const void* d_src, uint64_t src_bytes, const uint8_t* bytes,
                       const uint32_t* lens, uint32_t n_patterns, uint32_t* counts_out, uint64_t* pattern_counts_out,
                       mod_set_match* matches_out, uint64_t cap, uint64_t* total_out)
{
    MOD_ABI_BEGIN
    if (!pattern_counts_out)
        return fail(MOD_ERR_ARG, "mod_find_set_batch: null argument");
    mod_pattern_set* set = nullptr;
    int rc = find_batch_run("mod_find_set_batch", descs, n, d_src, src_bytes, counts_out, pattern_counts_out,
                            8ull * n_patterns, matches_out, sizeof(mod_set_match), cap, total_out,
                            [&](mod_plan* plan, uint32_t* d_counts, uint8_t* d_aux, uint8_t* d_list, uint64_t* d_total) {
                                const int r = mod_pattern_set_create(bytes, lens, n_patterns, &set);
                                return r != MOD_OK ? r : mod_plan_find_set(plan, d_src, set, nullptr, d_counts, (uint64_t*)d_aux,
                                                                           (mod_set_match*)d_list, cap, d_total, nullptr);
                            });
    mod_pattern_set_destroy(set);
    if (rc != MOD_OK)
        return rc;
    std::sort(matches_out, matches_out + std::min(*total_out, cap), [](const mod_set_match& a, const mod_set_match& b) {
        return a.desc != b.desc ? a.desc < b.desc : a.pos != b.pos ? a.pos < b.pos : a.pattern < b.pattern;
    });
    return MOD_OK;
    MOD_ABI_END("mod_find_set_batch")
}

int mod_cycle_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, void* dst,
                    uint64_t dst_bytes)
{
    MOD_ABI_BEGIN
    if (n == 0)
        return MOD_OK;
    if (!descs)
        return fail(MOD_ERR_ARG, "mod_cycle_batch: descs is null");
    if (!src || !dst)
        return fail(MOD_ERR_ARG, "mod_cycle_batch: null buffer");
    int src_dev = -1, dst_dev = -1;
    const bool src_is_dev = pointer_device(src, &src_dev), dst_is_dev = pointer_device(dst, &dst_dev);
    if (src_is_dev != dst_is_dev || (src_is_dev && src_dev != dst_dev))
        return fail(MOD_ERR_ARG, "mod_cycle_batch: src and dst must both be host pointers or both live on one device");

    if (src_is_dev) {
        DeviceGuard guard;
        int rc = guard.enter(src_dev);
        if (rc != MOD_OK)
            return rc;
        mod_plan* plan = nullptr;
        rc = mod_plan_create(descs, n, src_bytes, dst_bytes, (uint32_t)((uintptr_t)dst & 15u), &plan);
        if (rc != MOD_OK)
            return rc;
        rc = mod_plan_run(plan, src, dst, nullptr);
        cudaError_t e = cudaStreamSynchronize(nullptr);
        mod_plan_destroy(plan);
        if (rc != MOD_OK)
            return rc;
        CUDA_TRY(e);
        return MOD_OK;
    }
    DeviceCtx* c = nullptr;
    int rc = acquire(-1, &c);
    if (rc != MOD_OK)
        return rc;
    return batch_host(*c, descs, n, (const uint8_t*)src, src_bytes, (uint8_t*)dst, dst_bytes);
    MOD_ABI_END("mod_cycle_batch")
}

int mod_cycle_batch_sharded(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, void* dst,
                            uint64_t dst_bytes, uint64_t dev_mask)
{
    MOD_ABI_BEGIN
    if (n == 0)
        return MOD_OK;
    if (!descs)
        return fail(MOD_ERR_ARG, "mod_cycle_batch_sharded: descs is null");
    if (!src || !dst)
        return fail(MOD_ERR_ARG, "mod_cycle_batch_sharded: null buffer");
    int dev = -1;
    if (pointer_device(src, &dev) || pointer_device(dst, &dev))
        return fail(MOD_ERR_ARG, "mod_cycle_batch_sharded: src and dst must be host buffers");
    int rc = validate_descs("mod_cycle_batch_sharded", descs, n, src_bytes, dst_bytes);
    if (rc != MOD_OK)
        return rc;
    return for_each_device(dev_mask, [=](int rank, int world, DeviceCtx& c) -> int {
        if (world == 1)
            return batch_host(c, descs, n, (const uint8_t*)src, src_bytes, (uint8_t*)dst, dst_bytes);
        const int64_t count = mod_shard_descs(descs, n, rank, world, nullptr, 0);
        if (count < 0)
            return (int)count;
        if (count == 0)
            return MOD_OK;
        std::vector<mod_desc> shard((size_t)count);
        const int64_t got = mod_shard_descs(descs, n, rank, world, shard.data(), (uint64_t)count);
        if (got < 0)
            return (int)got;
        return batch_host(c, shard.data(), (uint64_t)got, (const uint8_t*)src, src_bytes, (uint8_t*)dst, dst_bytes);
    });
    MOD_ABI_END("mod_cycle_batch_sharded")
}

/* ---- offset-range sharding (pure host logic) ------------------------------------------------------ */

int mod_shard_range(uint64_t total, int rank, int world, uint64_t* begin, uint64_t* end)
{
    if (world <= 0 || rank < 0 || rank >= world || !begin || !end)
        return fail(MOD_ERR_ARG, "mod_shard_range: bad rank %d / world %d", rank, world);
    const uint64_t share = ((total / (uint64_t)world) + 15u) & ~15ull;
    uint64_t b = std::min(total, share * (uint64_t)rank);
    uint64_t e = (rank == world - 1) ? total : std::min(total, share * (uint64_t)(rank + 1));
    *begin = b;
    *end = e;
    return MOD_OK;
}

int64_t mod_group_descs(const mod_desc* descs, uint64_t n, uint64_t group_bytes, uint64_t dst_phase, uint64_t modulus,
                        mod_desc* out, uint8_t* closes, uint64_t out_cap)
{
    MOD_ABI_BEGIN
    if (n && !descs)
        return fail(MOD_ERR_ARG, "mod_group_descs: descs is null");
    if (modulus < 16 || (modulus & (modulus - 1)) != 0 || group_bytes < modulus)
        return fail(MOD_ERR_ARG, "mod_group_descs: modulus must be a power of two >= 16 and <= group_bytes");
    modcut::Cut cut;
    modcut::cut_into_groups(descs, n, group_bytes, dst_phase, modulus, cut);
    if (out || closes) {
        if (cut.pieces.size() > out_cap || !out || !closes)
            return fail(MOD_ERR_ARG, "mod_group_descs: %zu pieces do not fit the output capacity", cut.pieces.size());
        std::copy(cut.pieces.begin(), cut.pieces.end(), out);
        std::copy(cut.closes.begin(), cut.closes.end(), closes);
    }
    return (int64_t)cut.pieces.size();
    MOD_ABI_END("mod_group_descs")
}

int64_t mod_shard_descs(const mod_desc* descs, uint64_t n, int rank, int world, mod_desc* out, uint64_t out_cap)
{
    if (world <= 0 || rank < 0 || rank >= world)
        return fail(MOD_ERR_ARG, "mod_shard_descs: bad rank %d / world %d", rank, world);
    if (n && !descs)
        return fail(MOD_ERR_ARG, "mod_shard_descs: descs is null");
    uint64_t total = 0;
    for (uint64_t i = 0; i < n; ++i)
        total += descs[i].len;
    // this rank owns cumulative payload bytes [lo, hi)
    const uint64_t lo = (uint64_t)(((unsigned __int128)total * (unsigned)rank) / (unsigned)world);
    const uint64_t hi = (rank == world - 1) ? total
                                            : (uint64_t)(((unsigned __int128)total * (unsigned)(rank + 1)) / (unsigned)world);
    // A boundary that falls inside an entry is moved down to the nearest position whose destination
    // offset is 16-byte aligned; the rule depends only on (entry, boundary) so all ranks agree.
    auto cut_at = [](const mod_desc& d, uint64_t raw) -> uint64_t {
        const uint64_t mis = (d.dst_off + raw) & 15u;
        return raw > mis ? raw - mis : 0;
    };
    uint64_t count = 0, cum = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const mod_desc& d = descs[i];
        const uint64_t c0 = cum, c1 = cum + d.len;
        cum = c1;
        if (d.len == 0 || c1 <= lo || c0 >= hi)
            continue;
        const uint64_t b = (lo <= c0) ? 0 : cut_at(d, lo - c0);
        const uint64_t e = (hi >= c1) ? d.len : cut_at(d, hi - c0);
        if (e <= b)
            continue;
        if (out) {
            if (count >= out_cap)
                return fail(MOD_ERR_ARG, "mod_shard_descs: output capacity %llu too small", (unsigned long long)out_cap);
            mod_desc& o = out[count];
            o.src_off = d.src_off + b;
            o.dst_off = d.dst_off + b;
            o.len = (uint32_t)(e - b);
            o.key = b ? mod_key_jump(d.key, b) : d.key;
        }
        ++count;
    }
    return (int64_t)count;
}

}  // extern "C"
