// tests/cpp/mock_abi.cpp -- TEST INFRASTRUCTURE.  A stand-in for the CUDA library's C ABI that
// answers the facade's calls with the CPU ORACLE (oracle/cycle_oracle.c), so the host-side C++
// (CArk, ArkHeader, the CLI) can be exercised end to end on a box without a GPU.  It is linked only
// into the test binaries of tests/_build (tests/searchutil.py); the product library never contains it.
//
// "Device" memory is host memory, "streams" run synchronously at enqueue time, and a plan is the
// descriptor list plus the same first-tile prefix the real library computes (8 KiB tiles of one
// entry each), so mod_plan_tile_range / mod_plan_run_window can be answered for whole-entry ranges --
// the only kind the facade issues.
//
// MOD_MOCK_DEVICES=<n> (default 1) makes it report n devices.  Like the CUDA runtime, each thread is
// bound to a device (mod_init, 0 until then); plans and streams remember the device they were created
// on, and mod_plan_run_window refuses to run unless the caller, the plan and the stream agree (the real
// library's plan_check_device; a stream of another device is a CUDA error there).
#include <cstdlib>
#include <cstring>

#include "mock_abi.h"

static thread_local int tl_device = 0;

static int mock_device_count()
{
    const char* v = std::getenv("MOD_MOCK_DEVICES");
    const int n = v && *v ? std::atoi(v) : 1;
    return n > 0 ? n : 1;
}

static uint64_t tiles_for_entry(uint32_t h0, uint32_t len)
{
    if (!len)
        return 0;
    const uint64_t chunks = ((uint64_t)h0 + len + 15u) >> 4;
    return (chunks + 511) / 512;
}

extern "C" {

int mod_abi_version(void) { return MOD_ABI_VERSION; }
int mod_device_count(void) { return mock_device_count(); }
int mod_init(int device)
{
    if (device < 0 || device >= mock_device_count())
        return MOD_ERR_ARG;
    tl_device = device;
    return MOD_OK;
}
int mod_current_device(void) { return tl_device; }
int mod_is_device_pointer(const void*) { return 0; }
void mod_shutdown(void) {}
const char* mod_last_error(void) { return "mock ABI (oracle-backed, tests only)"; }
uint64_t mod_launch_count(void) { return 0; }
void* mod_host_alloc(uint64_t bytes) { return std::malloc(bytes ? bytes : 1); }
int mod_host_free(void* p)
{
    std::free(p);
    return MOD_OK;
}
void* mod_device_alloc(uint64_t bytes) { return std::malloc(bytes ? bytes : 1); }
int mod_device_free(void* p)
{
    std::free(p);
    return MOD_OK;
}
int mod_memcpy_h2d(void* d, const void* h, uint64_t bytes, void*)
{
    std::memcpy(d, h, bytes);
    return MOD_OK;
}
int mod_memcpy_d2h(void* h, const void* d, uint64_t bytes, void*)
{
    std::memcpy(h, d, bytes);
    return MOD_OK;
}
int mod_stream_sync(void*) { return MOD_OK; }
void* mod_stream_create(void) { return new mock_stream{tl_device}; }
int mod_stream_destroy(void* s)
{
    delete (mock_stream*)s;
    return MOD_OK;
}
int mod_cycle(void* data, uint64_t len, int32_t key)
{
    oracle_cycle_at((unsigned char*)data, len, key, 0);
    return MOD_OK;
}
int mod_cycle_sharded(void* data, uint64_t len, int32_t key, uint64_t) { return mod_cycle(data, len, key); }
int32_t mod_key_jump(int32_t key, uint64_t pos) { return oracle_key_jump(key, pos); }
int mod_cycle_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, void* dst, uint64_t dst_bytes)
{
    for (uint64_t i = 0; i < n; ++i)
        if (descs[i].src_off + descs[i].len > src_bytes || descs[i].dst_off + descs[i].len > dst_bytes)
            return MOD_ERR_ARG;
    static_assert(sizeof(mod_desc) == sizeof(oracle_desc), "descriptor layouts must match");
    oracle_cycle_batch((const oracle_desc*)descs, n, (const unsigned char*)src, (unsigned char*)dst);
    return MOD_OK;
}

int mod_plan_create(const mod_desc* descs, uint64_t n, uint64_t src_bytes, uint64_t dst_bytes, uint32_t dst_align, mod_plan** out)
{
    for (uint64_t i = 0; i < n; ++i)
        if (descs[i].src_off + descs[i].len > src_bytes || descs[i].dst_off + descs[i].len > dst_bytes)
            return MOD_ERR_ARG;
    mod_plan* p = new mod_plan();
    p->descs.assign(descs, descs + n);
    p->dst_align = dst_align;
    p->device = tl_device;
    p->first_tile.resize(n + 1);
    uint64_t tiles = 0;
    for (uint64_t i = 0; i < n; ++i) {
        p->first_tile[i] = tiles;
        tiles += tiles_for_entry((uint32_t)((dst_align + descs[i].dst_off) & 15u), descs[i].len);
    }
    p->first_tile[n] = tiles;
    *out = p;
    return MOD_OK;
}
int mod_plan_destroy(mod_plan* plan)
{
    delete plan;
    return MOD_OK;
}
int mod_plan_tile_range(const mod_plan* plan, uint64_t e0, uint64_t e1, uint64_t* t0, uint64_t* t1)
{
    if (e0 > e1 || e1 > plan->descs.size())
        return MOD_ERR_ARG;
    *t0 = plan->first_tile[e0];
    *t1 = plan->first_tile[e1];
    return MOD_OK;
}
int mod_plan_run_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                        uint64_t src_win_bytes, void* dst_win, uint64_t dst_win_off, uint64_t dst_win_bytes, void* stream)
{
    if (plan->device != tl_device || (stream && ((const mock_stream*)stream)->device != tl_device))
        return MOD_ERR_ARG;
    if ((((uintptr_t)dst_win - dst_win_off) & 15u) != plan->dst_align)
        return MOD_ERR_ALIGN;
    for (size_t e = 0; e < plan->descs.size(); ++e) {
        if (plan->first_tile[e + 1] <= t0 || plan->first_tile[e] >= t1 || plan->first_tile[e + 1] == plan->first_tile[e])
            continue;
        if (plan->first_tile[e] < t0 || plan->first_tile[e + 1] > t1)
            return MOD_ERR_ARG;  // the mock only runs whole entries
        const mod_desc& d = plan->descs[e];
        if (d.src_off < src_win_off || d.src_off + d.len > src_win_off + src_win_bytes || d.dst_off < dst_win_off ||
            d.dst_off + d.len > dst_win_off + dst_win_bytes)
            return MOD_ERR_ARG;
        oracle_desc one{d.src_off - src_win_off, d.dst_off - dst_win_off, d.len, d.key};
        oracle_cycle_batch(&one, 1, (const unsigned char*)src_win, (unsigned char*)dst_win);
    }
    return MOD_OK;
}
}
