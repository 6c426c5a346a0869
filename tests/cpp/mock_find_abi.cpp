// tests/cpp/mock_find_abi.cpp -- TEST INFRASTRUCTURE.  The search entry points of the C ABI (mod_plan_find,
// mod_plan_find_window, mod_find_batch) answered on the CPU: the oracle's Cycle of each descriptor, then every
// start position compared.  Linked next to tests/cpp/mock_abi.cpp into tests/_build/modulate_mock_find, so
// CArk::FindInFiles and -find / -findhex run end to end without a GPU.
//
// A plan and a stream are mock_abi.cpp's objects; the two definitions below repeat that file's, token for
// token (one definition per program, as C++ requires of a class defined in several translation units).
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/modulate_b200.h"

extern "C" void oracle_cycle_at(unsigned char* data, uint64_t size, int32_t key, uint64_t pos);

struct mod_plan {
    std::vector<mod_desc> descs;
    std::vector<uint64_t> first_tile;  // n + 1
    uint32_t dst_align = 0;
    int device = 0;
};

struct mock_stream {
    int device;
};

static void mock_find_entry(const mod_desc& d, uint32_t index, const unsigned char* src, const uint8_t* pattern, uint32_t len,
                            uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total)
{
    std::vector<unsigned char> bytes(src + d.src_off, src + d.src_off + d.len);
    oracle_cycle_at(bytes.data(), bytes.size(), d.key, 0);
    for (uint64_t i = 0; i + len <= bytes.size(); ++i) {
        if (std::memcmp(bytes.data() + i, pattern, len) != 0)
            continue;
        ++counts[index];
        if (*total < cap)
            matches[*total] = mod_match{index, (uint32_t)i};
        ++*total;
    }
}

extern "C" {

int mod_plan_find_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                         uint64_t src_win_bytes, const uint8_t* pattern, uint32_t len, uint32_t* counts, mod_match* matches,
                         uint64_t cap, uint64_t* total, void* stream)
{
    if (!pattern || len == 0 || len > 64)
        return MOD_ERR_ARG;
    // like the real library: the calling thread, the plan and the stream must be on one device
    const int device = mod_current_device();
    if (plan->device != device || (stream && ((const mock_stream*)stream)->device != device))
        return MOD_ERR_ARG;
    for (size_t e = 0; e < plan->descs.size(); ++e) {
        if (plan->first_tile[e + 1] <= t0 || plan->first_tile[e] >= t1 || plan->first_tile[e + 1] == plan->first_tile[e])
            continue;
        if (plan->first_tile[e] < t0 || plan->first_tile[e + 1] > t1)
            return MOD_ERR_ARG;  // the mock only runs whole entries
        const mod_desc& d = plan->descs[e];
        if (d.src_off != d.dst_off || d.src_off < src_win_off || d.src_off + d.len > src_win_off + src_win_bytes)
            return MOD_ERR_ARG;
        mock_find_entry(d, (uint32_t)e, (const unsigned char*)src_win - src_win_off, pattern, len, counts, matches, cap, total);
    }
    return MOD_OK;
}

int mod_plan_find(const mod_plan* plan, const void* src, const uint8_t* pattern, uint32_t len, uint32_t* counts,
                  mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    return mod_plan_find_window(plan, 0, plan->first_tile.back(), src, 0, UINT64_MAX / 2, pattern, len, counts, matches, cap,
                                total, stream);
}

int mod_find_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, const uint8_t* pattern,
                   uint32_t len, uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total)
{
    if (!pattern || len == 0 || len > 64)
        return MOD_ERR_ARG;
    *total = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (descs[i].src_off + descs[i].len > src_bytes)
            return MOD_ERR_ARG;
        counts[i] = 0;
        mock_find_entry(descs[i], (uint32_t)i, (const unsigned char*)src, pattern, len, counts, matches, cap, total);
    }
    return MOD_OK;
}
}
