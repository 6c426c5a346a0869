// tests/cpp/mock_find_masked_abi.cpp -- TEST INFRASTRUCTURE.  The masked and case-insensitive search entry points of
// the C ABI (mod_plan_find_masked, mod_plan_find_masked_window, mod_find_masked_batch, mod_pattern_set_create_nocase)
// answered on the CPU: the oracle's Cycle of each descriptor, then every start compared under the mask or after ASCII
// case folding.  It also answers the set entry points of tests/cpp/mock_find_set_abi.cpp (mod_pattern_set_create /
// _destroy, mod_plan_find_set, mod_plan_find_set_window, mod_find_set_batch), with sets that may be folded, so it is
// linked next to tests/cpp/mock_abi.cpp and mock_find_abi.cpp IN PLACE of mock_find_set_abi.cpp.  Then
// CArk::FindMaskedInFiles and -findi / -findwild / -findilist run end to end without a GPU; linked with
// mock_find_set_abi.cpp instead, the facade sees a library without them.
//
// A plan and a stream are mock_abi.cpp's objects; the definitions below repeat that file's, token for token.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <set>
#include <string>
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

struct mod_pattern_set {
    std::vector<std::string> patterns;
    int device = 0;
    bool fold = false;  // mod_pattern_set_create_nocase: upper-cased patterns, entry bytes folded before the compare
};

static unsigned char mock_fold(unsigned char c) { return c >= 'a' && c <= 'z' ? (unsigned char)(c - 0x20) : c; }

static void mock_find_set_entry(const mod_desc& d, uint32_t index, const unsigned char* src, const mod_pattern_set& set,
                                uint32_t owned, uint32_t* counts, uint64_t* pattern_counts, mod_set_match* matches, uint64_t cap,
                                uint64_t* total)
{
    std::vector<unsigned char> bytes(src + d.src_off, src + d.src_off + d.len);
    oracle_cycle_at(bytes.data(), bytes.size(), d.key, 0);
    if (set.fold)
        for (unsigned char& c : bytes)
            c = mock_fold(c);
    for (uint64_t i = 0; i < bytes.size() && i < owned; ++i) {
        for (uint32_t j = 0; j < set.patterns.size(); ++j) {
            const std::string& p = set.patterns[j];
            if (i + p.size() > bytes.size() || std::memcmp(bytes.data() + i, p.data(), p.size()) != 0)
                continue;
            ++counts[index];
            ++pattern_counts[j];
            if (*total < cap)
                matches[*total] = mod_set_match{index, (uint32_t)i, j};
            ++*total;
        }
    }
}

// The body of mod_pattern_set_create and mod_pattern_set_create_nocase.
static int mock_set_create(const uint8_t* bytes, const uint32_t* lens, uint32_t n, bool fold, mod_pattern_set** out)
{
    if (!out || !bytes || !lens || n == 0 || n > 256)
        return MOD_ERR_ARG;
    mod_pattern_set* set = new mod_pattern_set();
    set->fold = fold;
    uint64_t at = 0;
    for (uint32_t j = 0; j < n; ++j) {
        if (lens[j] == 0 || lens[j] > 64) {
            delete set;
            return MOD_ERR_ARG;
        }
        std::string p((const char*)bytes + at, lens[j]);
        if (fold)
            for (char& c : p)
                c = (char)mock_fold((unsigned char)c);
        set->patterns.push_back(p);
        at += lens[j];
    }
    if (std::set<std::string>(set->patterns.begin(), set->patterns.end()).size() != n) {
        delete set;
        return MOD_ERR_ARG;
    }
    set->device = mod_current_device();
    *out = set;
    return MOD_OK;
}

static bool mock_mask_ok(const uint8_t* pattern, const uint8_t* mask, uint32_t len)
{
    if (!pattern || !mask || len == 0 || len > 64)
        return false;
    for (uint32_t k = 0; k < len; ++k)
        if (mask[k])
            return true;
    return false;
}

static void mock_find_masked_entry(const mod_desc& d, uint32_t index, const unsigned char* src, const uint8_t* pattern,
                                   const uint8_t* mask, uint32_t len, uint32_t* counts, mod_match* matches, uint64_t cap,
                                   uint64_t* total)
{
    std::vector<unsigned char> bytes(src + d.src_off, src + d.src_off + d.len);
    oracle_cycle_at(bytes.data(), bytes.size(), d.key, 0);
    for (uint64_t i = 0; i + len <= bytes.size(); ++i) {
        bool hit = true;
        for (uint32_t k = 0; k < len && hit; ++k)
            hit = ((bytes[i + k] ^ pattern[k]) & mask[k]) == 0;
        if (!hit)
            continue;
        ++counts[index];
        if (*total < cap)
            matches[*total] = mod_match{index, (uint32_t)i};
        ++*total;
    }
}

extern "C" {

int mod_plan_find_masked_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                                uint64_t src_win_bytes, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                                uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    if (!mock_mask_ok(pattern, mask, len))
        return MOD_ERR_ARG;
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
        mock_find_masked_entry(d, (uint32_t)e, (const unsigned char*)src_win - src_win_off, pattern, mask, len, counts, matches,
                               cap, total);
    }
    return MOD_OK;
}

int mod_plan_find_masked(const mod_plan* plan, const void* src, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                         uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    return mod_plan_find_masked_window(plan, 0, plan->first_tile.back(), src, 0, UINT64_MAX / 2, pattern, mask, len, counts,
                                       matches, cap, total, stream);
}

int mod_find_masked_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, const uint8_t* pattern,
                          const uint8_t* mask, uint32_t len, uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total)
{
    if (!mock_mask_ok(pattern, mask, len))
        return MOD_ERR_ARG;
    *total = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (descs[i].src_off + descs[i].len > src_bytes)
            return MOD_ERR_ARG;
        counts[i] = 0;
        mock_find_masked_entry(descs[i], (uint32_t)i, (const unsigned char*)src, pattern, mask, len, counts, matches, cap, total);
    }
    return MOD_OK;
}

int mod_pattern_set_create_nocase(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out)
{
    return mock_set_create(bytes, lens, n, true, out);
}

int mod_pattern_set_create(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out)
{
    return mock_set_create(bytes, lens, n, false, out);
}

int mod_pattern_set_destroy(mod_pattern_set* set)
{
    delete set;
    return MOD_OK;
}

int mod_plan_find_set_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                             uint64_t src_win_bytes, const mod_pattern_set* set, const uint32_t* owned, uint32_t* counts,
                             uint64_t* pattern_counts, mod_set_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    if (!plan || !set)
        return MOD_ERR_ARG;
    // like the real library: the calling thread, the plan, the set and the stream must be on one device
    const int device = mod_current_device();
    if (plan->device != device || set->device != device || (stream && ((const mock_stream*)stream)->device != device))
        return MOD_ERR_ARG;
    for (size_t e = 0; e < plan->descs.size(); ++e) {
        if (plan->first_tile[e + 1] <= t0 || plan->first_tile[e] >= t1 || plan->first_tile[e + 1] == plan->first_tile[e])
            continue;
        if (plan->first_tile[e] < t0 || plan->first_tile[e + 1] > t1)
            return MOD_ERR_ARG;  // the mock only runs whole entries
        const mod_desc& d = plan->descs[e];
        if (d.src_off != d.dst_off || d.src_off < src_win_off || d.src_off + d.len > src_win_off + src_win_bytes)
            return MOD_ERR_ARG;
        mock_find_set_entry(d, (uint32_t)e, (const unsigned char*)src_win - src_win_off, *set, owned ? owned[e] : UINT32_MAX,
                            counts, pattern_counts, matches, cap, total);
    }
    return MOD_OK;
}

int mod_plan_find_set(const mod_plan* plan, const void* src, const mod_pattern_set* set, const uint32_t* owned, uint32_t* counts,
                      uint64_t* pattern_counts, mod_set_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    if (!plan)
        return MOD_ERR_ARG;
    return mod_plan_find_set_window(plan, 0, plan->first_tile.back(), src, 0, UINT64_MAX / 2, set, owned, counts, pattern_counts,
                                    matches, cap, total, stream);
}

int mod_find_set_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, const uint8_t* bytes,
                       const uint32_t* lens, uint32_t n_patterns, uint32_t* counts, uint64_t* pattern_counts,
                       mod_set_match* matches, uint64_t cap, uint64_t* total)
{
    mod_pattern_set* set = nullptr;
    const int rc = mod_pattern_set_create(bytes, lens, n_patterns, &set);
    if (rc != MOD_OK)
        return rc;
    *total = 0;
    std::fill(pattern_counts, pattern_counts + n_patterns, 0);
    for (uint64_t i = 0; i < n; ++i) {
        if (descs[i].src_off + descs[i].len > src_bytes) {
            delete set;
            return MOD_ERR_ARG;
        }
        counts[i] = 0;
        mock_find_set_entry(descs[i], (uint32_t)i, (const unsigned char*)src, *set, UINT32_MAX, counts, pattern_counts, matches,
                            cap, total);
    }
    delete set;
    return MOD_OK;
}
}
