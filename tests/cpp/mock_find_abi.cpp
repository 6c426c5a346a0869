// tests/cpp/mock_find_abi.cpp -- TEST INFRASTRUCTURE.  The search entry points of the C ABI answered on the CPU, so
// CArk's searches and every search command of the CLI run end to end without a GPU.  Every entry point is one scan
// per entry: the oracle's Cycle, then, for each pattern, every start i < owned where ((b ^ v) & m) == 0 for every
// pattern byte (v, m) and entry byte b, with b folded for a folded set.  The exact search is the scan with an all-0xFF
// mask; a single-pattern search is a one-pattern set.
//
// MOCK_SEARCH_ABI picks the library generation the mock stands for, so that the facade can be linked against a
// library that predates a search:
//   0  no search entry points;
//   1  mod_plan_find, mod_plan_find_window, mod_find_batch;
//   2  adds the pattern sets (mod_pattern_set_create / _destroy, mod_plan_find_set, _window, mod_find_set_batch);
//   3  adds mod_plan_find_masked, mod_plan_find_masked_window, mod_find_masked_batch, mod_pattern_set_create_nocase.
#ifndef MOCK_SEARCH_ABI
#define MOCK_SEARCH_ABI 3
#endif

#if MOCK_SEARCH_ABI >= 1
#include <algorithm>
#include <memory>
#include <set>
#include <string>

#include "mock_abi.h"

struct mod_pattern_set {
    std::vector<std::string> values, masks;
    bool fold = false;  // mod_pattern_set_create_nocase: upper-cased values, entry bytes folded before the compare
    int device = 0;
};

// Where a search's results go: a set search counts per pattern and lists mod_set_match, a single one lists mod_match.
struct mock_results {
    uint32_t* counts;
    uint64_t* pattern_counts;
    mod_match* matches;
    mod_set_match* set_matches;
    uint64_t cap;
    uint64_t* total;
};

static unsigned char mock_fold(unsigned char c) { return c >= 'a' && c <= 'z' ? (unsigned char)(c - 0x20) : c; }

// Appends pattern (value, mask) to `set`; a NULL mask is the exact pattern.  False for what the library refuses.
static bool add_pattern(mod_pattern_set& set, const uint8_t* value, const uint8_t* mask, uint32_t len)
{
    if (!value || len == 0 || len > 64)
        return false;
    std::string v((const char*)value, len), m = mask ? std::string((const char*)mask, len) : std::string(len, '\xff');
    if (m.find_first_not_of('\0') == std::string::npos)
        return false;
    if (set.fold)
        for (char& c : v)
            c = (char)mock_fold((unsigned char)c);
    set.values.push_back(v);
    set.masks.push_back(m);
    return true;
}

static void scan_entry(const mod_desc& d, uint32_t index, const unsigned char* src, const mod_pattern_set& set, uint32_t owned,
                       const mock_results& out)
{
    std::vector<unsigned char> bytes(src + d.src_off, src + d.src_off + d.len);
    oracle_cycle_at(bytes.data(), bytes.size(), d.key, 0);
    if (set.fold)
        for (unsigned char& c : bytes)
            c = mock_fold(c);
    for (uint64_t i = 0; i < bytes.size() && i < owned; ++i) {
        for (uint32_t j = 0; j < set.values.size(); ++j) {
            const std::string &v = set.values[j], &m = set.masks[j];
            bool hit = i + v.size() <= bytes.size();
            for (size_t k = 0; k < v.size() && hit; ++k)
                hit = ((bytes[i + k] ^ (unsigned char)v[k]) & (unsigned char)m[k]) == 0;
            if (!hit)
                continue;
            ++out.counts[index];
            if (out.pattern_counts)
                ++out.pattern_counts[j];
            if (*out.total < out.cap) {
                if (out.set_matches)
                    out.set_matches[*out.total] = mod_set_match{index, (uint32_t)i, j};
                else
                    out.matches[*out.total] = mod_match{index, (uint32_t)i};
            }
            ++*out.total;
        }
    }
}

// Every entry of tiles [t0, t1) of the plan, after the checks the real library makes that the facade can trip: the
// calling thread, the plan, the set and the stream on one device; whole entries only (the facade issues no other
// range); the plan built with dst_off == src_off; each entry inside the source window.
static int scan_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                       uint64_t src_win_bytes, const mod_pattern_set* set, const uint32_t* owned, const mock_results& out,
                       void* stream)
{
    if (!plan || !set)
        return MOD_ERR_ARG;
    const int device = mod_current_device();
    if (plan->device != device || set->device != device || (stream && ((const mock_stream*)stream)->device != device))
        return MOD_ERR_ARG;
    for (size_t e = 0; e < plan->descs.size(); ++e) {
        if (plan->first_tile[e + 1] <= t0 || plan->first_tile[e] >= t1 || plan->first_tile[e + 1] == plan->first_tile[e])
            continue;
        if (plan->first_tile[e] < t0 || plan->first_tile[e + 1] > t1)
            return MOD_ERR_ARG;
        const mod_desc& d = plan->descs[e];
        if (d.src_off != d.dst_off || d.src_off < src_win_off || d.src_off + d.len > src_win_off + src_win_bytes)
            return MOD_ERR_ARG;
        scan_entry(d, (uint32_t)e, (const unsigned char*)src_win - src_win_off, *set, owned ? owned[e] : UINT32_MAX, out);
    }
    return MOD_OK;
}

// The body of the batch calls: results start from zero, every descriptor inside the source.
static int scan_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, const mod_pattern_set& set,
                      const mock_results& out)
{
    *out.total = 0;
    if (out.pattern_counts)
        std::fill(out.pattern_counts, out.pattern_counts + set.values.size(), 0);
    for (uint64_t i = 0; i < n; ++i) {
        if (descs[i].src_off + descs[i].len > src_bytes)
            return MOD_ERR_ARG;
        out.counts[i] = 0;
        scan_entry(descs[i], (uint32_t)i, (const unsigned char*)src, set, UINT32_MAX, out);
    }
    return MOD_OK;
}

// mod_plan_find_window and mod_plan_find_masked_window: a one-pattern set of the calling device.
static int find_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                       uint64_t src_win_bytes, const uint8_t* pattern, const uint8_t* mask, uint32_t len, uint32_t* counts,
                       mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    mod_pattern_set one;
    one.device = mod_current_device();
    if (!add_pattern(one, pattern, mask, len))
        return MOD_ERR_ARG;
    return scan_window(plan, t0, t1, src_win, src_win_off, src_win_bytes, &one, nullptr,
                       mock_results{counts, nullptr, matches, nullptr, cap, total}, stream);
}

static int find_plan(const mod_plan* plan, const void* src, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                     uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    if (!plan)
        return MOD_ERR_ARG;
    return find_window(plan, 0, plan->first_tile.back(), src, 0, UINT64_MAX / 2, pattern, mask, len, counts, matches, cap,
                       total, stream);
}

static int find_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, const uint8_t* pattern,
                      const uint8_t* mask, uint32_t len, uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total)
{
    mod_pattern_set one;
    if (!add_pattern(one, pattern, mask, len))
        return MOD_ERR_ARG;
    return scan_batch(descs, n, src, src_bytes, one, mock_results{counts, nullptr, matches, nullptr, cap, total});
}
#endif

#if MOCK_SEARCH_ABI >= 2
// mod_pattern_set_create and mod_pattern_set_create_nocase: 1..256 distinct patterns, compared folded when `fold`.
static int set_create(const uint8_t* bytes, const uint32_t* lens, uint32_t n, bool fold, mod_pattern_set** out)
{
    if (!out || !bytes || !lens || n == 0 || n > 256)
        return MOD_ERR_ARG;
    std::unique_ptr<mod_pattern_set> set(new mod_pattern_set());
    set->fold = fold;
    set->device = mod_current_device();
    uint64_t at = 0;
    for (uint32_t j = 0; j < n; ++j) {
        if (!add_pattern(*set, bytes + at, nullptr, lens[j]))
            return MOD_ERR_ARG;
        at += lens[j];
    }
    if (std::set<std::string>(set->values.begin(), set->values.end()).size() != n)
        return MOD_ERR_ARG;
    *out = set.release();
    return MOD_OK;
}
#endif

extern "C" {

#if MOCK_SEARCH_ABI >= 1
int mod_plan_find_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                         uint64_t src_win_bytes, const uint8_t* pattern, uint32_t len, uint32_t* counts, mod_match* matches,
                         uint64_t cap, uint64_t* total, void* stream)
{
    return find_window(plan, t0, t1, src_win, src_win_off, src_win_bytes, pattern, nullptr, len, counts, matches, cap, total,
                       stream);
}

int mod_plan_find(const mod_plan* plan, const void* src, const uint8_t* pattern, uint32_t len, uint32_t* counts,
                  mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    return find_plan(plan, src, pattern, nullptr, len, counts, matches, cap, total, stream);
}

int mod_find_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, const uint8_t* pattern,
                   uint32_t len, uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total)
{
    return find_batch(descs, n, src, src_bytes, pattern, nullptr, len, counts, matches, cap, total);
}
#endif

#if MOCK_SEARCH_ABI >= 2
int mod_pattern_set_create(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out)
{
    return set_create(bytes, lens, n, false, out);
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
    return scan_window(plan, t0, t1, src_win, src_win_off, src_win_bytes, set, owned,
                       mock_results{counts, pattern_counts, nullptr, matches, cap, total}, stream);
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
    const int rc = set_create(bytes, lens, n_patterns, false, &set);
    if (rc != MOD_OK)
        return rc;
    std::unique_ptr<mod_pattern_set> owner(set);
    return scan_batch(descs, n, src, src_bytes, *set, mock_results{counts, pattern_counts, nullptr, matches, cap, total});
}
#endif

#if MOCK_SEARCH_ABI >= 3
int mod_plan_find_masked_window(const mod_plan* plan, uint64_t t0, uint64_t t1, const void* src_win, uint64_t src_win_off,
                                uint64_t src_win_bytes, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                                uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    if (!mask)
        return MOD_ERR_ARG;
    return find_window(plan, t0, t1, src_win, src_win_off, src_win_bytes, pattern, mask, len, counts, matches, cap, total,
                       stream);
}

int mod_plan_find_masked(const mod_plan* plan, const void* src, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                         uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total, void* stream)
{
    if (!mask)
        return MOD_ERR_ARG;
    return find_plan(plan, src, pattern, mask, len, counts, matches, cap, total, stream);
}

int mod_find_masked_batch(const mod_desc* descs, uint64_t n, const void* src, uint64_t src_bytes, const uint8_t* pattern,
                          const uint8_t* mask, uint32_t len, uint32_t* counts, mod_match* matches, uint64_t cap, uint64_t* total)
{
    if (!mask)
        return MOD_ERR_ARG;
    return find_batch(descs, n, src, src_bytes, pattern, mask, len, counts, matches, cap, total);
}

int mod_pattern_set_create_nocase(const uint8_t* bytes, const uint32_t* lens, uint32_t n, mod_pattern_set** out)
{
    return set_create(bytes, lens, n, true, out);
}
#endif
}
