// tests/cpp/mock_abi.h -- TEST INFRASTRUCTURE.  The objects the CPU mock of the C ABI (mock_abi.cpp, and the search
// entry points in mock_find_abi.cpp) shares between its translation units, and the oracle it answers with
// (oracle/cycle_oracle.c).  A plan is the descriptor list plus the real library's first-tile prefix (8 KiB tiles of
// one entry each); a plan and a stream remember the device they were created on.
#pragma once

#include <cstdint>
#include <vector>

#include "../../include/modulate_b200.h"

extern "C" {
void oracle_cycle_at(unsigned char* data, uint64_t size, int32_t key, uint64_t pos);
int32_t oracle_key_jump(int32_t key, uint64_t pos);
struct oracle_desc {
    uint64_t src_off, dst_off;
    uint32_t len;
    int32_t key;
};
void oracle_cycle_batch(const oracle_desc* d, uint64_t n, const unsigned char* src, unsigned char* dst);
}

struct mod_plan {
    std::vector<mod_desc> descs;
    std::vector<uint64_t> first_tile;  // n + 1
    uint32_t dst_align = 0;
    int device = 0;
};

struct mock_stream {
    int device;
};
