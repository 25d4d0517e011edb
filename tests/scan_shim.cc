// Host build of the hash-range scan's predicates in dbeel_b200/csrc/device_fns.cuh (the same text nvcc compiles as device
// code), exported with a C ABI so tests/test_scan_ranges.py can pin them without a GPU.
#include <stdint.h>
#include <string.h>

#include "../dbeel_b200/csrc/device_fns.cuh"

using namespace dbeel;

static uint64_t ld_le(const uint8_t *p, uint64_t avail) { // the classify kernel's u64 load; bytes past `avail` read 0xAA
    uint8_t b[8];
    for (int i = 0; i < 8; i++) b[i] = (uint64_t)i < avail ? p[i] : 0xAA;
    uint64_t v;
    memcpy(&v, b, 8);
    return v;
}

extern "C" {

int shim_hash_in_range(uint32_t h, uint32_t start, uint32_t end, uint32_t mode) { return hash_in_range(h, start, end, mode) ? 1 : 0; }

int shim_entry_readable(uint64_t offset, uint32_t full_size, uint64_t data_len) { return entry_readable(offset, full_size, data_len) ? 1 : 0; }

// the classify kernel's decode of one entry of n bytes: klen first, dlen and the timestamp only when the key fits
int shim_entry_decodes(const uint8_t *b, uint64_t n) {
    const uint64_t klen = ld_le(b, n);
    if (!entry_key_fits(n, klen)) return 0;
    uint64_t lo, hi;
    memcpy(&lo, b + n - 16, 8);
    memcpy(&hi, b + n - 8, 8);
    return entry_decodes(n, klen, ld_le(b + 8 + klen, n - 8 - klen), lo, hi) ? 1 : 0;
}
}
