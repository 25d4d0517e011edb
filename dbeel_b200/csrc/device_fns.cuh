// device_fns.cuh -- the scalar building blocks of the compaction kernels.
//
// Everything here is free of CUDA-only types: nvcc compiles it as `__device__` code, and
// g++ compiles the very same text into a host test shim (tests/host_shim.cc) so the
// arithmetic can be exercised on a box without a GPU.  Memory access is abstracted behind small loader callables so the
// kernels can use their own (vectorised, read-only-path) loads.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define DB_HD __device__ __forceinline__
#define DB_HOST_HD __host__ __device__ __forceinline__ // also called by host code of the engine (host/scan_plan.h)
#else
#define DB_HD inline
#define DB_HOST_HD inline
#endif

namespace dbeel {

// ------------------------------------------------------------------------------------
// Merge record: 16 bytes per input entry, the only thing the merge passes move.
//
//   x,y  key bytes [L, L+8)  as a big-endian u64 (x = high word), zero padded
//   z    key bytes [L+8, L+11) in bits 31..8, zero padded; bits 7..0 = clamp
//        clamp = min(klen - L, 12); 12 means "the key continues past the window"
//   w    gid = position of the entry in the concatenation of all input runs
//        (run-major), so gid order == (run position, index in run)
//
// L is the length of the byte prefix shared by every key of the job.  Comparing (x,y,z)
// as an unsigned tuple orders keys exactly like Rust's Vec<u8>::cmp (mod.rs:77-79)
// whenever the tuples differ or clamp < 12; equal tuples with clamp == 12 need the bytes
// past the window (full compare).
struct Rec {
    uint32_t x, y, z, w;
};

constexpr uint32_t kWindowBytes = 11;
constexpr uint32_t kClampBeyond = 12;
constexpr uint32_t kMaxPrefix = 255;

DB_HD uint64_t bswap64(uint64_t v) {
    v = ((v & 0x00FF00FF00FF00FFULL) << 8) | ((v >> 8) & 0x00FF00FF00FF00FFULL);
    v = ((v & 0x0000FFFF0000FFFFULL) << 16) | ((v >> 16) & 0x0000FFFF0000FFFFULL);
    return (v << 32) | (v >> 32);
}

// w0 / w1: little-endian loads of key bytes [L, L+8) and [L+8, L+16); bytes at or past the
// end of the key may hold anything.  rem = klen - L (bytes of key available from L).
DB_HD Rec make_rec(uint64_t w0, uint64_t w1, uint64_t rem, uint32_t gid) {
    uint64_t hi = bswap64(w0);
    if (rem < 8) hi = rem ? (hi & (~0ULL << (8 * (8 - rem)))) : 0;
    uint32_t nz = rem > 8 ? (rem - 8 > 3 ? 3u : (uint32_t)(rem - 8)) : 0u; // valid bytes in z
    uint32_t zb = ((uint32_t)(w1 & 0xFF) << 24) | ((uint32_t)((w1 >> 8) & 0xFF) << 16) |
                  ((uint32_t)((w1 >> 16) & 0xFF) << 8);
    zb = nz ? (zb & (~0u << (8 * (4 - nz)))) : 0u;
    uint32_t clamp = rem > kWindowBytes ? kClampBeyond : (uint32_t)rem;
    Rec r;
    r.x = (uint32_t)(hi >> 32);
    r.y = (uint32_t)hi;
    r.z = zb | clamp;
    r.w = gid;
    return r;
}

// -1 / 0 / +1 on the window; *undecided = 1 when the tuples tie and both keys continue.
DB_HD int rec_cmp_window(const Rec &a, const Rec &b, int *undecided) {
    *undecided = 0;
    if (a.x != b.x) return a.x < b.x ? -1 : 1;
    if (a.y != b.y) return a.y < b.y ? -1 : 1;
    if (a.z != b.z) return a.z < b.z ? -1 : 1;
    if ((a.z & 0xFF) == kClampBeyond) *undecided = 1;
    return 0;
}

// ------------------------------------------------------------------------------------
// SipHash-1-3 over `write_usize(klen) ++ key` -- what `Hash for Vec<u8>` feeds
// siphasher::sip::SipHasher13 (bloomfilter 1.0.12's item.hash(sip)).  The 8-byte length
// prefix keeps the key's 8-byte words aligned with SipHash's message words.
// ld(j) returns the little-endian u64 at key bytes [8j, 8j+8); bytes past klen are ignored.

#define DB_ROTL64(v, b) (((v) << (b)) | ((v) >> (64 - (b))))
#define DB_SIPROUND(v0, v1, v2, v3)                                     \
    do {                                                                \
        v0 += v1; v1 = DB_ROTL64(v1, 13); v1 ^= v0; v0 = DB_ROTL64(v0, 32); \
        v2 += v3; v3 = DB_ROTL64(v3, 16); v3 ^= v2;                     \
        v0 += v3; v3 = DB_ROTL64(v3, 21); v3 ^= v0;                     \
        v2 += v1; v1 = DB_ROTL64(v1, 17); v1 ^= v2; v2 = DB_ROTL64(v2, 32); \
    } while (0)

struct SipState {
    uint64_t v0, v1, v2, v3;
};

DB_HD SipState sip_init(uint64_t k0, uint64_t k1) {
    SipState s;
    s.v0 = k0 ^ 0x736f6d6570736575ULL;
    s.v1 = k1 ^ 0x646f72616e646f6dULL;
    s.v2 = k0 ^ 0x6c7967656e657261ULL;
    s.v3 = k1 ^ 0x7465646279746573ULL;
    return s;
}

DB_HD void sip_compress(SipState &s, uint64_t m) {
    s.v3 ^= m;
    DB_SIPROUND(s.v0, s.v1, s.v2, s.v3);
    s.v0 ^= m;
}

DB_HD uint64_t sip_finish(SipState &s, uint64_t last_block) {
    sip_compress(s, last_block);
    s.v2 ^= 0xff;
    DB_SIPROUND(s.v0, s.v1, s.v2, s.v3);
    DB_SIPROUND(s.v0, s.v1, s.v2, s.v3);
    DB_SIPROUND(s.v0, s.v1, s.v2, s.v3);
    return s.v0 ^ s.v1 ^ s.v2 ^ s.v3;
}

// Both bloom hashes in one walk over the key (the two hashers differ only in their keys).
template <class LoadU64>
DB_HD void sip13_pair_vec_u8(const uint64_t k[4], uint64_t klen, LoadU64 ld, uint64_t *h0, uint64_t *h1) {
    SipState a = sip_init(k[0], k[1]);
    SipState b = sip_init(k[2], k[3]);
    sip_compress(a, klen); // write_usize(len)
    sip_compress(b, klen);
    uint64_t nfull = klen >> 3;
    for (uint64_t j = 0; j < nfull; j++) {
        uint64_t m = ld(j);
        sip_compress(a, m);
        sip_compress(b, m);
    }
    uint32_t tail = (uint32_t)(klen & 7);
    uint64_t last = ((klen + 8) & 0xff) << 56;
    if (tail) last |= ld(nfull) & (~0ULL >> (8 * (8 - tail)));
    *h0 = sip_finish(a, last);
    *h1 = sip_finish(b, last);
}

// ------------------------------------------------------------------------------------
// Bloom bit positions (bloomfilter 1.0.12 bloom_hash + set).

constexpr uint64_t kBloomPrime = 0xFFFFFFFFFFFFFFC5ULL;

DB_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// h % d with magic = floor(2^64 / d), d >= 2: the estimate is low by at most one.
DB_HD uint64_t fastmod(uint64_t h, uint64_t d, uint64_t magic) {
    uint64_t q = mulhi64(h, magic);
    uint64_t r = h - q * d;
    return r >= d ? r - d : r;
}

// g_i of the double-hashing scheme: i = 0 -> h0, 1 -> h1, else (h0 + i*h1 mod 2^64) % prime.
DB_HD uint64_t bloom_hash_i(uint64_t h0, uint64_t h1, uint32_t i) {
    if (i == 0) return h0;
    if (i == 1) return h1;
    uint64_t g = h0 + (uint64_t)i * h1;
    return g >= kBloomPrime ? g - kBloomPrime : g; // prime > 2^63: at most one subtraction
}

// All k bit positions of one key, g_i computed incrementally: (h0 + i*h1) mod 2^64 is a running wrapping sum,
// so no per-probe multiply.  set_bit(bit) is called k_num times, in the order Bloom::set sets them.
template <class SetBit>
DB_HD void bloom_probe_all(uint64_t h0, uint64_t h1, uint32_t k_num, uint64_t bits, uint64_t bits_magic, SetBit set_bit) {
    set_bit(fastmod(h0, bits, bits_magic));
    if (k_num < 2) return;
    set_bit(fastmod(h1, bits, bits_magic));
    uint64_t acc = h0 + h1; // h0 + 1*h1
    for (uint32_t i = 2; i < k_num; i++) {
        acc += h1; // h0 + i*h1, wrapping
        const uint64_t g = acc >= kBloomPrime ? acc - kBloomPrime : acc;
        set_bit(fastmod(g, bits, bits_magic));
    }
}

// ------------------------------------------------------------------------------------
// Byte realignment for the gather kernel: 16 output bytes starting `sh` bytes into the
// 32-byte window {A, B} (A = lower-address 16 bytes).  sh in [0, 15]; B unused if sh == 0.

DB_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t bits) {
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, bits);
#else
    return bits ? (lo >> bits) | (hi << (32 - bits)) : lo;
#endif
}

DB_HD void realign16(const uint32_t A[4], const uint32_t B[4], uint32_t sh, uint32_t out[4]) {
    uint32_t bits = (sh & 3) * 8;
    uint32_t w0, w1, w2, w3, w4;
    switch (sh >> 2) {
    case 0: w0 = A[0]; w1 = A[1]; w2 = A[2]; w3 = A[3]; w4 = B[0]; break;
    case 1: w0 = A[1]; w1 = A[2]; w2 = A[3]; w3 = B[0]; w4 = B[1]; break;
    case 2: w0 = A[2]; w1 = A[3]; w2 = B[0]; w3 = B[1]; w4 = B[2]; break;
    default: w0 = A[3]; w1 = B[0]; w2 = B[1]; w3 = B[2]; w4 = B[3]; break;
    }
    out[0] = funnel_r(w0, w1, bits);
    out[1] = funnel_r(w1, w2, bits);
    out[2] = funnel_r(w2, w3, bits);
    out[3] = funnel_r(w3, w4, bits);
}

// 32 output bytes starting `s0` (0..31) bytes into the 64-byte window w[0..16) (little-endian words, lower address first).
// Words of the window that hold no wanted byte may contain anything.
DB_HD void window32(const uint32_t w[16], uint32_t s0, uint32_t out[8]) {
    const uint32_t bits = (s0 & 3) * 8;
    const bool s4 = (s0 & 16) != 0, s2 = (s0 & 8) != 0, s1 = (s0 & 4) != 0;
    uint32_t c[13], d[11], e[9]; // after the 16-, 8- and 4-byte steps
    for (int i = 0; i < 12; i++) c[i] = s4 ? w[i + 4] : w[i];
    c[12] = s4 ? 0u : w[12]; // only read when the shift is below 16 bytes
    for (int i = 0; i < 11; i++) d[i] = s2 ? c[i + 2] : c[i];
    for (int i = 0; i < 9; i++) e[i] = s1 ? d[i + 1] : d[i];
    for (int i = 0; i < 8; i++) out[i] = funnel_r(e[i], e[i + 1], bits);
}

// out = bytes [0, t) of T followed by bytes [t, 32) of H, t in 0..32.
DB_HD void blend32(const uint32_t T[8], const uint32_t H[8], uint32_t t, uint32_t out[8]) {
    const uint32_t wfull = t >> 2, bits = (t & 3) * 8;
    const uint32_t mmix = bits ? (0xFFFFFFFFu >> (32 - bits)) : 0u;
    for (uint32_t q = 0; q < 8; q++) {
        const uint32_t mk = q < wfull ? 0xFFFFFFFFu : (q == wfull ? mmix : 0u);
        out[q] = (T[q] & mk) | (H[q] & ~mk);
    }
}

// ------------------------------------------------------------------------------------
// i128 timestamp order (mod.rs:80) on the two little-endian halves.

DB_HD bool ts_greater(uint64_t alo, uint64_t ahi, uint64_t blo, uint64_t bhi) {
    if (ahi != bhi) return (int64_t)ahi > (int64_t)bhi;
    return alo > blo;
}

// Does this i128 nanosecond count decode as a timestamp (utils/timestamp_nanos.rs:15-24 ->
// time 0.3 OffsetDateTime::from_unix_timestamp_nanos)?  The crate floor-divides by 1e9, casts the quotient to
// i64 (wrapping) and range-checks the seconds against years -9999 ..= 9999.  Only the WAL replay needs it: there an
// undecodable entry is skipped, not fatal (lsm_tree.rs:562-566).
DB_HD bool ts_decodes(uint64_t lo, uint64_t hi) {
    const bool neg = (int64_t)hi < 0;
    uint64_t mlo = lo, mhi = hi;
    if (neg) { // magnitude = two's complement negation (2^127 fits in the unsigned pair)
        mlo = ~lo + 1;
        mhi = ~hi + (mlo == 0 ? 1 : 0);
    }
    constexpr uint64_t D = 1000000000ull;
    // long division of mhi:mlo by D; only the low 64 bits of the quotient survive the `as i64`
    uint64_t r = mhi % D;
    uint64_t t = (r << 32) | (mlo >> 32); // r < 2^30: fits
    const uint64_t q1 = t / D;
    r = t % D;
    t = (r << 32) | (mlo & 0xFFFFFFFFull);
    const uint64_t q0 = t / D;
    r = t % D;
    uint64_t q = (q1 << 32) + q0; // wraps like the cast does
    if (neg) q = ~(q + (r != 0 ? 1 : 0)) + 1; // floor for negatives, then negate (mod 2^64)
    const int64_t secs = (int64_t)q;
    return secs >= -377705116800ll && secs <= 253402300799ll;
}

// ------------------------------------------------------------------------------------
// murmur3_32 (crate murmur3 0.5.2 = MurmurHash3_x86_32): hash_bytes / hash_string of src/shards.rs:95-101, the hash the
// consistent-hash ring routes keys by.  ld64(q) returns the little-endian u64 at bytes [8q, 8q + 8) of the message; bytes
// at or past `len` may hold anything.

DB_HD uint32_t rotl32(uint32_t v, uint32_t r) { return (v << r) | (v >> (32 - r)); }

DB_HD uint32_t murmur3_mix_k(uint32_t k) {
    k *= 0xcc9e2d51u;
    k = rotl32(k, 15);
    return k * 0x1b873593u;
}

template <class LoadU64>
DB_HD uint32_t murmur3_32(uint64_t len, uint32_t seed, LoadU64 ld64) {
    uint32_t h = seed;
    const uint64_t nblocks = len >> 2;
    uint64_t w = 0;
    for (uint64_t b = 0; b < nblocks; b++) {
        if ((b & 1) == 0) w = ld64(b >> 1);
        const uint32_t k = (b & 1) ? (uint32_t)(w >> 32) : (uint32_t)w;
        h ^= murmur3_mix_k(k);
        h = rotl32(h, 13);
        h = h * 5u + 0xe6546b64u;
    }
    const uint32_t tail = (uint32_t)(len & 3);
    if (tail) {
        if ((nblocks & 1) == 0) w = ld64(nblocks >> 1);
        uint32_t k = (nblocks & 1) ? (uint32_t)(w >> 32) : (uint32_t)w;
        k &= 0xFFFFFFFFu >> (8 * (4 - tail));
        h ^= murmur3_mix_k(k);
    }
    h ^= (uint32_t)len;
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}

// Two murmur3_32 hashes (two seeds) in one walk over the message.
template <class LoadU64>
DB_HD void murmur3_32_pair(uint64_t len, uint32_t seed_a, uint32_t seed_b, LoadU64 ld64, uint32_t *out_a, uint32_t *out_b) {
    uint32_t ha = seed_a, hb = seed_b;
    const uint64_t nblocks = len >> 2;
    uint64_t w = 0;
    for (uint64_t b = 0; b < nblocks; b++) {
        if ((b & 1) == 0) w = ld64(b >> 1);
        const uint32_t k = murmur3_mix_k((b & 1) ? (uint32_t)(w >> 32) : (uint32_t)w);
        ha = rotl32(ha ^ k, 13) * 5u + 0xe6546b64u;
        hb = rotl32(hb ^ k, 13) * 5u + 0xe6546b64u;
    }
    const uint32_t tail = (uint32_t)(len & 3);
    if (tail) {
        if ((nblocks & 1) == 0) w = ld64(nblocks >> 1);
        uint32_t k = (nblocks & 1) ? (uint32_t)(w >> 32) : (uint32_t)w;
        k = murmur3_mix_k(k & (0xFFFFFFFFu >> (8 * (4 - tail))));
        ha ^= k;
        hb ^= k;
    }
    uint32_t h[2] = {ha ^ (uint32_t)len, hb ^ (uint32_t)len};
    for (int i = 0; i < 2; i++) {
        h[i] ^= h[i] >> 16;
        h[i] *= 0x85ebca6bu;
        h[i] ^= h[i] >> 13;
        h[i] *= 0xc2b2ae35u;
        h[i] ^= h[i] >> 16;
    }
    *out_a = h[0];
    *out_b = h[1];
}

// MyShard::owns_key with replica_index 0 (shards.rs:586-598, is_between :103-109): the position, on the ascending ring of
// shard hashes, of the shard that owns key_hash -- the first one whose hash is GREATER than key_hash, wrapping to 0.
template <class LoadRing>
DB_HD uint32_t ring_owner(uint32_t n_shards, uint32_t key_hash, LoadRing ring) {
    uint32_t lo = 0, hi = n_shards; // first position with ring(pos) > key_hash
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (ring(mid) > key_hash) hi = mid; else lo = mid + 1;
    }
    return lo == n_shards ? 0u : lo;
}

// ------------------------------------------------------------------------------------
// Hash-range scans (the iterator behind shard migration: migrate_actions, src/tasks/migration.rs:62-131, over
// LSMTree::iter_filter, src/storage_engine/lsm_tree.rs:133-282).

// between_cmp (migration.rs:54-60).  Scan mode 0 (DBEEL_SCAN_REFERENCE) is the literal predicate: a wrapped range
// (end < start) holds for every hash, start == end for none.  Mode 1 (DBEEL_SCAN_EXACT) reads a wrapped range as
// [start, 2^32) u [0, end).
DB_HD bool hash_in_range(uint32_t hash, uint32_t start, uint32_t end, uint32_t mode) {
    if (end < start) return mode ? (hash >= start || hash < end) : (hash < start || hash >= end);
    return start <= hash && hash < end;
}

// AsyncIter::read_one's read of one entry (lsm_tree.rs:250-262): read_at(offset, full_size) on the .data file.  The
// reference asserts full_size != 0 (cached_file_reader.rs:82) and panics on bytes past the end of the file; both stop a
// scan.  data_len is the .data file's length.
DB_HOST_HD bool entry_readable(uint64_t offset, uint32_t full_size, uint64_t data_len) {
    return full_size != 0 && offset <= data_len && (uint64_t)full_size <= data_len - offset;
}

// bincode Entry of EXACTLY full_size bytes (reject_trailing_bytes, utils/bincode.rs): klen:u64 | key | dlen:u64 | data |
// ts:i128, i.e. 8 + klen + 8 + dlen + 16 == full_size.  entry_key_fits is the part that depends on klen alone (dlen lies
// behind the key); entry_decodes is the whole rule, timestamp range included (utils/timestamp_nanos.rs).
DB_HD bool entry_key_fits(uint64_t full_size, uint64_t klen) { return full_size >= 32 && klen <= full_size - 32; }
DB_HD bool entry_decodes(uint64_t full_size, uint64_t klen, uint64_t dlen, uint64_t ts_lo, uint64_t ts_hi) {
    return entry_key_fits(full_size, klen) && dlen == full_size - 32 - klen && ts_decodes(ts_lo, ts_hi);
}

} // namespace dbeel
