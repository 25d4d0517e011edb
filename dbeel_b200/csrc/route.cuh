// route.cuh -- cfg5's shard routing on the GPU: hash every arrival's key with murmur3_32 (seed 0), find the shard that
// owns the hash on the consistent-hash ring, and split the arrival stream into one stream per shard, arrival order kept.
//
// Reference: hash_bytes / hash_string (src/shards.rs:95-101), the ring of shard names "<node>-<cpu id>"
// (shards.rs:213-214, sorted by hash :657-670), MyShard::owns_key with replica_index 0 (shards.rs:586-598: a shard owns
// [previous shard's hash, its own hash), is_between :103-109) as checked per request in src/tasks/db_server.rs:119-122.
//
// Only the 16-byte index records move.  A routed record keeps pointing into the batch's .data, so a shard's stream is an
// arrival batch with SPARSE offsets: dbeel_flush_many_sparse_device flushes it without copying a payload byte twice.
//
//   k_route_hash     per arrival: validate the frame, murmur3_32(key), owner; per-block histogram of owners
//                    (kClassIn: the owner -- any per-entry class id -- is already in shard_of; the hash-range scan,
//                    scan.cuh, classifies there and drops every entry at or after its stop ordinal here)
//   k_route_scan     one CTA per shard: exclusive scan of that shard's column over the blocks
//   k_route_starts   one warp: shard start positions (counts, bytes) -> pinned host block
//   k_route_scatter  per arrival: stable position = shard start + blocks before + warps before + lanes before
//                    (it moves whatever 16-byte record `index` holds: the scan hands it res records, kernels.cuh K4)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_fns.cuh"
#include "kernels.cuh"

namespace dbeel {

constexpr int kRouteThreads = 256;      // one arrival per thread
constexpr uint32_t kRouteMaxShards = 256; // smem: 8 warps x 256 counters

struct RouteParams {
    const uint8_t *data;
    uint64_t data_len;
    const uint4 *index;
    uint32_t n;
    const uint32_t *ring; // [n_shards] ascending shard hashes (device)
    uint32_t n_shards;
    uint32_t n_blocks;
    uint32_t *shard_of;               // [n] ring position per arrival (0xFFFFFFFF: undecodable)
    uint32_t *hist;                   // [n_blocks][n_shards] counts, then (k_route_scan) arrivals of the shard in earlier blocks
    unsigned long long *totals;       // [3 * n_shards + 1]: counts | payload bytes | starts ; [3 n_shards] = first bad record
    uint4 *out_index;                 // [n] routed records, shard-major
    unsigned long long *hash64;       // [n] arrival order: (murmur3_32(key, kCutSeed) << 32) | murmur3_32(key, 0), or null
    unsigned long long *out_hash64;   // [n] the same, shard-major (input of k_memtable_cuts)
    const unsigned long long *stop;   // k_route_hash<true>: (stop ordinal << 2) | reason -- entries at or after it count nowhere
};

constexpr uint32_t kCutSeed = 0x9747b28cu; // second murmur seed: the pair is the 64-bit key identity of the memtable cut

template <bool kClassIn>
__global__ void __launch_bounds__(kRouteThreads) k_route_hash(RouteParams p) {
    pdl_trigger();
    pdl_wait();
    __shared__ uint32_t s_cnt[kRouteMaxShards];
    __shared__ unsigned long long s_bytes[kRouteMaxShards];
    const uint32_t tid = threadIdx.x;
    for (uint32_t s = tid; s < p.n_shards; s += kRouteThreads) { s_cnt[s] = 0; s_bytes[s] = 0; }
    __syncthreads();
    const uint32_t i = blockIdx.x * (uint32_t)kRouteThreads + tid;
    if (kClassIn) {
        if (i < p.n) {
            uint32_t c = p.shard_of[i];
            if (c != 0xFFFFFFFFu && (unsigned long long)i >= (*p.stop >> 2)) { // behind the record that ends the scan
                c = 0xFFFFFFFFu;
                p.shard_of[i] = c;
            }
            if (c != 0xFFFFFFFFu) {
                atomicAdd(&s_cnt[c], 1u);
                atomicAdd(&s_bytes[c], (unsigned long long)__ldg(&p.index[i]).w);
            }
        }
    } else if (i < p.n) {
        const uint4 rec = __ldg(&p.index[i]);
        const uint64_t off = (uint64_t)rec.x | ((uint64_t)rec.y << 32);
        uint32_t owner = 0xFFFFFFFFu;
        if (rec.z >= 8 && (uint64_t)rec.w >= (uint64_t)rec.z + 24 && off <= p.data_len && (uint64_t)rec.w <= p.data_len - off) {
            const uint8_t *key = p.data + off + 8;
            uint32_t h, h2;
            murmur3_32_pair(rec.z - 8, 0u, kCutSeed, [key](uint64_t q) { return ld_u64_unaligned_narrow(key + 8 * q); }, &h, &h2);
            if (p.hash64) p.hash64[i] = ((unsigned long long)h2 << 32) | h;
            const uint32_t *ring = p.ring;
            owner = ring_owner(p.n_shards, h, [ring](uint32_t s) { return __ldg(&ring[s]); });
            atomicAdd(&s_cnt[owner], 1u);
            atomicAdd(&s_bytes[owner], (unsigned long long)rec.w);
        } else {
            atomicMin(&p.totals[3 * p.n_shards], (unsigned long long)i);
        }
        p.shard_of[i] = owner;
    }
    __syncthreads();
    for (uint32_t s = tid; s < p.n_shards; s += kRouteThreads) {
        p.hist[(uint64_t)blockIdx.x * p.n_shards + s] = s_cnt[s];
        if (s_bytes[s]) atomicAdd(&p.totals[p.n_shards + s], s_bytes[s]);
    }
}

__global__ void __launch_bounds__(1024) k_route_scan(RouteParams p) {
    pdl_trigger();
    pdl_wait();
    __shared__ unsigned long long s_b[32];
    __shared__ uint32_t s_c[32];
    const uint32_t s = blockIdx.x;
    uint32_t carry = 0;
    for (uint32_t b0 = 0; b0 < p.n_blocks; b0 += 1024) {
        const uint32_t b = b0 + threadIdx.x;
        const uint32_t v = b < p.n_blocks ? p.hist[(uint64_t)b * p.n_shards + s] : 0u;
        unsigned long long vb = 0, tb;
        uint32_t vc = v, tc;
        __syncthreads();
        block_excl_scan_1024(vb, vc, s_b, s_c, &tb, &tc);
        if (b < p.n_blocks) p.hist[(uint64_t)b * p.n_shards + s] = carry + vc;
        carry += tc;
    }
    if (threadIdx.x == 0) p.totals[s] = carry;
}

__global__ void k_route_starts(RouteParams p, unsigned long long *host_totals) {
    pdl_trigger();
    pdl_wait();
    if (threadIdx.x == 0) {
        unsigned long long acc = 0;
        for (uint32_t s = 0; s < p.n_shards; s++) {
            p.totals[2 * p.n_shards + s] = acc;
            acc += p.totals[s];
        }
    }
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < 3 * p.n_shards + 1; k += blockDim.x) host_totals[k] = p.totals[k];
    __threadfence_system();
}

__global__ void __launch_bounds__(kRouteThreads) k_route_scatter(RouteParams p) {
    pdl_trigger();
    pdl_wait();
    __shared__ uint32_t s_warp[kRouteThreads / 32][kRouteMaxShards]; // arrivals of shard s in warp w, then in the warps before w
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (uint32_t k = tid; k < (kRouteThreads / 32) * kRouteMaxShards; k += kRouteThreads) (&s_warp[0][0])[k] = 0;
    __syncthreads();
    const uint32_t i = blockIdx.x * (uint32_t)kRouteThreads + tid;
    const uint32_t owner = i < p.n ? p.shard_of[i] : 0xFFFFFFFFu;
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, owner);
    const uint32_t before = __popc(peers & ((1u << lane) - 1u)); // same shard, earlier arrival, same warp
    if (owner != 0xFFFFFFFFu && before == 0) s_warp[warp][owner] = __popc(peers);
    __syncthreads();
    for (uint32_t s = tid; s < p.n_shards; s += kRouteThreads) {
        uint32_t acc = 0;
        for (uint32_t w = 0; w < kRouteThreads / 32; w++) {
            const uint32_t c = s_warp[w][s];
            s_warp[w][s] = acc;
            acc += c;
        }
    }
    __syncthreads();
    if (owner == 0xFFFFFFFFu) return;
    const unsigned long long pos = p.totals[2 * p.n_shards + owner] + p.hist[(uint64_t)blockIdx.x * p.n_shards + owner] +
                                   s_warp[warp][owner] + before;
    p.out_index[pos] = __ldg(&p.index[i]);
    if (p.out_hash64) p.out_hash64[pos] = p.hash64[i];
}

// ------------------------------------------------------------------------------------
// Memtable-full trigger on the device (a11: lsm_tree.rs:747-765, the flush starts right after the insert that makes the
// tree hold `capacity` keys).  Input: one shard's stream of 64-bit key identities in arrival order; output: where every
// memtable ends.  One CTA per stream walks it 1024 arrivals at a time with a hash SET of the current memtable's keys in
// shared memory: insert (CAS), decide which thread of the chunk saw each new key FIRST (atomicMin of the thread index),
// prefix-sum those flags, and cut at the arrival that brings the count to `capacity`.
//
// The identity is a pair of murmur3 hashes, not the key bytes: two different keys colliding on all 64 bits would make a
// memtable one key too large.  The flush reports every memtable's exact distinct count, so callers verify
// items == capacity for every memtable but the last of a stream and fall back to dbeel_memtable_cut (exact, host) if not.

// Round 2 also tried 2048 arrivals per step with the next step prefetched (16.8 ms for the cfg5 stream instead of 22.3) and, on
// top of that, one table access per warp and key (__match_any_sync + a shuffle): the latter measured 33.0 ms on the same stream
// (profiles/r02_v5_bench_cfg5_n2.json, r02_v6_bench_cfg5.json) -- match.any costs more than the contention it removes.  This is
// the version of profiles/r02_v2_bench_cfg5.json (22.3 ms), restored as it was measured and tested.
constexpr uint32_t kCutSlots = 16384; // shared memory: 128 KB of identities + 64 KB of first-seen thread ids
constexpr uint32_t kCutMaxCapacity = 9216; // load factor <= (capacity + 1024) / slots = 0.625

struct CutParams {
    const unsigned long long *hash64; // shard-major
    const unsigned long long *starts; // [n_streams + 1] device
    uint32_t n_streams, capacity, max_cuts;
    const uint32_t *cut_base;         // [n_streams] device: first slot of stream s in `cuts`
    uint32_t *cuts;                   // arrivals of the stream consumed up to and including each FULL memtable
    uint32_t *n_cuts;                 // [n_streams]
};

__global__ void __launch_bounds__(1024) k_memtable_cuts(CutParams p) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(128) uint8_t s_raw[];
    unsigned long long *tab = reinterpret_cast<unsigned long long *>(s_raw);
    uint32_t *first = reinterpret_cast<uint32_t *>(s_raw + 8ull * kCutSlots);
    __shared__ unsigned long long s_b[32];
    __shared__ uint32_t s_c[32];
    __shared__ uint32_t s_cut;
    const uint32_t tid = threadIdx.x, stream = blockIdx.x;
    const unsigned long long base = p.starts[stream];
    const uint32_t n = (uint32_t)(p.starts[stream + 1] - base);
    const unsigned long long *h64 = p.hash64 + base;
    uint32_t *cuts = p.cuts + p.cut_base[stream];
    for (uint32_t k = tid; k < kCutSlots; k += 1024) { tab[k] = 0; first[k] = 0; }
    __syncthreads();
    uint32_t pos = 0, count = 0, ncut = 0;
    while (pos < n) {
        const uint32_t i = pos + tid;
        const bool act = i < n;
        unsigned long long h = act ? h64[i] : 0;
        if (act && h == 0) h = 1; // 0 marks an empty slot
        uint32_t slot = 0;
        bool won = false;
        if (act) {
            slot = (uint32_t)(h ^ (h >> 29)) & (kCutSlots - 1);
            while (true) {
                const unsigned long long cur = atomicCAS(&tab[slot], 0ull, h);
                if (cur == 0) { won = true; break; }
                if (cur == h) break;
                slot = (slot + 1) & (kCutSlots - 1);
            }
        }
        if (tid == 0) s_cut = 0xFFFFFFFFu;
        if (won) first[slot] = 0xFFFFFFFFu; // new in this chunk: someone's thread id goes here
        __syncthreads();
        if (act && first[slot] != 0) atomicMin(&first[slot], tid + 1);
        __syncthreads();
        const uint32_t flag = (act && first[slot] == tid + 1) ? 1u : 0u;
        unsigned long long vb = 0, tb;
        uint32_t vc = flag, tc;
        block_excl_scan_1024(vb, vc, s_b, s_c, &tb, &tc);
        if (flag && count + vc + 1 == p.capacity) s_cut = tid; // the insert that fills the tree
        __syncthreads();
        const uint32_t cut = s_cut;
        if (cut != 0xFFFFFFFFu) {
            pos += cut + 1;
            if (tid == 0 && ncut < p.max_cuts) cuts[ncut] = pos;
            ncut++;
            count = 0;
            for (uint32_t k = tid; k < kCutSlots; k += 1024) { tab[k] = 0; first[k] = 0; }
        } else {
            if (won) first[slot] = 0; // the key is old news for the chunks that follow
            count += tc;
            pos += 1024;
        }
        __syncthreads();
    }
    if (tid == 0) p.n_cuts[stream] = ncut;
}

} // namespace dbeel
