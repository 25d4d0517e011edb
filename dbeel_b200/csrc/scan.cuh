// scan.cuh -- hash-range scans of a tree on the GPU: the iterator behind shard migration.
//
// Reference: migrate_actions (src/tasks/migration.rs:62-131) walks the whole tree through LSMTree::iter_filter
// (src/storage_engine/lsm_tree.rs:133-282): every SSTable's records in index order, then the memtables; every entry whose
// murmur3_32(key) falls in one of the hash ranges goes to the FIRST range that holds (between_cmp, :54-60); the first
// record the iterator cannot yield ends the whole scan (`while let Ok(Some(entry))`, :96).
//
// One pass classifies every record, the routing kernels (route.cuh) split the survivors by range, and the compaction
// engine's offsets / gather kernels (kernels.cuh K4b, K5) pack them:
//
//   k_scan_classify   per record (global ordinal over all tables): index record, read / decode rule, murmur3_32(key),
//                     first matching range -> cls[i]; res record of every selected entry -> rec[i]; atomicMin of the
//                     ordinal (and reason) of every record that stops the scan
//   k_route_hash<true>, k_route_scan, k_route_starts, k_route_scatter
//                     stable split by range of the records before the stop, res records range-major
//   k_scan_plan       one CTA: range starts -> seg[0] (k_flush_table's group starts), entries to emit -> ctl->span,
//                     or nothing at all when the output does not fit the caller's buffers
//   k_scan_res_tiles  per 128 res records: bytes and entries (what k_resolve leaves for the offsets scan)
//   k_scan_tiles, k_scan_chunks, k_emit, k_gather32 / k_gather, k_flush_table, k_rebase_index
//                     exactly as a flush-many job runs them: every range's output is one file-relative SSTable
//
// The streamed form (dbeel_scan_ranges_stream) runs the same sequence once per partition (host/scan_plan.h: a run of
// consecutive records whose .data spans and index slices sit in a ring slot), with partition-local ordinals.  What
// crosses partitions stays on the device, so no partition waits for the host to learn about the one before it:
//
//   k_scan_part_enter      the partition's stop word: 0 (keep nothing) when an earlier partition stopped the scan
//   k_scan_rebase_stream   instead of k_rebase_index: .index offsets relative to the start of the range's whole stream
//   k_scan_part_leave      fold the partition's stop into the global one, add its per-range (bytes, items) to the running
//                          totals, write every range's piece (place in the output, stream offsets) to the pinned header
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_fns.cuh"
#include "kernels.cuh"
#include "route.cuh"

namespace dbeel {

constexpr uint32_t kScanMaxRanges = 256; // = kRouteMaxShards: one routing class per range
constexpr uint32_t kScanNone = 0xFFFFFFFFu;
constexpr uint32_t kScanStopDecode = 1u, kScanStopRead = 2u; // DBEEL_SCAN_DECODE / DBEEL_SCAN_READ
constexpr uint32_t kScanOverCap = 32u;                        // Ctl::flags: the output does not fit the caller's buffers

struct ScanTable {
    const uint8_t *data;
    uint64_t data_len;
    const uint4 *index;
    uint32_t base; // ordinal of the table's record 0
    uint32_t n;    // records (index_len / 16, never 0: the scan ends in front of an empty table)
};

struct ScanParams {
    const ScanTable *tables;
    uint32_t n_tables;
    uint32_t n;            // ordinals [0, n) are scanned
    const uint2 *ranges;   // [n_ranges] {start, end}
    uint32_t n_ranges;
    uint32_t mode;         // 0 = DBEEL_SCAN_REFERENCE, 1 = DBEEL_SCAN_EXACT
    uint32_t *cls;         // [n] range of every record, kScanNone = not selected (or it stops the scan)
    uint4 *rec;            // [n] {src_ptr lo, hi, 8 + klen, full_size} of every selected record (the rest untouched)
    unsigned long long *stop; // (first stopping ordinal << 2) | reason; host-initialised
    unsigned long long *totals; // route totals: counts | bytes | starts, per range
    Ctl *ctl;
    Seg *seg;              // [n_ranges] first res position of every range
    unsigned long long data_cap, index_cap;
};

__global__ void __launch_bounds__(256) k_scan_classify(ScanParams p) {
    __shared__ uint2 s_rng[kScanMaxRanges];
    const uint32_t tid = threadIdx.x;
    for (uint32_t k = tid; k < p.n_ranges; k += 256) s_rng[k] = p.ranges[k];
    __syncthreads();
    const uint32_t i = blockIdx.x * 256u + tid;
    if (i >= p.n) return;
    uint32_t lo = 0, hi = p.n_tables; // the table holding ordinal i: last one whose base <= i
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(&p.tables[mid].base) <= i) lo = mid; else hi = mid;
    }
    const ScanTable &t = p.tables[lo];
    const uint8_t *data = t.data;
    const uint4 ir = __ldg(&t.index[i - __ldg(&t.base)]); // neighbouring threads: neighbouring records
    const uint64_t off = (uint64_t)ir.x | ((uint64_t)ir.y << 32);
    const uint32_t fs = ir.w;
    uint32_t reason = 0, c = kScanNone;
    if (!entry_readable(off, fs, __ldg(&t.data_len))) {
        reason = kScanStopRead;
    } else {
        const uint8_t *ent = data + off;
        const uint64_t klen = ld_u64_unaligned_narrow(ent);
        bool ok = entry_key_fits(fs, klen);
        if (ok) {
            const uint64_t dlen = ld_u64_unaligned_narrow(ent + 8 + klen);
            const uint64_t ts_lo = ld_u64_unaligned_narrow(ent + fs - 16), ts_hi = ld_u64_unaligned_narrow(ent + fs - 8);
            ok = entry_decodes(fs, klen, dlen, ts_lo, ts_hi);
        }
        if (!ok) {
            reason = kScanStopDecode;
        } else {
            const uint8_t *key = ent + 8;
            const uint32_t h = murmur3_32(klen, 0u, [key](uint64_t q) { return ld_u64_unaligned_narrow(key + 8 * q); });
            for (uint32_t k = 0; k < p.n_ranges; k++)
                if (hash_in_range(h, s_rng[k].x, s_rng[k].y, p.mode)) { c = k; break; }
            if (c != kScanNone) {
                const unsigned long long src = (unsigned long long)(uintptr_t)ent;
                p.rec[i] = make_uint4((uint32_t)src, (uint32_t)(src >> 32), (uint32_t)(8 + klen), fs);
            }
        }
    }
    p.cls[i] = c;
    if (reason) atomicMin(p.stop, ((unsigned long long)i << 2) | reason);
}

// After k_route_starts: per-range starts for k_flush_table and the emitted entry count for the offsets scan -- or, when
// the selected bytes exceed a cap, an empty output (span 0: every later kernel writes nothing) and a flag for the host.
__global__ void k_scan_plan(ScanParams p) {
    if (threadIdx.x == 0) {
        unsigned long long count = 0, bytes = 0;
        for (uint32_t r = 0; r < p.n_ranges; r++) { count += p.totals[r]; bytes += p.totals[p.n_ranges + r]; }
        const bool fits = bytes <= p.data_cap && 16ull * count <= p.index_cap;
        p.ctl->span = fits ? (uint32_t)count : 0u;
        p.ctl->total = (uint32_t)count;
        p.ctl->flags = fits ? 0u : kScanOverCap;
    }
    for (uint32_t r = threadIdx.x; r < p.n_ranges; r += blockDim.x)
        p.seg[r] = Seg{(uint32_t)p.totals[2 * p.n_ranges + r], (uint32_t)p.totals[r]};
}

// The per-tile (bytes, entries) of the res records that k_resolve leaves for k_scan_tiles (kResolveThreads per tile).
__global__ void __launch_bounds__(kResolveThreads) k_scan_res_tiles(Params p, const uint4 *res) {
    __shared__ unsigned long long s_b[kResolveThreads / 32];
    __shared__ uint32_t s_c[kResolveThreads / 32];
    const uint32_t span = p.ctl->span;
    const uint32_t i0 = blockIdx.x * (uint32_t)kResolveThreads;
    if (i0 >= span) return;
    const uint32_t i = i0 + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long b = 0;
    uint32_t c = 0;
    if (i < span) { b = __ldg(&res[i]).w; c = 1; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        b += __shfl_down_sync(0xFFFFFFFFu, b, o);
        c += __shfl_down_sync(0xFFFFFFFFu, c, o);
    }
    if (lane == 0) { s_b[warp] = b; s_c[warp] = c; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (uint32_t w = 1; w < kResolveThreads / 32; w++) { b += s_b[w]; c += s_c[w]; }
        p.tile_bytes[blockIdx.x] = b;
        p.tile_count[blockIdx.x] = c;
    }
}

// ---- the streamed scan's cross-partition state

// One thread.  global_stop: (global ordinal << 2) | reason of the record that stopped the scan, ~0 = none yet.
__global__ void k_scan_part_enter(unsigned long long *local_stop, const unsigned long long *global_stop) {
    *local_stop = *global_stop == ~0ull ? ~0ull : 0ull; // 0: k_route_hash<true> drops every record of this partition
}

// k_rebase_index for a partition of a streamed scan: the offsets k_emit wrote count from the partition's output start;
// every range's stream continues where the range's pieces of the earlier partitions ended (run_tot[2 r], before
// k_scan_part_leave adds this partition).
__global__ void __launch_bounds__(256) k_scan_rebase_stream(Params p, const unsigned long long *run_tot) {
    const uint32_t e = blockIdx.x * 256u + threadIdx.x;
    if (e >= p.ctl->out_items) return;
    uint32_t lo = 0, hi = p.n_groups; // last range whose first entry is <= e (empty ranges share a boundary)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (p.mem_table[2 * mid + 1] <= e) lo = mid; else hi = mid;
    }
    uint4 rec = p.out_index[e];
    const unsigned long long off = ((unsigned long long)rec.x | ((unsigned long long)rec.y << 32)) - p.mem_table[2 * lo] + run_tot[2 * lo];
    rec.x = (uint32_t)off;
    rec.y = (uint32_t)(off >> 32);
    p.out_index[e] = rec;
}

// The per-range row of the pinned header (host/device mapped) that k_scan_part_leave writes for every partition.
struct ScanPieceRow {
    unsigned long long data_at, data_len; // .data bytes [data_at, data_at + data_len) of the partition's output
    unsigned long long items;             // .index records [items_at, items_at + items) of it
    unsigned long long items_at;
    unsigned long long stream_data_off, stream_items_off; // where they go in the range's stream (.index: 16 x items_off)
};

// One CTA.  mem_table: k_flush_table's rows of the partition; run_tot[2 r] / [2 r + 1]: .data bytes / items of range r
// written by the earlier partitions.  hdr: the global stop word, then n_ranges rows.
__global__ void k_scan_part_leave(const unsigned long long *mem_table, uint32_t n_ranges, const unsigned long long *local_stop,
                                  unsigned long long *global_stop, unsigned long long first_ordinal, unsigned long long *run_tot,
                                  unsigned long long *hdr) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long l = *local_stop;
        if (*global_stop == ~0ull && l != ~0ull) *global_stop = ((first_ordinal + (l >> 2)) << 2) | (l & 3);
        hdr[0] = *global_stop;
    }
    ScanPieceRow *rows = reinterpret_cast<ScanPieceRow *>(hdr + 1);
    for (uint32_t r = threadIdx.x; r < n_ranges; r += blockDim.x) {
        const unsigned long long b0 = mem_table[2 * r], b1 = mem_table[2 * (r + 1)], i0 = mem_table[2 * r + 1], i1 = mem_table[2 * (r + 1) + 1];
        ScanPieceRow row;
        row.data_at = b0;
        row.data_len = b1 - b0;
        row.items_at = i0;
        row.items = i1 - i0;
        row.stream_data_off = run_tot[2 * r];
        row.stream_items_off = run_tot[2 * r + 1];
        rows[r] = row;
        run_tot[2 * r] += b1 - b0;
        run_tot[2 * r + 1] += i1 - i0;
    }
    __threadfence_system(); // visible to the host before the stream reports completion
}

} // namespace dbeel
