// dbeel_compact.cu -- engine + C ABI (include/dbeel_compact.h) over the kernels in kernels.cuh.
//
// One engine = one GPU + one stream + a grow-only device workspace.  A compaction job is a
// fixed sequence of kernel launches with no host round trip in between; the only host sync
// is the final read-back of the 300-byte control block (output lengths, flags).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <deque>
#include <memory>
#include <new>
#include <thread>
#include <string>
#include <vector>

#include "../../include/dbeel_compact.h"
#include "kernels.cuh"
#include "merge_final.cuh"
#include "gather_async.cuh"
#include "gather_fb.cuh"
#include "lookup.cuh"
#include "route.cuh"
#include "scan.cuh"
#include "wal.cuh"
#include "host/scan_plan.h"
#include "host/stream_pump.h"

using namespace dbeel;

namespace {

constexpr uint64_t kAlign = 256;
inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

enum { EV_START = 0, EV_EXTRACT, EV_MERGE, EV_RESOLVE, EV_GATHER, EV_H2D0, EV_H2D1, EV_D2H0, EV_D2H1, EV_COUNT };

} // namespace

struct dbeel_engine {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[EV_COUNT] = {};
    // device workspace (grow-only)
    uint8_t *ws = nullptr;
    uint64_t ws_cap = 0;
    // device staging for the host entry points (grow-only)
    uint8_t *stage_in = nullptr, *stage_out = nullptr;
    uint64_t stage_in_cap = 0, stage_out_cap = 0;
    // pipelined host path: second staging pair, copy streams, shared bloom buffer
    uint8_t *stage_in2 = nullptr, *stage_out2 = nullptr, *bloom_dev = nullptr;
    uint64_t stage_in2_cap = 0, stage_out2_cap = 0, bloom_dev_cap = 0;
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[2] = {}, ev_comp[2] = {}, ev_d2h[2] = {};
    int pipeline = 1;                   // DBEEL_PIPELINE: 0 = single-shot host path
    uint64_t pipeline_min_bytes = 64ull << 20;
    uint64_t partition_bytes = 256ull << 20; // DBEEL_PARTITION_MB
    int partition_taper = 1;                 // DBEEL_PARTITION_TAPER: small first / last partitions (A/B switch)
    // streaming host path (dbeel_compact_stream): pinned rings the file bytes pass through, the runs' .index files, the filter
    // on its way out (grow-only, page-locked)
    uint8_t *ring_in = nullptr, *ring_out = nullptr, *pin_index = nullptr, *pin_bloom = nullptr;
    uint64_t ring_in_cap = 0, ring_out_cap = 0, pin_index_cap = 0, pin_bloom_cap = 0;
    int stream_ring = 3;                     // DBEEL_STREAM_RING: slots per ring (>= 2)
    // pinned host block: job header going down, control block coming back
    uint8_t *wal_ws = nullptr; // WAL replay: doubling tables + the arrival index (grow-only)
    uint64_t wal_ws_cap = 0;
    uint8_t *route_ws = nullptr; // shard routing: owners, block histograms, totals (grow-only)
    uint64_t route_ws_cap = 0;
    uint8_t *pin = nullptr;
    uint8_t *pin_dev = nullptr; // the same block as the GPU sees it (mapped: kernels read the header / write the control block)
    uint64_t pin_cap = 0;
    dbeel_stats stats = {};
    std::string err;
    bool busy = false;
    // asynchronous jobs (dbeel_compact_submit)
    std::thread worker;
    std::atomic<int> async_state{0}; // 0 idle, 1 running, 2 finished (status in async_status)
    int async_status = 0;
    std::vector<dbeel_run> async_runs;
    dbeel_compact_opts async_opts = {};
    uint8_t async_seed[32] = {};
    int sm_count = 148;
    int merge_variant = 1;      // DBEEL_MERGE: 0 = one CTA per tile with plain loads, 1 = persistent TMA (default)
    int narrow_loads = 1;       // DBEEL_NARROW: .L2::64B loads for random accesses in extract / resolve (A/B switch)
    int gather_variant = 10;    // DBEEL_GATHER: 10 = k_gather32 with the lean entry-boundary pass (default), 0 = 16 bytes per lane (k_gather),
                                //               1 = 32 bytes per lane + 256-bit stores (k_gather32, round 1's boundary pass),
                                //               2 = 1 with the payload staged into shared memory by TMA bulk copies (k_gather_tma)
    int fused_emit = 0;         // DBEEL_FUSED_EMIT: 1 = resolve + offsets scan + .index writes in one kernel (single jobs), 0 = four kernels
    int bloom_side = 0;         // DBEEL_BLOOM_SIDE: 1 = k_bloom_res on a second stream (measured: kernels of two streams do not co-run, the
                                // filter pass just moves in front of k_emit: +0.16 ms per job, DESIGN.md); 0 = the gather's fused epilogue
    cudaStream_t s_side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int fused_final = 0;        // DBEEL_FUSED_FINAL: 1 = last merge level + resolve + offsets scan + .index writes in one persistent kernel
                                // (k_merge_final, single compactions: 0.4 GB less DRAM traffic per cfg2 job, but 0.45 ms against 0.34 ms for
                                // the five kernels it replaces -- latency-bound at 2 CTAs/SM, DESIGN.md), 0 = the five kernels
    int fin_ctas_per_sm = 0;    // co-resident k_merge_final CTAs per SM (occupancy query at engine creation): its chained scan needs them all resident
    int pdl = 0;                // DBEEL_PDL: 1 = the job's kernels are launched with programmatic stream serialization (griddepcontrol)
    int stage_events = 1;       // DBEEL_STAGE_EVENTS: 0 = no per-stage event records inside a job (stage_ms read 0)
    int extract_persist = 6;    // DBEEL_EXTRACT_PERSIST: > 0 = k_extract runs as that many CTAs per SM, each thread fetching the next step's index
                                // records while the current step's entry headers travel
    int bloom_in_extract = 0;   // DBEEL_BLOOM_EXTRACT: 1 = k_extract hashes, k_resolve sets the bits (measured slower: DESIGN.md); 0 = the gather's fused epilogue
};

namespace {

int fail(dbeel_engine *e, int code, const char *what, cudaError_t ce = cudaSuccess) {
    char buf[512];
    if (ce != cudaSuccess)
        snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorName(ce), cudaGetErrorString(ce));
    else
        snprintf(buf, sizeof buf, "%s", what);
    if (e) e->err = buf;
    return code;
}

#define CU(call)                                                            \
    do {                                                                    \
        cudaError_t ce_ = (call);                                           \
        if (ce_ != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, #call, ce_); \
    } while (0)

int ensure_device(dbeel_engine *e, uint8_t **buf, uint64_t *cap, uint64_t need) {
    if (need <= *cap) return DBEEL_OK;
    if (*buf) { cudaFree(*buf); *buf = nullptr; *cap = 0; }
    uint64_t want = align_up(need + need / 8, 1 << 20);
    cudaError_t ce = cudaMalloc(reinterpret_cast<void **>(buf), want);
    if (ce != cudaSuccess) {
        cudaGetLastError();
        want = align_up(need, 1 << 20);
        ce = cudaMalloc(reinterpret_cast<void **>(buf), want);
    }
    if (ce != cudaSuccess) { cudaGetLastError(); return fail(e, DBEEL_ERR_NOMEM, "cudaMalloc(workspace)", ce); }
    *cap = want;
    return DBEEL_OK;
}

int ensure_pinned(dbeel_engine *e, uint64_t need) {
    if (need <= e->pin_cap) return DBEEL_OK;
    if (e->pin) cudaFreeHost(e->pin);
    e->pin = nullptr;
    e->pin_dev = nullptr;
    e->pin_cap = 0;
    cudaError_t ce = cudaHostAlloc(reinterpret_cast<void **>(&e->pin), need, cudaHostAllocMapped);
    if (ce != cudaSuccess) { cudaGetLastError(); return fail(e, DBEEL_ERR_NOMEM, "cudaHostAlloc", ce); }
    ce = cudaHostGetDevicePointer(reinterpret_cast<void **>(&e->pin_dev), e->pin, 0);
    if (ce != cudaSuccess) { cudaGetLastError(); return fail(e, DBEEL_ERR_CUDA, "cudaHostGetDevicePointer", ce); }
    e->pin_cap = need;
    return DBEEL_OK;
}

// grow-only page-locked host buffer (the streaming path's rings)
int ensure_host(dbeel_engine *e, uint8_t **buf, uint64_t *cap, uint64_t need) {
    if (need <= *cap) return DBEEL_OK;
    if (*buf) { cudaFreeHost(*buf); *buf = nullptr; *cap = 0; }
    const uint64_t want = align_up(need + need / 8, 1 << 20);
    cudaError_t ce = cudaHostAlloc(reinterpret_cast<void **>(buf), want, cudaHostAllocDefault);
    if (ce != cudaSuccess) { cudaGetLastError(); *buf = nullptr; return fail(e, DBEEL_ERR_NOMEM, "cudaHostAlloc(stream ring)", ce); }
    *cap = want;
    return DBEEL_OK;
}

int stream_threads() {
    static const int n = [] {
        if (const char *v = getenv("DBEEL_IO_THREADS")) return std::max(1, atoi(v));
        const unsigned hw = std::thread::hardware_concurrency();
        return (int)std::min(8u, std::max(2u, hw / 8)); // readers and writers each (measured on the 128-thread box: 8 + 8 = 16 + 16, 32 + 32 loses)
    }();
    return n;
}

// n independent pieces of callback I/O over a few threads; the first nonzero return code wins
template <class F>
int parallel_pieces(size_t n, F fn) {
    std::atomic<size_t> next{0};
    std::atomic<int> err{0};
    auto work = [&]() {
        for (size_t k = next.fetch_add(1); k < n && !err.load(); k = next.fetch_add(1)) {
            const int rc = fn(k);
            if (rc) { int z = 0; err.compare_exchange_strong(z, rc); }
        }
    };
    const int nt = (int)std::min<size_t>((size_t)stream_threads(), n);
    std::vector<std::thread> pool;
    for (int i = 1; i < nt; i++) pool.emplace_back(work);
    work();
    for (auto &t : pool) t.join();
    return err.load();
}

void default_opts(dbeel_compact_opts *o) {
    o->keep_tombstones = 0;
    o->flags = 0;
    o->bloom_min_size = DBEEL_DEFAULT_BLOOM_MIN_SIZE;
    o->bloom_fp = DBEEL_DEFAULT_BLOOM_FP;
    o->bloom_seed = nullptr;
}

// Kernel launch with (optionally) the programmatic-stream-serialization attribute: the kernel may be scheduled while its
// predecessor in the stream drains; every kernel starts with griddepcontrol.wait, so stream order is kept (kernels.cuh).
template <typename... KArgs, typename... Args>
void launch_k(const dbeel_engine *e, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = e->pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

struct JobShape {
    uint64_t n_total = 0; // sum of index_len / 16
    uint64_t data_total = 0;
    uint64_t index_total = 0; // sum of index_len (raw)
    uint64_t bloom_file = 0;  // 0 = no bloom
    uint64_t bloom_bits = 0, bloom_words = 0;
    uint32_t bloom_k = 0;
};

int shape_of(const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *o, bool flush, JobShape *s) {
    for (uint32_t r = 0; r < n_runs; r++) {
        s->n_total += runs[r].index_len / DBEEL_INDEX_ENTRY_SIZE;
        s->data_total += runs[r].data_len;
        s->index_total += runs[r].index_len;
    }
    // lsm_tree.rs:1026-1034: sized for the INPUT entry count, enabled on input .data bytes
    if (!flush && s->n_total > 0 && s->data_total > o->bloom_min_size) {
        uint64_t bytes = dbeel_bloom_bitmap_bytes(s->n_total, o->bloom_fp);
        s->bloom_bits = bytes * 8;
        s->bloom_words = (s->bloom_bits + 31) / 32;
        s->bloom_k = dbeel_bloom_k_num(s->bloom_bits, s->n_total);
        s->bloom_file = 8 + 4 * s->bloom_words + 8 + 8 + 4 + 144;
    }
    return DBEEL_OK;
}

// Set when a job is one key-range partition of a larger compaction (host entry point, section "pipelined").
struct JobExtra {
    const uint64_t *off_base = nullptr; // [n_runs] .data offset of each run slice's first byte; data pointers are pre-biased
    uint64_t out_offset_base = 0;       // .data bytes the earlier partitions wrote
    bool external_bloom = false;        // the filter belongs to the whole compaction: set bits only
    BloomParams bloom = {};
    dbeel_flush_table *flush_table = nullptr; // flush-many: one row per batch (host memory), filled on success
    // compact-many: runs[] holds all jobs' runs back to back; job g = runs[job_first[g] .. job_first[g+1])
    uint32_t n_jobs = 0;
    const uint32_t *job_first = nullptr;     // [n_jobs + 1]
    const int32_t *job_keep = nullptr;       // [n_jobs] keep_tombstones
    const BloomParams *job_bloom = nullptr;  // [n_jobs] device-side filter of each job (words == null: none)
    dbeel_job_result *job_results = nullptr; // [n_jobs] filled on success (bloom_off / bloom_len are the caller's)
    bool sparse_offsets = false;        // WAL replay: the batch's .data is the log itself, records do not abut
    uint64_t data_bytes = 0;            // with sparse_offsets: sum of the records' sizes (the output bound)
};

// The whole device-resident job.  `runs` / `out` hold device pointers.
int run_job_device(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *o,
                   bool flush, dbeel_out *out, bool record_start, const JobExtra *extra = nullptr) {
    JobShape sh;
    shape_of(runs, n_runs, o, flush, &sh);
    if (extra && (extra->external_bloom || extra->n_jobs)) sh.bloom_file = 0; // compact-many: per-job filters, sized by the caller
    const uint64_t span_total = sh.data_total; // address span of the inputs (sh.data_total becomes the payload bound)
    if (extra && extra->sparse_offsets) sh.data_total = extra->data_bytes;
    (void)span_total;
    if (n_runs > DBEEL_MAX_RUNS) return fail(e, DBEEL_ERR_TOO_MANY_RUNS, "too many runs");
    if (sh.n_total >= 0xFFFFFFFEull) return fail(e, DBEEL_ERR_TOO_MANY_ENTRIES, "too many entries");
    if (out->data_cap < sh.data_total || out->index_cap < sh.n_total * 16 || out->bloom_cap < sh.bloom_file)
        return fail(e, DBEEL_ERR_CAPACITY, "output buffer smaller than dbeel_compact_bound");
    for (uint32_t r = 0; r < n_runs; r++) {
        if ((runs[r].data_len && !runs[r].data) || (runs[r].index_len >= 16 && !runs[r].index))
            return fail(e, DBEEL_ERR_INVALID_ARG, "null run buffer");
        // .data may start anywhere (every access realigns; tables left by dbeel_flush_many / dbeel_compact_many are slices of
        // one output stream); .index is read as 16-byte records
        if ((uintptr_t)runs[r].index & 15) return fail(e, DBEEL_ERR_INVALID_ARG, "device .index buffers must be 16-byte aligned");
    }
    if (((uintptr_t)out->data | (uintptr_t)out->index | (uintptr_t)out->bloom) & 15)
        return fail(e, DBEEL_ERR_INVALID_ARG, "device output buffers must be 16-byte aligned");
    if ((sh.data_total && !out->data) || (sh.n_total && !out->index) || (sh.bloom_file && !out->bloom))
        return fail(e, DBEEL_ERR_INVALID_ARG, "null output buffer");

    dbeel_stats &st = e->stats;
    float h2d = st.ms_h2d; // set by the host wrapper before we get here
    memset(&st, 0, sizeof st);
    st.ms_h2d = h2d;
    st.input_bytes = sh.data_total + sh.index_total;
    st.entries_in = sh.n_total;
    out->data_len = out->index_len = out->bloom_len = out->items_written = 0;

    const uint32_t N = (uint32_t)sh.n_total;
    if (N == 0) return DBEEL_OK; // nothing decodable: empty output, no bloom

    // ---- plan the levels
    Params p;
    memset(&p, 0, sizeof p);
    p.n_runs = n_runs;
    p.n_total = N;
    p.keep_tombstones = o->keep_tombstones ? 1 : 0;
    p.mode_flush = flush ? 1 : 0;
    uint32_t levels = 0;
    const bool many = flush && extra && extra->flush_table;
    const bool jobs = !flush && extra && extra->n_jobs;
    if (jobs) {
        // every job gets the same power-of-two number of leaf slots (its runs, then empty segments): log2(slots)
        // pairwise levels finish every job and never pair runs of two different ones
        uint32_t max_runs = 1;
        for (uint32_t g = 0; g < extra->n_jobs; g++) max_runs = std::max(max_runs, extra->job_first[g + 1] - extra->job_first[g]);
        uint32_t slots = 1;
        while (slots < max_runs) slots <<= 1;
        if ((uint64_t)slots * extra->n_jobs > (1ull << 20)) return fail(e, DBEEL_ERR_TOO_MANY_RUNS, "compact-many: too many run slots");
        p.group_slots = slots;
        p.n_groups = extra->n_jobs;
        p.nseg[0] = slots * extra->n_jobs;
        while ((1u << levels) < slots) {
            p.nseg[levels + 1] = p.nseg[levels] / 2;
            levels++;
        }
    } else if (many) {
        p.n_groups = n_runs;
        // every memtable gets the same power-of-two number of leaf slots (sort tiles), so log2(slots) merge levels
        // finish all memtables and never pair segments of two different ones
        uint64_t max_tiles = 1;
        for (uint32_t r = 0; r < n_runs; r++) {
            const uint64_t t = (runs[r].index_len / DBEEL_INDEX_ENTRY_SIZE + kMergeTile - 1) / kMergeTile;
            max_tiles = t > max_tiles ? t : max_tiles;
        }
        uint32_t slots = 1;
        while (slots < max_tiles) slots <<= 1;
        if (slots > (1u << kMaxLevels) || (uint64_t)slots * n_runs > (1ull << 24))
            return fail(e, DBEEL_ERR_TOO_MANY_ENTRIES, "flush-many: too many sort tiles");
        p.flush_slots = slots;
        p.nseg[0] = slots * n_runs;
        while ((1u << levels) < slots) {
            p.nseg[levels + 1] = p.nseg[levels] / 2;
            levels++;
        }
        for (uint32_t r = 0; r < n_runs; r++)
            if (runs[r].index_len >= DBEEL_INDEX_ENTRY_SIZE) { p.flush_ref_run = r; break; }
    } else {
        p.nseg[0] = flush ? (N + kMergeTile - 1) / kMergeTile : n_runs;
        if (p.nseg[0] > (1u << kMaxLevels)) return fail(e, DBEEL_ERR_TOO_MANY_ENTRIES, "arrival batch too large for one flush");
        while (p.nseg[levels] > 1) {
            p.nseg[levels + 1] = (p.nseg[levels] + 1) / 2;
            levels++;
        }
    }
    p.n_levels = levels;

    // ---- carve the workspace
    uint64_t off = 0;
    auto carve = [&](uint64_t bytes) { uint64_t o2 = off; off = align_up(off + bytes, kAlign); return o2; };
    // header block (host-initialised, one H2D copy): ctl | runs | first_bad | first_mismatch
    const uint64_t o_ctl = carve(sizeof(Ctl));
    const uint64_t o_runs = carve(sizeof(RunDesc) * n_runs);
    const uint64_t o_fbad = carve(4ull * n_runs);
    const uint64_t o_fmis = carve(4ull * n_runs);
    const uint64_t o_groups = carve(jobs ? sizeof(GroupDesc) * (uint64_t)extra->n_jobs : 0);
    const uint64_t header_bytes = off;
    uint64_t o_seg[kMaxLevels + 1], o_tb[kMaxLevels];
    for (uint32_t l = 0; l <= levels; l++) o_seg[l] = carve(sizeof(Seg) * p.nseg[l]);
    for (uint32_t l = 0; l < levels; l++) o_tb[l] = carve(4ull * (p.nseg[l + 1] + 1));
    const uint64_t tiles_ub = (uint64_t)(N + kFinNominal - 1) / kFinNominal + (p.nseg[0] + 1) / 2; // kFinNominal < kMergeTile: covers both
    const uint64_t bounds_ub = tiles_ub + (p.nseg[0] + 1) / 2 + 1;
    const uint64_t o_part = carve(4 * bounds_ub);
    const uint64_t o_pext = carve(4 * bounds_ub);
    const uint64_t o_bnd = carve(16 * (bounds_ub + 1));
    const uint64_t o_tbnd = carve(4 * (tiles_ub + 1));
    const uint64_t res_tiles = (uint64_t)(N + kResolveThreads - 1) / kResolveThreads;
    const uint64_t o_tbytes = carve(res_tiles * 8), o_tcount = carve(res_tiles * 4);
    const uint64_t res_chunks = (res_tiles + 1023) / 1024;
    const uint64_t o_cbytes = carve(res_chunks * 8), o_ccount = carve(res_chunks * 4);
    const uint64_t o_reca = carve(16ull * N), o_recb = carve(16ull * N);
    const uint64_t o_src = carve(8ull * N);
    const uint64_t n_groups = p.n_groups;
    const uint64_t o_memtab = carve(n_groups ? 16ull * (n_groups + 1) : 0);
    const uint64_t gather_tiles = (sh.data_total + kGatherTileBytes - 1) / kGatherTileBytes;
    const uint64_t o_tfirst = carve(4ull * (gather_tiles + 2));
    const bool ref_reader = !flush && !jobs && (o->flags & DBEEL_FLAG_REFERENCE_READER);
    const uint64_t o_fix = carve(ref_reader ? 16ull * N : 0);
    // single job with a filter: k_extract leaves both SipHash values of every key here and k_resolve sets the survivors' bits
    const bool hash_early = e->bloom_in_extract && !flush && !jobs && (sh.bloom_file || (extra && extra->external_bloom && extra->bloom.words));
    const uint64_t o_hash = carve(hash_early ? 16ull * N : 0);
    // single compaction: resolve, the offsets scan and the .index writes in one kernel (chained scan over the tiles)
    const bool fused_emit = e->fused_emit && !flush && !jobs && !many && !hash_early && !(e->bloom_side && sh.bloom_file);
    // single compaction: the last merge level, resolve, the offsets scan and the .index writes in one persistent kernel
    const bool fused_final = e->fused_final && e->fin_ctas_per_sm > 0 && !flush && !jobs && !many && !hash_early && !fused_emit && levels >= 1 &&
                             !(e->bloom_side && sh.bloom_file);
    const uint64_t fin_tiles_ub = (uint64_t)(N + kFinNominal - 1) / kFinNominal + 1;
    p.fin_tile = fused_final ? (uint32_t)kFinNominal : 0u;
    const uint64_t scan_bytes = fused_emit ? 16ull * res_tiles + 64 : (fused_final ? 16ull * fin_tiles_ub + 64 : 0);
    const uint64_t o_scan = carve(scan_bytes);
    int rc = ensure_device(e, &e->ws, &e->ws_cap, off);
    if (rc) return rc;
    rc = ensure_pinned(e, header_bytes + align_up(sizeof(Ctl), 64) + 64 + (n_groups ? 16ull * (n_groups + 1) : 0));
    if (rc) return rc;

    uint8_t *ws = e->ws;
    p.ctl = reinterpret_cast<Ctl *>(ws + o_ctl);
    p.runs = reinterpret_cast<RunDesc *>(ws + o_runs);
    p.first_bad = reinterpret_cast<uint32_t *>(ws + o_fbad);
    p.first_mismatch = reinterpret_cast<uint32_t *>(ws + o_fmis);
    for (uint32_t l = 0; l <= levels; l++) p.seg[l] = reinterpret_cast<Seg *>(ws + o_seg[l]);
    for (uint32_t l = 0; l < levels; l++) p.tile_base[l] = reinterpret_cast<uint32_t *>(ws + o_tb[l]);
    p.part = reinterpret_cast<uint32_t *>(ws + o_part);
    p.part_ext = reinterpret_cast<uint32_t *>(ws + o_pext);
    p.bnd = reinterpret_cast<uint4 *>(ws + o_bnd);
    p.tile_bnd = reinterpret_cast<uint32_t *>(ws + o_tbnd);
    p.tile_bytes = reinterpret_cast<unsigned long long *>(ws + o_tbytes);
    p.tile_count = reinterpret_cast<uint32_t *>(ws + o_tcount);
    p.chunk_bytes = reinterpret_cast<unsigned long long *>(ws + o_cbytes);
    p.chunk_count = reinterpret_cast<uint32_t *>(ws + o_ccount);
    p.rec_a = reinterpret_cast<Rec *>(ws + o_reca);
    p.rec_b = reinterpret_cast<Rec *>(ws + o_recb);
    p.src_ptr = reinterpret_cast<unsigned long long *>(ws + o_src);
    p.tile_first = reinterpret_cast<uint32_t *>(ws + o_tfirst);
    p.tile_first_n = (uint32_t)(gather_tiles + 2);
    p.mem_table = reinterpret_cast<unsigned long long *>(ws + o_memtab);
    p.ref_reader = ref_reader ? 1 : 0;
    p.fix_index = reinterpret_cast<uint4 *>(ws + o_fix);
    p.hash_rec = hash_early ? reinterpret_cast<uint4 *>(ws + o_hash) : nullptr;
    p.scan_state = reinterpret_cast<unsigned long long *>(ws + o_scan);
    p.scan_ticket = reinterpret_cast<uint32_t *>(ws + o_scan + 16ull * res_tiles);
    p.out_data = static_cast<uint8_t *>(out->data);
    p.out_index = static_cast<uint4 *>(out->index);

    // ---- header block
    uint8_t *h = e->pin;
    memset(h, 0, header_bytes);
    RunDesc *hr = reinterpret_cast<RunDesc *>(h + o_runs);
    uint32_t *hb = reinterpret_cast<uint32_t *>(h + o_fbad), *hm = reinterpret_cast<uint32_t *>(h + o_fmis);
    uint32_t base = 0;
    for (uint32_t r = 0; r < n_runs; r++) {
        hr[r].data = static_cast<const uint8_t *>(runs[r].data);
        hr[r].off_base = extra && extra->off_base ? extra->off_base[r] : 0;
        hr[r].data_len = hr[r].off_base + runs[r].data_len;
        hr[r].index = static_cast<const uint4 *>(runs[r].index);
        hr[r].n_in = (uint32_t)(runs[r].index_len / DBEEL_INDEX_ENTRY_SIZE);
        hr[r].base = base;
        hb[r] = hr[r].n_in;
        hm[r] = 0xFFFFFFFFu;
        base += hr[r].n_in;
    }
    if (jobs) {
        GroupDesc *hg = reinterpret_cast<GroupDesc *>(h + o_groups);
        for (uint32_t g = 0; g < extra->n_jobs; g++) {
            const uint32_t r0 = extra->job_first[g], r1 = extra->job_first[g + 1];
            hg[g].first_run = r0;
            hg[g].n_runs = r1 - r0;
            hg[g].pos_end = r1 > r0 ? hr[r1 - 1].base + hr[r1 - 1].n_in : (r0 < n_runs ? hr[r0].base : base);
            hg[g].keep_tombstones = extra->job_keep[g] ? 1 : 0;
            hg[g].bloom = extra->job_bloom[g];
        }
        p.groups = reinterpret_cast<const GroupDesc *>(ws + o_groups);
    }

    // ---- bloom
    uint8_t seed[32];
    if (sh.bloom_file) {
        if (o->bloom_seed) {
            memcpy(seed, o->bloom_seed, 32);
        } else { // Bloom::new -> getrandom(&mut seed)
            FILE *f = fopen("/dev/urandom", "rb");
            if (!f || fread(seed, 1, 32, f) != 32) {
                if (f) fclose(f);
                return fail(e, DBEEL_ERR_INVALID_ARG, "no entropy source for the bloom seed");
            }
            fclose(f);
        }
        p.bloom.words = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(out->bloom) + 8);
        p.bloom.bits = sh.bloom_bits;
        p.bloom.bits_magic = (uint64_t)((((unsigned __int128)1) << 64) / sh.bloom_bits);
        p.bloom.k_num = sh.bloom_k;
        for (int i = 0; i < 4; i++) memcpy(&p.bloom.sip[i], seed + 8 * i, 8);
    }
    if (extra) {
        p.sparse_offsets = extra->sparse_offsets ? 1 : 0;
        p.out_offset_base = extra->out_offset_base;
        if (extra->external_bloom) p.bloom = extra->bloom;
    }

    cudaStream_t s = e->stream;
    uint32_t launches = 0;
    // The header goes down and the control block comes back through kernels that touch the mapped pinned block, not
    // through cudaMemcpyAsync: a small copy on this stream would queue on a copy engine behind whatever bulk transfer
    // of the pipelined host path is in flight there (measured: every partition's kernels waited for the previous
    // partition's 200 MB D2H).  The compute stream carries kernels and event records only.
    if (record_start) CU(cudaEventRecord(e->ev[EV_START], s)); // ms_total covers the header upload and the filter's memset too
    launch_k(e, k_copy_words, (uint32_t)((header_bytes / 4 + 255) / 256), 256, 0, s, reinterpret_cast<uint32_t *>(ws),
             reinterpret_cast<const uint32_t *>(e->pin_dev), (uint32_t)(header_bytes / 4));
    launches++;
    if (sh.bloom_file) CU(cudaMemsetAsync(out->bloom, 0, sh.bloom_file, s));
    if (scan_bytes) CU(cudaMemsetAsync(ws + o_scan, 0, scan_bytes, s));

    // ---- K0/K1: prefix, validate, extract (+ conditional redo when a run was truncated)
    const uint32_t g256 = (N + 255) / 256;
    const uint32_t gext = (N + 256 * kExtractEPT - 1) / (256 * kExtractEPT);
    auto launch_extract = [&](uint32_t grid, int mode) {
        if (ref_reader && hash_early) launch_k(e, k_extract<true, true, true>, grid, 256, 0, s, p, mode);
        else if (ref_reader) launch_k(e, k_extract<true, true, false>, grid, 256, 0, s, p, mode);
        else if (hash_early) launch_k(e, k_extract<true, false, true>, grid, 256, 0, s, p, mode);
        else if (e->narrow_loads && e->extract_persist > 0 && mode == 0) // one resident wave, index records fetched a step ahead
            launch_k(e, k_extract<true, false, false, true>, std::min<uint32_t>(grid, (uint32_t)(e->sm_count * e->extract_persist)), 256, 0, s, p, mode);
        else if (e->narrow_loads) launch_k(e, k_extract<true, false, false>, grid, 256, 0, s, p, mode);
        else launch_k(e, k_extract<false, false, false>, grid, 256, 0, s, p, mode);
    };
    if (flush) {
        launch_k(e, k_flush_prefix_init, 1, 1, 0, s, p);
        launch_k(e, k_flush_prefix, g256, 256, 0, s, p);
        launch_extract(gext, 0);
        launch_k(e, k_plan, 1, 1024, 0, s, p);
        launch_k(e, k_block_sort, p.nseg[0], kMergeThreads, 0, s, p);
    } else {
        launch_k(e, k_common_prefix, 1, 32, 0, s, p, 0);
        launch_extract(gext, 0);
        if (ref_reader) { // all four are no-ops unless an index record disagrees with its .data (lsm_tree.rs:1158-1170)
            launch_k(e, k_ref_repair, n_runs, 1024, 0, s, p);
            launch_k(e, k_ref_reset, 1, 256, 0, s, p);
            launch_k(e, k_common_prefix, 1, 32, 0, s, p, 2);
            launch_extract(gext < 592 ? gext : 592, 2);
            launches += 4;
        }
        launch_k(e, k_common_prefix, 1, 32, 0, s, p, 1); // both no-ops unless a run was truncated
        launch_extract(gext < 592 ? gext : 592, 1);
        launch_k(e, k_plan, 1, 1024, 0, s, p);
    }
    launches += 5;
    if (!flush && (o->flags & DBEEL_FLAG_VERIFY_SORTED)) {
        launch_k(e, k_verify_sorted, g256, 256, 0, s, p);
        launches++;
    }
    const bool stage_ev = e->stage_events != 0;
    if (stage_ev) CU(cudaEventRecord(e->ev[EV_EXTRACT], s));

    // ---- K2/K3: merge levels, ping-pong between rec_a and rec_b
    const Rec *src = p.rec_a;
    Rec *dst = p.rec_b;
    if (sh.bloom_file) { // independent of everything else: its launch overlaps the merges
        launch_k(e, k_bloom_frame, 1, 1, 0, s, static_cast<uint8_t *>(out->bloom), sh.bloom_words, p.bloom);
        launches++;
    }
    for (uint32_t l = 0; l < levels; l++) {
        uint32_t pairs = p.nseg[l + 1];
        const bool last_fused = fused_final && l + 1 == levels;
        const uint64_t tl = last_fused ? kFinNominal : kMergeTile;
        uint64_t t_ub = (uint64_t)(N + tl - 1) / tl + pairs;
        uint64_t b_ub = t_ub + pairs;
        if (last_fused && stage_ev) CU(cudaEventRecord(e->ev[EV_MERGE], s)); // the fused last level is booked under ms_resolve
        launch_k(e, k_merge_partition, (uint32_t)((b_ub + 7) / 8), kPartitionThreads, 0, s, p, l, src); // one warp per boundary
        if (last_fused) { // persistent; merged tile -> resolve -> chained scan -> .index, all from shared memory
            uint64_t grid = (uint64_t)e->sm_count * e->fin_ctas_per_sm;
            if (grid > t_ub) grid = t_ub;
            if (e->narrow_loads) launch_k(e, k_merge_final<true>, (uint32_t)grid, kFinThreads, kFinSmem, s, p, l, src);
            else launch_k(e, k_merge_final<false>, (uint32_t)grid, kFinThreads, kFinSmem, s, p, l, src);
        } else if (e->merge_variant == 0) { // one CTA per tile, plain loads (kept as the A/B baseline of the TMA kernel)
            launch_k(e, k_merge, (uint32_t)t_ub, kMergeThreads, 0, s, p, l, src, dst);
        } else { // persistent, TMA bulk loads / stores + mbarrier
            uint64_t grid = (uint64_t)e->sm_count * kMergeCtasPerSM;
            if (grid > t_ub) grid = t_ub;
            launch_k(e, k_merge_tma, (uint32_t)grid, kMergeThreads, 2 * kMergeBufRecs * sizeof(Rec), s, p, l, src, dst);
        }
        launches += 2;
        if (last_fused) break; // src stays the last level's input: nothing was written to dst
        const Rec *t = src;
        src = dst;
        dst = const_cast<Rec *>(t);
    }
    if (!fused_final && stage_ev) CU(cudaEventRecord(e->ev[EV_MERGE], s));

    // ---- K4: resolve + scan + .index
    if (jobs) {
        launch_k(e, k_bloom_frames, (extra->n_jobs + 127) / 128, 128, 0, s, p.groups, extra->n_jobs);
        launches++;
    }
    uint4 *res = reinterpret_cast<uint4 *>(dst); // the ping-pong buffer that does not hold the merged order
    const bool side_bloom = e->bloom_side && !flush && !jobs && !hash_early && p.bloom.words != nullptr;
    p.bloom_elsewhere = side_bloom ? 1 : 0;
    if (!fused_final) {
        if (hash_early) launch_k(e, k_resolve<true, false, true>, (uint32_t)res_tiles, kResolveThreads, 0, s, p, src, res);
        else if (fused_emit) launch_k(e, k_resolve<true, true, false>, (uint32_t)res_tiles, kResolveThreads, 0, s, p, src, res);
        else if (e->narrow_loads) launch_k(e, k_resolve<true, false, false>, (uint32_t)res_tiles, kResolveThreads, 0, s, p, src, res);
        else launch_k(e, k_resolve<false, false, false>, (uint32_t)res_tiles, kResolveThreads, 0, s, p, src, res);
        launches += 1;
    }
    if (side_bloom) { // fork: the filter is filled on the second stream while this one scans, emits and copies the payload
        CU(cudaEventRecord(e->ev_fork, s));
        CU(cudaStreamWaitEvent(e->s_side, e->ev_fork, 0));
        k_bloom_res<<<g256, 256, 0, e->s_side>>>(p, res);
        CU(cudaEventRecord(e->ev_join, e->s_side));
        launches++;
    }
    if (!fused_emit && !fused_final) {
        launch_k(e, k_scan_tiles, (uint32_t)res_chunks, 1024, 0, s, p);
        launch_k(e, k_scan_chunks, 1, 1024, 0, s, p);
        launch_k(e, k_emit, (uint32_t)res_tiles, kResolveThreads, 0, s, p, res);
        launches += 3;
    }
    if (n_groups) {
        launch_k(e, k_flush_table, (uint32_t)((n_groups + 1 + 127) / 128), 128, 0, s, p, res);
        launches++;
    }
    if (stage_ev) CU(cudaEventRecord(e->ev[EV_RESOLVE], s));

    // ---- K5: gather + bloom (fused epilogue)
    if (gather_tiles) {
        const bool al32 = ((uintptr_t)out->data & 31) == 0; // 256-bit stores
        if (e->gather_variant == 2 && al32) { // persistent, payload staged through shared memory by the bulk-copy engine
            uint64_t grid = (uint64_t)e->sm_count * DBEEL_GT_CTAS;
            if (grid > gather_tiles) grid = gather_tiles;
            launch_k(e, k_gather_tma, (uint32_t)grid, kGtThreads, kGtSmem, s, p);
        } else if (e->gather_variant == 3 && al32) { // persistent, next tile's metadata prefetched with cp.async
            uint64_t grid = (uint64_t)e->sm_count * DBEEL_GP_CTAS;
            if (grid > gather_tiles) grid = gather_tiles;
            launch_k(e, k_gather_p, (uint32_t)grid, kGatherThreads, 0, s, p);
        } else if (e->gather_variant == 4 && al32) { // k_gather32 + a fifth warp per CTA that only fills the filter
            launch_k(e, k_gather32<true, false, false>, (uint32_t)gather_tiles, kGatherThreads + 32, 0, s, p);
        } else if (e->gather_variant == 8 && al32) { // entry-boundary blocks built by the lane that owns them in the copy loop
            launch_k(e, k_gather_fb, (uint32_t)gather_tiles, kFbThreads, 0, s, p);
        } else if (e->gather_variant == 7 && al32) { // payload lands in shared memory (cp.async), boundary blocks + filter while it travels
            launch_k(e, k_gather_async, (uint32_t)gather_tiles, kGatherThreads, 0, s, p);
        } else if (e->gather_variant >= 9 && al32) { // the default: k_gather32 with the lean entry-boundary pass (LDG.E.256, one store per block)
            launch_k(e, k_gather32<false, false, false, true>, (uint32_t)gather_tiles, kGatherThreads, 0, s, p);
        } else if (e->gather_variant == 5 && al32) { // k_gather32, boundary blocks and filter on different warps (no gain)
            launch_k(e, k_gather32<false, true, false>, (uint32_t)gather_tiles, kGatherThreads, 0, s, p);
        } else if (e->gather_variant == 6 && al32 && p.bloom.words != nullptr && p.hash_rec == nullptr && !p.bloom_elsewhere &&
                   gather_tiles + (N + kGatherThreads - 1) / kGatherThreads < 0x7FFFFFFFull) {
            // k_gather32 with the filter on CTAs of their own, interleaved with the copy CTAs of the same grid
            p.bloom_ctas = (uint32_t)((N + kGatherThreads - 1) / kGatherThreads); // one key per thread; N bounds the output entries
            launch_k(e, k_gather32<false, false, true>, (uint32_t)(gather_tiles + p.bloom_ctas), kGatherThreads, 0, s, p);
        } else if (e->gather_variant >= 1 && al32) { // k_gather32, filter as the copy CTA's epilogue
            launch_k(e, k_gather32<false, false, false>, (uint32_t)gather_tiles, kGatherThreads, 0, s, p);
        } else {
            launch_k(e, k_gather, (uint32_t)gather_tiles, kGatherThreads, 0, s, p);
        }
    }
    launches++;
    if (jobs) { // per-job filters: their own pass over the output entries
        launch_k(e, k_bloom_many, g256, 256, 0, s, p);
        launches++;
    }
    if (n_groups) { // only now may the .index offsets become file-relative: the gather kernel reads them as stream offsets
        launch_k(e, k_rebase_index, g256, 256, 0, s, p);
        launches++;
    }
    if (side_bloom) CU(cudaStreamWaitEvent(s, e->ev_join, 0)); // join: the job ends when both streams are done
    CU(cudaEventRecord(e->ev[EV_GATHER], s));
    CU(cudaGetLastError());

    // ---- control block back
    static_assert(sizeof(Ctl) % 4 == 0, "the control block is published word by word");
    Ctl *hc = reinterpret_cast<Ctl *>(e->pin + header_bytes);
    const uint64_t o_hmt = header_bytes + align_up(sizeof(Ctl), 64);
    unsigned long long *hmt = reinterpret_cast<unsigned long long *>(e->pin + o_hmt);
    launch_k(e, k_publish, 1, 256, 0, s, reinterpret_cast<uint32_t *>(e->pin_dev + header_bytes), reinterpret_cast<const uint32_t *>(p.ctl),
             (uint32_t)(sizeof(Ctl) / 4), reinterpret_cast<uint32_t *>(e->pin_dev + o_hmt),
             reinterpret_cast<const uint32_t *>(p.mem_table), n_groups ? (uint32_t)(4 * (n_groups + 1)) : 0u);
    launches++;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s));

    st.kernel_launches = launches;
    st.merge_passes = levels;
    st.key_prefix_len = hc->prefix_len;
    st.entries_valid = hc->total;
    st.runs_truncated = hc->runs_truncated;
    st.index_repaired = (hc->flags & kFlagRepaired) ? 1 : 0;
    if (record_start) cudaEventElapsedTime(&st.ms_total, e->ev[EV_START], e->ev[EV_GATHER]);
    if (stage_ev) {
        if (record_start) cudaEventElapsedTime(&st.ms_extract, e->ev[EV_START], e->ev[EV_EXTRACT]);
        cudaEventElapsedTime(&st.ms_merge, e->ev[EV_EXTRACT], e->ev[EV_MERGE]);
        cudaEventElapsedTime(&st.ms_resolve, e->ev[EV_MERGE], e->ev[EV_RESOLVE]);
        cudaEventElapsedTime(&st.ms_gather, e->ev[EV_RESOLVE], e->ev[EV_GATHER]);
    }
    if (hc->flags & (kFlagUnsorted | kFlagVerifyFailed))
        return fail(e, DBEEL_ERR_UNSORTED_RUN, "an input run is not strictly ascending by key");
    if (hc->out_data_len > sh.data_total) // only possible with a caller-supplied payload bound (sparse batches)
        return fail(e, DBEEL_ERR_CAPACITY, "payload bound of a sparse batch is lower than the bytes it holds");

    out->data_len = hc->out_data_len;
    out->items_written = hc->out_items;
    out->index_len = (uint64_t)hc->out_items * 16;
    out->bloom_len = sh.bloom_file;
    st.entries_out = hc->out_items;
    st.output_bytes = out->data_len + out->index_len + out->bloom_len;
    st.gather_bytes = 2 * out->data_len + out->index_len + 8ull * hc->out_items; // read + write payload, read index + src_ptr
    st.partitions = 1;
    if (jobs) {
        for (uint32_t g = 0; g < extra->n_jobs; g++) {
            dbeel_job_result &row = extra->job_results[g];
            row.data_off = hmt[2 * g];
            row.data_len = hmt[2 * (g + 1)] - hmt[2 * g];
            row.items_written = hmt[2 * (g + 1) + 1] - hmt[2 * g + 1];
            row.index_off = hmt[2 * g + 1] * 16;
            row.index_len = row.items_written * 16;
        }
    }
    if (many) {
        for (uint32_t r = 0; r < n_runs; r++) {
            dbeel_flush_table &row = extra->flush_table[r];
            row.data_off = hmt[2 * r];
            row.data_len = hmt[2 * (r + 1)] - hmt[2 * r];
            row.items = hmt[2 * (r + 1) + 1] - hmt[2 * r + 1];
            row.index_off = hmt[2 * r + 1] * 16;
            row.index_len = row.items * 16;
        }
    }
    return DBEEL_OK;
}

// ------------------------------------------------------------------------------------
// Pipelined host entry point.  A compaction whose inputs live in host memory is PCIe-bound
// (~45 ms in + ~36 ms out vs ~2 ms of kernels for 2.5 GB), so the job is cut into key-range
// partitions: partition i's slices of every run go down on one stream while partition i-1 is
// merged and partition i-2's output goes up on a third -- both PCIe directions stay busy.
// Every key lives in exactly one partition (all runs are cut at the same splitter keys with
// lower_bound), partitions are emitted in key order, .index offsets continue across partitions
// (out_offset_base) and all partitions set bits in one shared bloom filter sized for the whole
// compaction, so the output files are byte-identical to the single-shot path.

constexpr int kFallbackSingleShot = -1000; // internal: inputs need the single-shot path (corrupt / odd)

struct HostRun {
    const uint8_t *data;
    uint64_t data_len;
    const uint8_t *index;
    uint64_t n;
};

struct HostRec {
    uint64_t off;
    uint32_t ks, fs;
};

inline bool host_rec(const HostRun &r, uint64_t i, HostRec *out) {
    const uint8_t *p = r.index + 16 * i;
    memcpy(&out->off, p, 8);
    memcpy(&out->ks, p + 8, 4);
    memcpy(&out->fs, p + 12, 4);
    return out->ks >= 8 && (uint64_t)out->fs >= (uint64_t)out->ks + 24 && out->off <= r.data_len &&
           (uint64_t)out->fs <= r.data_len - out->off;
}

inline int host_key_cmp(const uint8_t *a, uint32_t al, const uint8_t *b, uint32_t bl) {
    const uint32_t m = al < bl ? al : bl;
    const int c = m ? memcmp(a, b, m) : 0;
    if (c) return c;
    return (al > bl) - (al < bl);
}

struct Splitter {
    const uint8_t *key;
    uint32_t klen;
    uint64_t weight;
};

// io != null: the streaming variant (dbeel_compact_stream).  The runs' pointers are ignored: the .index files are pulled
// whole into pinned memory first (16 bytes per entry), the keys the planner looks at come through small reads, and the
// .data slices of partition c travel file -> pinned ring -> device while the outputs travel device -> pinned ring -> file
// on the threads of a StreamPump (host/stream_pump.h).
int run_job_host_pipelined(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *o,
                           dbeel_out *out, const JobShape &sh, const dbeel_stream_io *io = nullptr) {
    // ---- 1. splitters from weighted samples of every run
    std::vector<HostRun> hr(n_runs);
    for (uint32_t r = 0; r < n_runs; r++)
        hr[r] = HostRun{io ? nullptr : static_cast<const uint8_t *>(runs[r].data), runs[r].data_len,
                        io ? nullptr : static_cast<const uint8_t *>(runs[r].index), runs[r].index_len / DBEEL_INDEX_ENTRY_SIZE};
    uint64_t P = (sh.data_total + sh.index_total + e->partition_bytes - 1) / e->partition_bytes;
    if (P > 64) P = 64;
    if (P < 2) return kFallbackSingleShot;
    if (io) { // the .index files, whole, into page-locked memory (they are also what the H2D copies of the index slices read)
        std::vector<uint64_t> ioff(n_runs);
        uint64_t need = 0;
        for (uint32_t r = 0; r < n_runs; r++) {
            ioff[r] = need;
            need += align_up(hr[r].n * 16 + 16, kAlign);
        }
        int rc = ensure_host(e, &e->pin_index, &e->pin_index_cap, need);
        if (rc) return rc;
        std::vector<StreamPump::ReadTask> rt;
        for (uint32_t r = 0; r < n_runs; r++) {
            hr[r].index = e->pin_index + ioff[r];
            for (uint64_t done = 0; done < hr[r].n * 16; done += StreamPump::kPiece)
                rt.push_back(StreamPump::ReadTask{0, r, DBEEL_STREAM_INDEX, done, std::min<uint64_t>(StreamPump::kPiece, hr[r].n * 16 - done),
                                                  e->pin_index + ioff[r] + done});
        }
        rc = parallel_pieces(rt.size(), [&](size_t k) { return io->read(io->ctx, rt[k].run, rt[k].kind, rt[k].off, rt[k].len, rt[k].dst); });
        if (rc) return fail(e, rc, "stream read callback failed (.index)");
    }
    // a key the planner compares: in memory, or fetched through the read callback into `store`
    std::deque<std::vector<uint8_t>> key_store;
    int key_rc = 0;
    auto key_of = [&](uint32_t r, const HostRec &rec, bool keep) -> const uint8_t * {
        if (!io) return hr[r].data + rec.off + 8;
        if (!keep && !key_store.empty()) key_store.pop_back(); // the previous probe's scratch
        key_store.emplace_back(rec.ks - 8 ? rec.ks - 8 : 1);
        if (rec.ks > 8) {
            const int rc = io->read(io->ctx, r, DBEEL_STREAM_DATA, rec.off + 8, rec.ks - 8, key_store.back().data());
            if (rc && !key_rc) key_rc = rc;
        }
        return key_store.back().data();
    };
    constexpr uint64_t kSamples = 256;
    std::vector<Splitter> samples;
    for (uint32_t r = 0; r < n_runs; r++) {
        const uint64_t n = hr[r].n;
        if (!n) continue;
        const uint64_t cnt = n < kSamples ? n : kSamples;
        for (uint64_t q = 0; q < cnt; q++) {
            const uint64_t i = (2 * q + 1) * n / (2 * cnt);
            HostRec rec;
            if (!host_rec(hr[r], i, &rec)) return kFallbackSingleShot;
            samples.push_back(Splitter{key_of(r, rec, true), rec.ks - 8, n / cnt + 1});
        }
    }
    if (key_rc) return fail(e, key_rc, "stream read callback failed (sample keys)");
    if (io) key_store.emplace_back(1); // scratch slot the probes below recycle
    if (samples.empty()) return kFallbackSingleShot;
    std::sort(samples.begin(), samples.end(), [](const Splitter &a, const Splitter &b) {
        return host_key_cmp(a.key, a.klen, b.key, b.klen) < 0;
    });
    uint64_t wsum = 0;
    for (auto &sm : samples) wsum += sm.weight;
    // Partition sizes: the pipeline's fill (nothing to merge until the first partition is down) and drain (nothing but
    // the last partition's D2H) cost one partition's transfer each, so the first and last partitions are small:
    // 1/4, 1/2, 1, 1, ..., 1, 1/2, 1/4 of the nominal size.
    std::vector<double> share;
    if (P >= 4 && e->partition_taper) {
        share = {0.25, 0.5};
        const uint64_t mid = P - 1 > 59 ? 59 : P - 1; // 2P-1 quarter units short of the total: one more full partition
        for (uint64_t k = 0; k < mid; k++) share.push_back(1.0);
        share.push_back(0.5);
        share.push_back(0.25);
    } else {
        share.assign(P, 1.0);
    }
    double share_sum = 0;
    for (double v : share) share_sum += v;
    std::vector<Splitter> cuts;
    {
        uint64_t acc = 0;
        size_t next = 0; // the cut after partition `next`
        double target = share[0] / share_sum;
        for (auto &sm : samples) {
            acc += sm.weight;
            if (next + 1 < share.size() && (double)acc >= target * (double)wsum) {
                if (cuts.empty() || host_key_cmp(cuts.back().key, cuts.back().klen, sm.key, sm.klen) < 0) cuts.push_back(sm);
                while (next + 1 < share.size() && (double)acc >= target * (double)wsum) {
                    next++;
                    target += share[next] / share_sum;
                }
            }
        }
    }
    const uint32_t np = (uint32_t)cuts.size() + 1;
    if (np < 2) return kFallbackSingleShot;

    // ---- 2. cut every run at every splitter (lower_bound: equal keys of all runs land in the same partition)
    std::vector<std::vector<uint64_t>> lo(n_runs, std::vector<uint64_t>(np + 1, 0));
    std::vector<std::vector<uint64_t>> boff(n_runs, std::vector<uint64_t>(np + 1, 0)); // .data offset at each cut
    for (uint32_t r = 0; r < n_runs; r++) {
        const uint64_t n = hr[r].n;
        lo[r][np] = n;
        for (uint32_t c = 0; c < np - 1; c++) {
            uint64_t a = c ? lo[r][c] : 0, b = n;
            while (a < b) {
                const uint64_t mid = (a + b) >> 1;
                HostRec rec;
                if (!host_rec(hr[r], mid, &rec)) return kFallbackSingleShot;
                if (host_key_cmp(key_of(r, rec, false), rec.ks - 8, cuts[c].key, cuts[c].klen) < 0) a = mid + 1; else b = mid;
            }
            lo[r][c + 1] = a;
        }
        uint64_t end = 0;
        if (n) {
            HostRec last;
            if (!host_rec(hr[r], n - 1, &last)) return kFallbackSingleShot;
            end = last.off + last.fs;
        }
        for (uint32_t c = 0; c <= np; c++) {
            const uint64_t i = lo[r][c];
            if (i >= n) { boff[r][c] = end; continue; }
            HostRec rec;
            if (!host_rec(hr[r], i, &rec)) return kFallbackSingleShot;
            if (i) { // the offsets chain must hold across the cut (inside a slice the GPU checks it)
                HostRec prev;
                if (!host_rec(hr[r], i - 1, &prev) || prev.off + prev.fs != rec.off) return kFallbackSingleShot;
            } else if (rec.off != 0) {
                return kFallbackSingleShot;
            }
            boff[r][c] = rec.off;
        }
    }

    if (key_rc) return fail(e, key_rc, "stream read callback failed (splitter probes)");

    // ---- 3. staging: two input and two output buffers sized for the largest partition
    uint64_t max_in = 0, max_out = 0;
    for (uint32_t c = 0; c < np; c++) {
        uint64_t in = 0, d = 0, ix = 0;
        for (uint32_t r = 0; r < n_runs; r++) {
            const uint64_t dl = boff[r][c + 1] - boff[r][c], il = (lo[r][c + 1] - lo[r][c]) * 16;
            in += align_up(dl + 32, kAlign) + align_up(il + 16, kAlign);
            d += dl;
            ix += il;
        }
        const uint64_t o2 = align_up(d + 16, kAlign) + align_up(ix + 16, kAlign);
        max_in = in > max_in ? in : max_in;
        max_out = o2 > max_out ? o2 : max_out;
    }
    int rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, max_in);
    if (!rc) rc = ensure_device(e, &e->stage_in2, &e->stage_in2_cap, max_in);
    if (!rc) rc = ensure_device(e, &e->stage_out, &e->stage_out_cap, max_out);
    if (!rc) rc = ensure_device(e, &e->stage_out2, &e->stage_out2_cap, max_out);
    if (!rc && sh.bloom_file) rc = ensure_device(e, &e->bloom_dev, &e->bloom_dev_cap, sh.bloom_file + 16);
    if (rc) return rc;
    if (!e->s_h2d) {
        CU(cudaStreamCreateWithFlags(&e->s_h2d, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CU(cudaEventCreateWithFlags(&e->ev_h2d[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&e->ev_comp[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&e->ev_d2h[i], cudaEventDisableTiming));
        }
    }
    uint8_t *sin[2] = {e->stage_in, e->stage_in2}, *sout[2] = {e->stage_out, e->stage_out2};
    // streaming: R-slot pinned rings on both sides, one event per partition for the writer threads, the pump itself.
    // Declared in this order so that the pump's threads are joined before the events they wait on are destroyed.
    struct EventList {
        std::vector<cudaEvent_t> ev;
        ~EventList() { for (auto &x : ev) if (x) cudaEventDestroy(x); }
    } ev_out;
    std::unique_ptr<StreamPump> pump;
    const uint32_t R = (uint32_t)std::max(2, e->stream_ring);
    if (io) {
        rc = ensure_host(e, &e->ring_in, &e->ring_in_cap, (uint64_t)R * max_in);
        if (!rc) rc = ensure_host(e, &e->ring_out, &e->ring_out_cap, (uint64_t)R * max_out);
        if (!rc && sh.bloom_file) rc = ensure_host(e, &e->pin_bloom, &e->pin_bloom_cap, sh.bloom_file);
        if (rc) return rc;
        ev_out.ev.assign(np, nullptr);
        for (uint32_t c = 0; c < np; c++) CU(cudaEventCreateWithFlags(&ev_out.ev[c], cudaEventDisableTiming | cudaEventBlockingSync));
        const int dev = e->device;
        EventList *evl = &ev_out;
        pump.reset(new StreamPump(io, np, R, stream_threads(), [evl](uint32_t c) { cudaEventSynchronize(evl->ev[c]); }, [dev]() { cudaSetDevice(dev); }));
        for (uint32_t c = 0; c < np; c++) {
            uint8_t *slot = e->ring_in + (uint64_t)(c % R) * max_in;
            uint64_t pos = 0;
            for (uint32_t r = 0; r < n_runs; r++) {
                const uint64_t dl = boff[r][c + 1] - boff[r][c], il = (lo[r][c + 1] - lo[r][c]) * 16;
                if (dl) pump->add_read(c, r, DBEEL_STREAM_DATA, boff[r][c], dl, slot + pos);
                pos += align_up(dl + 32, kAlign) + align_up(il + 16, kAlign);
            }
        }
        pump->start();
    }

    // ---- 4. the shared bloom filter
    JobExtra ex;
    ex.external_bloom = true;
    if (sh.bloom_file) {
        uint8_t seed[32];
        if (o->bloom_seed) {
            memcpy(seed, o->bloom_seed, 32);
        } else {
            FILE *f = fopen("/dev/urandom", "rb");
            if (!f || fread(seed, 1, 32, f) != 32) {
                if (f) fclose(f);
                return fail(e, DBEEL_ERR_INVALID_ARG, "no entropy source for the bloom seed");
            }
            fclose(f);
        }
        ex.bloom.words = reinterpret_cast<uint32_t *>(e->bloom_dev + 8);
        ex.bloom.bits = sh.bloom_bits;
        ex.bloom.bits_magic = (uint64_t)((((unsigned __int128)1) << 64) / sh.bloom_bits);
        ex.bloom.k_num = sh.bloom_k;
        for (int i = 0; i < 4; i++) memcpy(&ex.bloom.sip[i], seed + 8 * i, 8);
        CU(cudaMemsetAsync(e->bloom_dev, 0, sh.bloom_file, e->stream));
        k_bloom_frame<<<1, 1, 0, e->stream>>>(e->bloom_dev, sh.bloom_words, ex.bloom);
    }

    // ---- 5. the pipeline
    const bool trace = getenv("DBEEL_TRACE") != nullptr; // per-partition timeline on stderr (debug aid)
    std::vector<cudaEvent_t> tev;
    if (trace) {
        tev.resize(6 * (size_t)np);
        for (auto &ev : tev) CU(cudaEventCreate(&ev));
    }
    std::vector<uint64_t> off_base(n_runs);
    std::vector<dbeel_run> dr(n_runs);
    auto enqueue_h2d = [&](uint32_t c) -> int {
        uint8_t *base = sin[c & 1];
        uint64_t pos = 0;
        const uint8_t *slot = io ? e->ring_in + (uint64_t)(c % R) * max_in : nullptr;
        if (io) { // partition c's slices have to be in their ring slot
            const int prc = pump->wait_reads(c);
            if (prc) return fail(e, prc, "stream read callback failed (.data)");
        }
        if (trace) CU(cudaEventRecord(tev[6 * c + 0], e->s_h2d));
        for (uint32_t r = 0; r < n_runs; r++) {
            const uint64_t dl = boff[r][c + 1] - boff[r][c], il = (lo[r][c + 1] - lo[r][c]) * 16;
            if (dl) CU(cudaMemcpyAsync(base + pos, io ? slot + pos : hr[r].data + boff[r][c], dl, cudaMemcpyHostToDevice, e->s_h2d));
            pos += align_up(dl + 32, kAlign);
            if (il) CU(cudaMemcpyAsync(base + pos, hr[r].index + 16 * lo[r][c], il, cudaMemcpyHostToDevice, e->s_h2d));
            pos += align_up(il + 16, kAlign);
        }
        CU(cudaEventRecord(e->ev_h2d[c & 1], e->s_h2d));
        if (trace) CU(cudaEventRecord(tev[6 * c + 1], e->s_h2d));
        return DBEEL_OK;
    };
    dbeel_stats total = {};
    total.input_bytes = sh.data_total + sh.index_total;
    total.entries_in = sh.n_total;
    uint64_t out_data = 0, out_items = 0;
    uint8_t *h_data = static_cast<uint8_t *>(out->data), *h_index = static_cast<uint8_t *>(out->index);
    CU(cudaEventRecord(e->ev[EV_H2D0], e->stream));
    rc = enqueue_h2d(0);
    if (!rc && np > 1) rc = enqueue_h2d(1);
    if (rc) return rc;
    bool truncated = false;
    for (uint32_t c = 0; c < np; c++) {
        uint8_t *base = sin[c & 1];
        uint64_t pos = 0, dsum = 0, isum = 0;
        for (uint32_t r = 0; r < n_runs; r++) {
            const uint64_t dl = boff[r][c + 1] - boff[r][c], il = (lo[r][c + 1] - lo[r][c]) * 16;
            off_base[r] = boff[r][c];
            dr[r].data = base + pos - boff[r][c]; // biased: .data offset `off` lives at data + off
            dr[r].data_len = dl;
            pos += align_up(dl + 32, kAlign);
            dr[r].index = base + pos;
            dr[r].index_len = il;
            pos += align_up(il + 16, kAlign);
            dsum += dl;
            isum += il;
        }
        dbeel_out dout = {};
        dout.data = sout[c & 1];
        dout.data_cap = dsum;
        dout.index = sout[c & 1] + align_up(dsum + 16, kAlign);
        dout.index_cap = isum;
        ex.off_base = off_base.data();
        ex.out_offset_base = out_data;
        CU(cudaStreamWaitEvent(e->stream, e->ev_h2d[c & 1], 0));
        if (c >= 2) CU(cudaStreamWaitEvent(e->stream, e->ev_d2h[c & 1], 0)); // output buffer c&1 drained
        if (trace) CU(cudaEventRecord(tev[6 * c + 2], e->stream));
        rc = run_job_device(e, dr.data(), n_runs, o, false, &dout, /*record_start=*/true, &ex); // syncs e->stream
        if (rc) break;
        if (io) pump->release_input(c); // the kernels have read device buffer c & 1, which the H2D out of ring slot c mod R filled
        const dbeel_stats &ps = e->stats;
        if (ps.runs_truncated || ps.index_repaired) { truncated = true; break; } // the slices were cut by index offsets: redo exactly
        total.entries_valid += ps.entries_valid;
        total.kernel_launches += ps.kernel_launches;
        total.merge_passes = ps.merge_passes > total.merge_passes ? ps.merge_passes : total.merge_passes;
        total.key_prefix_len = ps.key_prefix_len;
        total.ms_total += ps.ms_total;
        total.ms_extract += ps.ms_extract;
        total.ms_merge += ps.ms_merge;
        total.ms_resolve += ps.ms_resolve;
        total.ms_gather += ps.ms_gather;
        total.gather_bytes += ps.gather_bytes;
        CU(cudaEventRecord(e->ev_comp[c & 1], e->stream));
        if (trace) CU(cudaEventRecord(tev[6 * c + 3], e->stream));
        CU(cudaStreamWaitEvent(e->s_d2h, e->ev_comp[c & 1], 0));
        if (trace) CU(cudaEventRecord(tev[6 * c + 4], e->s_d2h));
        if (io) { // device -> ring slot c mod R (once partition c - R has left it) -> the writer threads
            rc = pump->wait_out_slot(c);
            if (rc) { fail(e, rc, "stream write callback failed"); break; }
            uint8_t *oslot = e->ring_out + (uint64_t)(c % R) * max_out;
            uint8_t *oindex = oslot + align_up(dout.data_len + 16, kAlign);
            if (dout.data_len) CU(cudaMemcpyAsync(oslot, dout.data, dout.data_len, cudaMemcpyDeviceToHost, e->s_d2h));
            if (dout.index_len) CU(cudaMemcpyAsync(oindex, dout.index, dout.index_len, cudaMemcpyDeviceToHost, e->s_d2h));
            CU(cudaEventRecord(ev_out.ev[c], e->s_d2h));
            StreamPump::OutPart op;
            op.data = oslot; op.data_len = dout.data_len; op.data_off = out_data;
            op.index = oindex; op.index_len = dout.index_len; op.index_off = 16 * out_items;
            pump->publish_out(c, op);
        } else {
            if (dout.data_len) CU(cudaMemcpyAsync(h_data + out_data, dout.data, dout.data_len, cudaMemcpyDeviceToHost, e->s_d2h));
            if (dout.index_len) CU(cudaMemcpyAsync(h_index + 16 * out_items, dout.index, dout.index_len, cudaMemcpyDeviceToHost, e->s_d2h));
        }
        CU(cudaEventRecord(e->ev_d2h[c & 1], e->s_d2h));
        if (trace) CU(cudaEventRecord(tev[6 * c + 5], e->s_d2h));
        out_data += dout.data_len;
        out_items += dout.items_written;
        if (c + 2 < np) { // input buffer c&1 is free again (the job that read it has completed)
            rc = enqueue_h2d(c + 2);
            if (rc) break;
        }
    }
    if (rc || truncated) { // drain, then report / fall back to the exact single-shot semantics
        cudaStreamSynchronize(e->s_h2d);
        cudaStreamSynchronize(e->s_d2h);
        if (pump) pump->abort(rc ? rc : DBEEL_ERR_INVALID_ARG); // its threads are joined when it goes out of scope
        return rc ? rc : kFallbackSingleShot;
    }
    if (sh.bloom_file) {
        CU(cudaStreamWaitEvent(e->s_d2h, e->ev_comp[(np - 1) & 1], 0));
        CU(cudaMemcpyAsync(io ? (void *)e->pin_bloom : out->bloom, e->bloom_dev, sh.bloom_file, cudaMemcpyDeviceToHost, e->s_d2h));
    }
    CU(cudaStreamSynchronize(e->s_d2h));
    CU(cudaStreamSynchronize(e->s_h2d));
    if (io) {
        if (sh.bloom_file) {
            const int wrc = io->write(io->ctx, DBEEL_STREAM_BLOOM, 0, e->pin_bloom, sh.bloom_file);
            if (wrc) return fail(e, wrc, "stream write callback failed (.bloom)");
        }
        const int frc = pump->finish(); // every partition's bytes have gone through the write callback
        if (frc) return fail(e, frc, "stream write callback failed");
    }
    if (trace) {
        fprintf(stderr, "[dbeel trace] %u partitions; ms since the first H2D began: h2d[begin,end] kernels[begin,end] d2h[begin,end]\n", np);
        for (uint32_t c = 0; c < np; c++) {
            float t[6];
            for (int k = 0; k < 6; k++) cudaEventElapsedTime(&t[k], tev[0], tev[6 * c + k]);
            fprintf(stderr, "[dbeel trace] p%02u h2d %6.2f %6.2f  kernels %6.2f %6.2f  d2h %6.2f %6.2f\n", c, t[0], t[1], t[2], t[3], t[4], t[5]);
        }
        for (auto &ev : tev) cudaEventDestroy(ev);
    }
    out->data_len = out_data;
    out->items_written = out_items;
    out->index_len = out_items * 16;
    out->bloom_len = sh.bloom_file;
    total.entries_out = out_items;
    total.output_bytes = out->data_len + out->index_len + out->bloom_len;
    total.kernel_launches += sh.bloom_file ? 1 : 0;
    total.partitions = np;
    e->stats = total;
    return DBEEL_OK;
}

// host buffers in / out around run_job_device
int run_job_host(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *o, bool flush,
                 dbeel_out *out) {
    JobShape sh;
    shape_of(runs, n_runs, o, flush, &sh);
    if (n_runs > DBEEL_MAX_RUNS) return fail(e, DBEEL_ERR_TOO_MANY_RUNS, "too many runs");
    if (out->data_cap < sh.data_total || out->index_cap < sh.n_total * 16 || out->bloom_cap < sh.bloom_file)
        return fail(e, DBEEL_ERR_CAPACITY, "output buffer smaller than dbeel_compact_bound");
    for (uint32_t r = 0; r < n_runs; r++)
        if ((runs[r].data_len && !runs[r].data) || (runs[r].index_len && !runs[r].index))
            return fail(e, DBEEL_ERR_INVALID_ARG, "null run buffer");
    if (e->pipeline && !flush && !(o->flags & DBEEL_FLAG_VERIFY_SORTED) && sh.n_total < 0xFFFFFFFEull &&
        sh.data_total + sh.index_total >= e->pipeline_min_bytes) {
        int prc = run_job_host_pipelined(e, runs, n_runs, o, out, sh);
        if (prc != kFallbackSingleShot) return prc;
        out->data_len = out->index_len = out->bloom_len = out->items_written = 0;
    }

    // device staging: every buffer 256-aligned with 16 bytes of slack behind it
    uint64_t in_need = 0;
    for (uint32_t r = 0; r < n_runs; r++)
        in_need += align_up(runs[r].data_len + 16, kAlign) + align_up(runs[r].index_len + 16, kAlign);
    uint64_t out_need = align_up(sh.data_total + 16, kAlign) + align_up(sh.n_total * 16 + 16, kAlign) +
                        align_up(sh.bloom_file + 16, kAlign);
    int rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, in_need);
    if (rc) return rc;
    rc = ensure_device(e, &e->stage_out, &e->stage_out_cap, out_need);
    if (rc) return rc;

    cudaStream_t s = e->stream;
    std::vector<dbeel_run> dr(n_runs);
    CU(cudaEventRecord(e->ev[EV_H2D0], s));
    uint64_t off = 0;
    for (uint32_t r = 0; r < n_runs; r++) {
        dr[r].data = e->stage_in + off;
        dr[r].data_len = runs[r].data_len;
        if (runs[r].data_len)
            CU(cudaMemcpyAsync(e->stage_in + off, runs[r].data, runs[r].data_len, cudaMemcpyHostToDevice, s));
        off += align_up(runs[r].data_len + 16, kAlign);
        dr[r].index = e->stage_in + off;
        dr[r].index_len = runs[r].index_len;
        if (runs[r].index_len)
            CU(cudaMemcpyAsync(e->stage_in + off, runs[r].index, runs[r].index_len, cudaMemcpyHostToDevice, s));
        off += align_up(runs[r].index_len + 16, kAlign);
    }
    CU(cudaEventRecord(e->ev[EV_H2D1], s));
    CU(cudaEventRecord(e->ev[EV_START], s));

    dbeel_out dout = *out;
    dout.data = e->stage_out;
    dout.index = e->stage_out + align_up(sh.data_total + 16, kAlign);
    dout.bloom = sh.bloom_file ? static_cast<uint8_t *>(dout.index) + align_up(sh.n_total * 16 + 16, kAlign) : nullptr;
    rc = run_job_device(e, dr.data(), n_runs, o, flush, &dout, /*record_start=*/false);
    // run_job_device zeroes stats; its START event is ours
    if (rc) return rc;
    dbeel_stats &st = e->stats;
    if (sh.n_total) {
        cudaEventElapsedTime(&st.ms_h2d, e->ev[EV_H2D0], e->ev[EV_H2D1]);
        cudaEventElapsedTime(&st.ms_total, e->ev[EV_START], e->ev[EV_GATHER]);
        cudaEventElapsedTime(&st.ms_extract, e->ev[EV_START], e->ev[EV_EXTRACT]);
    }
    CU(cudaEventRecord(e->ev[EV_D2H0], s));
    if (dout.data_len) CU(cudaMemcpyAsync(out->data, dout.data, dout.data_len, cudaMemcpyDeviceToHost, s));
    if (dout.index_len) CU(cudaMemcpyAsync(out->index, dout.index, dout.index_len, cudaMemcpyDeviceToHost, s));
    if (dout.bloom_len) CU(cudaMemcpyAsync(out->bloom, dout.bloom, dout.bloom_len, cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(e->ev[EV_D2H1], s));
    CU(cudaStreamSynchronize(s));
    cudaEventElapsedTime(&st.ms_d2h, e->ev[EV_D2H0], e->ev[EV_D2H1]);
    out->data_len = dout.data_len;
    out->index_len = dout.index_len;
    out->bloom_len = dout.bloom_len;
    out->items_written = dout.items_written;
    return DBEEL_OK;
}

struct BusyGuard {
    dbeel_engine *e;
    explicit BusyGuard(dbeel_engine *e_) : e(e_) { e->busy = true; }
    ~BusyGuard() { e->busy = false; }
};

// ------------------------------------------------------------------------------------ N3: the storage edge
// dbeel_compact_stream for a job the pipeline does not take (too small to partition, an index the planner does not trust,
// a run that ended early): every file whole into page-locked memory, the single-shot host path, the outputs whole through
// the write callback -- the exact semantics of dbeel_compact, the callbacks just replace the caller's buffers.
struct HostBlock {
    uint8_t *p = nullptr;
    ~HostBlock() { if (p) cudaFreeHost(p); }
    bool alloc(uint64_t n) {
        if (cudaHostAlloc(reinterpret_cast<void **>(&p), n ? n : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); p = nullptr; }
        return p != nullptr;
    }
};

int run_job_stream_whole(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *o, const dbeel_stream_io *io,
                         dbeel_out *out, const JobShape &sh) {
    std::vector<uint64_t> doff(n_runs), ioff(n_runs);
    uint64_t pos = 0;
    for (uint32_t r = 0; r < n_runs; r++) {
        doff[r] = pos;
        pos += align_up(runs[r].data_len + 16, kAlign);
        ioff[r] = pos;
        pos += align_up(runs[r].index_len + 16, kAlign);
    }
    HostBlock in, ob;
    if (!in.alloc(pos)) return fail(e, DBEEL_ERR_NOMEM, "cudaHostAlloc(stream inputs)");
    std::vector<StreamPump::ReadTask> rt;
    std::vector<dbeel_run> hr(n_runs);
    for (uint32_t r = 0; r < n_runs; r++) {
        hr[r] = dbeel_run{in.p + doff[r], runs[r].data_len, in.p + ioff[r], runs[r].index_len};
        for (uint64_t d = 0; d < runs[r].data_len; d += StreamPump::kPiece)
            rt.push_back(StreamPump::ReadTask{0, r, DBEEL_STREAM_DATA, d, std::min<uint64_t>(StreamPump::kPiece, runs[r].data_len - d), in.p + doff[r] + d});
        for (uint64_t d = 0; d < runs[r].index_len; d += StreamPump::kPiece)
            rt.push_back(StreamPump::ReadTask{0, r, DBEEL_STREAM_INDEX, d, std::min<uint64_t>(StreamPump::kPiece, runs[r].index_len - d), in.p + ioff[r] + d});
    }
    int rc = parallel_pieces(rt.size(), [&](size_t k) { return io->read(io->ctx, rt[k].run, rt[k].kind, rt[k].off, rt[k].len, rt[k].dst); });
    if (rc) return fail(e, rc, "stream read callback failed");
    const uint64_t dc = sh.data_total, ic = sh.n_total * 16, bc = sh.bloom_file;
    const uint64_t o_index = align_up(dc + 16, kAlign), o_bloom = o_index + align_up(ic + 16, kAlign);
    if (!ob.alloc(o_bloom + align_up(bc + 16, kAlign))) return fail(e, DBEEL_ERR_NOMEM, "cudaHostAlloc(stream outputs)");
    dbeel_out o2 = {ob.p, dc, 0, ob.p + o_index, ic, 0, bc ? ob.p + o_bloom : nullptr, bc, 0, 0};
    const int saved = e->pipeline;
    e->pipeline = 0;
    rc = run_job_host(e, hr.data(), n_runs, o, false, &o2);
    e->pipeline = saved;
    if (rc) return rc;
    struct WTask { uint32_t kind; uint64_t off, len; const uint8_t *src; };
    std::vector<WTask> wt;
    for (uint64_t d = 0; d < o2.data_len; d += StreamPump::kPiece)
        wt.push_back(WTask{DBEEL_STREAM_DATA, d, std::min<uint64_t>(StreamPump::kPiece, o2.data_len - d), ob.p + d});
    for (uint64_t d = 0; d < o2.index_len; d += StreamPump::kPiece)
        wt.push_back(WTask{DBEEL_STREAM_INDEX, d, std::min<uint64_t>(StreamPump::kPiece, o2.index_len - d), ob.p + o_index + d});
    if (o2.bloom_len) wt.push_back(WTask{DBEEL_STREAM_BLOOM, 0, o2.bloom_len, ob.p + o_bloom});
    rc = parallel_pieces(wt.size(), [&](size_t k) { return io->write(io->ctx, wt[k].kind, wt[k].off, wt[k].src, wt[k].len); });
    if (rc) return fail(e, rc, "stream write callback failed");
    out->data_len = o2.data_len;
    out->index_len = o2.index_len;
    out->bloom_len = o2.bloom_len;
    out->items_written = o2.items_written;
    return DBEEL_OK;
}

int stream_entry(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts, const dbeel_stream_io *io,
                 dbeel_out *out) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!out || !io || !io->read || !io->write || (n_runs && !runs)) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (e->async_state.load(std::memory_order_acquire) != 0) return DBEEL_ERR_BUSY;
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    dbeel_compact_opts o;
    default_opts(&o);
    if (opts) o = *opts;
    if (!(o.bloom_fp > 0.0 && o.bloom_fp < 1.0)) return fail(e, DBEEL_ERR_INVALID_ARG, "bloom_fp must be in (0,1)");
    if (n_runs > DBEEL_MAX_RUNS) return fail(e, DBEEL_ERR_TOO_MANY_RUNS, "too many runs");
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    e->stats.ms_h2d = 0;
    out->data_len = out->index_len = out->bloom_len = out->items_written = 0;
    JobShape sh;
    shape_of(runs, n_runs, &o, false, &sh);
    if (e->pipeline && !(o.flags & DBEEL_FLAG_VERIFY_SORTED) && sh.n_total < 0xFFFFFFFEull &&
        sh.data_total + sh.index_total >= e->pipeline_min_bytes) {
        const int prc = run_job_host_pipelined(e, runs, n_runs, &o, out, sh, io);
        if (prc != kFallbackSingleShot) return prc;
        out->data_len = out->index_len = out->bloom_len = out->items_written = 0;
    }
    return run_job_stream_whole(e, runs, n_runs, &o, io, out, sh);
}

int entry(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts, dbeel_out *out,
          bool flush, bool device) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!out || (n_runs && !runs)) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    dbeel_compact_opts o;
    default_opts(&o);
    if (opts) o = *opts;
    if (!(o.bloom_fp > 0.0 && o.bloom_fp < 1.0)) return fail(e, DBEEL_ERR_INVALID_ARG, "bloom_fp must be in (0,1)");
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    e->stats.ms_h2d = 0;
    return device ? run_job_device(e, runs, n_runs, &o, flush, out, true) : run_job_host(e, runs, n_runs, &o, flush, out);
}


// ------------------------------------------------------------------------------------ N2: batched point lookups

constexpr uint64_t kBloomTrailer = 8 + 8 + 4 + 144; // nbits, bitmap_bits, k_num, 2 x SipHasher13 (9 x u64 each)

inline uint64_t rd64(const uint8_t *p) { uint64_t v; memcpy(&v, p, 8); return v; }
inline uint32_t rd32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }

// head = the file's first 8 bytes, tail = its last kBloomTrailer bytes (both in host memory)
int parse_bloom(dbeel_engine *e, const uint8_t *head, const uint8_t *tail, uint64_t file_len, TableDesc *t) {
    const uint64_t n_words = rd64(head);
    if (n_words > (1ull << 40) || file_len != 8 + 4 * n_words + kBloomTrailer) return fail(e, DBEEL_ERR_BAD_BLOOM, "bloom file length does not match its word count");
    t->bits = rd64(tail + 8); // Bloom.bitmap_bits (the BitVec's own nbits precedes it)
    t->k_num = rd32(tail + 16);
    if (t->bits < 2 || t->bits > 32 * n_words || t->k_num == 0) return fail(e, DBEEL_ERR_BAD_BLOOM, "bloom parameters out of range");
    t->bits_magic = (uint64_t)((((unsigned __int128)1) << 64) / t->bits);
    for (int h = 0; h < 2; h++) { // SipHasher13 { k0, k1, length, state { v0, v2, v1, v3 }, tail, ntail }
        t->sip[2 * h] = rd64(tail + 20 + 72 * h);
        t->sip[2 * h + 1] = rd64(tail + 20 + 72 * h + 8);
    }
    return DBEEL_OK;
}

int lookup_entry(dbeel_engine *e, const dbeel_table *tables, uint32_t n_tables, const void *keys, const uint64_t *key_off,
                 uint64_t n_keys, uint32_t mode, dbeel_lookup_result *results, bool device) {
    static_assert(sizeof(dbeel_lookup_result) == 16, "result rows are written as uint4");
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if ((n_tables && !tables) || (n_keys && (!key_off || !results))) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (mode > DBEEL_LOOKUP_EXACT) return fail(e, DBEEL_ERR_INVALID_ARG, "unknown lookup mode");
    if (n_tables > 65536) return fail(e, DBEEL_ERR_TOO_MANY_RUNS, "more than 65536 tables");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    e->stats = dbeel_stats{};
    if (n_keys == 0) return DBEEL_OK;
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    cudaStream_t s = e->stream;
    for (uint32_t i = 0; i < n_tables; i++) {
        const dbeel_table &t = tables[i];
        if (t.index_len % DBEEL_INDEX_ENTRY_SIZE) return fail(e, DBEEL_ERR_INVALID_ARG, "index length is not a multiple of 16");
        if ((t.data_len && !t.data) || (t.index_len && !t.index) || (t.bloom_len && !t.bloom)) return fail(e, DBEEL_ERR_INVALID_ARG, "null table buffer");
        if (t.bloom_len && (t.bloom_len < 8 + kBloomTrailer || (t.bloom_len - 8 - kBloomTrailer) % 4))
            return fail(e, DBEEL_ERR_BAD_BLOOM, "bloom file length is not 8 + 4 * words + 164");
        if (device && (((uintptr_t)t.index & 15) || ((uintptr_t)t.bloom & 3))) return fail(e, DBEEL_ERR_INVALID_ARG, "misaligned device buffer");
    }
    std::vector<TableDesc> td(n_tables);
    const uint8_t *d_keys = static_cast<const uint8_t *>(keys);
    const uint64_t *d_off = key_off;
    uint4 *d_res = reinterpret_cast<uint4 *>(results);
    int rc = ensure_pinned(e, std::max<uint64_t>(4096, (uint64_t)n_tables * (8 + kBloomTrailer) + n_tables * sizeof(TableDesc)));
    if (rc) return rc;
    uint8_t *pin_desc = e->pin + (uint64_t)n_tables * (8 + kBloomTrailer);
    if (device) {
        for (uint32_t i = 0; i < n_tables; i++) {
            const dbeel_table &t = tables[i];
            td[i] = TableDesc{static_cast<const uint8_t *>(t.data), t.data_len, static_cast<const uint4 *>(t.index),
                              t.index_len / DBEEL_INDEX_ENTRY_SIZE, nullptr, 0, 0, 0, 0, {0, 0, 0, 0}};
            if (!t.bloom_len) continue;
            const uint8_t *b = static_cast<const uint8_t *>(t.bloom);
            uint8_t *hp = e->pin + (uint64_t)i * (8 + kBloomTrailer);
            CU(cudaMemcpyAsync(hp, b, 8, cudaMemcpyDeviceToHost, s));
            CU(cudaMemcpyAsync(hp + 8, b + t.bloom_len - kBloomTrailer, kBloomTrailer, cudaMemcpyDeviceToHost, s));
            td[i].words = reinterpret_cast<const uint32_t *>(b + 8);
        }
        CU(cudaStreamSynchronize(s));
        for (uint32_t i = 0; i < n_tables; i++)
            if (tables[i].bloom_len) {
                const uint8_t *hp = e->pin + (uint64_t)i * (8 + kBloomTrailer);
                if ((rc = parse_bloom(e, hp, hp + 8, tables[i].bloom_len, &td[i]))) return rc;
            }
    } else { // host buffers: the tables, the keys and the offsets go down, the result rows come back
        if (!keys && key_off[n_keys]) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
        const uint64_t key_bytes = key_off[n_keys];
        uint64_t need = align_up(key_bytes + 16, kAlign) + align_up((n_keys + 1) * 8, kAlign);
        for (uint32_t i = 0; i < n_tables; i++)
            need += align_up(tables[i].data_len + 16, kAlign) + align_up(tables[i].index_len + 16, kAlign) + align_up(tables[i].bloom_len + 16, kAlign);
        rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, need);
        if (!rc) rc = ensure_device(e, &e->stage_out, &e->stage_out_cap, n_keys * 16);
        if (rc) return rc;
        uint64_t pos = 0;
        auto put = [&](const void *src, uint64_t len, uint64_t slack) -> const uint8_t * {
            uint8_t *dst = e->stage_in + pos;
            pos += align_up(len + slack, kAlign);
            if (len && cudaMemcpyAsync(dst, src, len, cudaMemcpyHostToDevice, s) != cudaSuccess) return nullptr;
            return dst;
        };
        d_keys = put(keys, key_bytes, 16);
        d_off = reinterpret_cast<const uint64_t *>(put(key_off, (n_keys + 1) * 8, 0));
        if (!d_keys || !d_off) return fail(e, DBEEL_ERR_CUDA, "cudaMemcpyAsync(keys)", cudaGetLastError());
        for (uint32_t i = 0; i < n_tables; i++) {
            const dbeel_table &t = tables[i];
            const uint8_t *dd = put(t.data, t.data_len, 16), *di = put(t.index, t.index_len, 16), *db = put(t.bloom, t.bloom_len, 16);
            if (!dd || !di || !db) return fail(e, DBEEL_ERR_CUDA, "cudaMemcpyAsync(table)", cudaGetLastError());
            td[i] = TableDesc{dd, t.data_len, reinterpret_cast<const uint4 *>(di), t.index_len / DBEEL_INDEX_ENTRY_SIZE, nullptr, 0, 0, 0, 0, {0, 0, 0, 0}};
            if (!t.bloom_len) continue;
            const uint8_t *b = static_cast<const uint8_t *>(t.bloom);
            if ((rc = parse_bloom(e, b, b + t.bloom_len - kBloomTrailer, t.bloom_len, &td[i]))) return rc;
            td[i].words = reinterpret_cast<const uint32_t *>(db + 8);
        }
        d_res = reinterpret_cast<uint4 *>(e->stage_out);
    }
    rc = ensure_device(e, &e->ws, &e->ws_cap, std::max<uint64_t>(4096, n_tables * sizeof(TableDesc)));
    if (rc) return rc;
    if (n_tables) {
        memcpy(pin_desc, td.data(), n_tables * sizeof(TableDesc));
        CU(cudaMemcpyAsync(e->ws, pin_desc, n_tables * sizeof(TableDesc), cudaMemcpyHostToDevice, s));
    }
    LookupParams lp{reinterpret_cast<const TableDesc *>(e->ws), n_tables, mode, d_keys, d_off, n_keys, d_res};
    CU(cudaEventRecord(e->ev[EV_START], s));
    k_lookup<<<(uint32_t)((n_keys + 255) / 256), 256, 0, s>>>(lp);
    CU(cudaGetLastError());
    CU(cudaEventRecord(e->ev[EV_GATHER], s));
    if (!device) CU(cudaMemcpyAsync(results, d_res, n_keys * 16, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    CU(cudaEventElapsedTime(&e->stats.ms_total, e->ev[EV_START], e->ev[EV_GATHER]));
    e->stats.kernel_launches = 1;
    e->stats.entries_in = n_keys;
    return DBEEL_OK;
}


// ------------------------------------------------------------------------------------ cfg5: shard routing

// batch / out_index / shard_of are device pointers; ring, counts, bytes live in host memory.
int route_entry(dbeel_engine *e, const dbeel_run *batch, const uint32_t *ring, uint32_t n_shards, void *out_index, uint64_t out_index_cap,
                uint32_t *shard_of, void *out_hash64, uint64_t *counts, uint64_t *bytes) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!batch || !ring || !counts || n_shards == 0) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (n_shards > kRouteMaxShards) return fail(e, DBEEL_ERR_INVALID_ARG, "more shards than DBEEL_MAX_SHARDS");
    for (uint32_t s = 1; s < n_shards; s++)
        if (ring[s - 1] >= ring[s]) return fail(e, DBEEL_ERR_INVALID_ARG, "ring hashes must be strictly ascending");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    const uint64_t n64 = batch->index_len / DBEEL_INDEX_ENTRY_SIZE;
    for (uint32_t s = 0; s < n_shards; s++) { counts[s] = 0; if (bytes) bytes[s] = 0; }
    if (n64 >= 0xFFFFFFF0ull) return fail(e, DBEEL_ERR_TOO_MANY_ENTRIES, "too many arrivals in one batch");
    if (n64 == 0) return DBEEL_OK;
    if (out_index_cap < n64 * 16 || !out_index) return fail(e, DBEEL_ERR_CAPACITY, "routed index buffer too small");
    if (((uintptr_t)batch->index | (uintptr_t)out_index) & 15) return fail(e, DBEEL_ERR_INVALID_ARG, "index buffers must be 16-byte aligned");
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    RouteParams p;
    p.data = static_cast<const uint8_t *>(batch->data);
    p.data_len = batch->data_len;
    p.index = static_cast<const uint4 *>(batch->index);
    p.n = (uint32_t)n64;
    p.n_shards = n_shards;
    p.n_blocks = (p.n + kRouteThreads - 1) / kRouteThreads;
    uint64_t off = 0;
    auto carve = [&](uint64_t b) { uint64_t o2 = off; off = align_up(off + b, kAlign); return o2; };
    const uint64_t o_ring = carve(4ull * n_shards), o_tot = carve(8ull * (3 * n_shards + 1));
    const uint64_t o_hist = carve(4ull * p.n_blocks * n_shards), o_owner = carve(shard_of ? 0 : 4ull * p.n);
    const uint64_t o_h64 = carve(out_hash64 ? 8ull * p.n : 0);
    int rc = ensure_device(e, &e->route_ws, &e->route_ws_cap, off);
    if (!rc) rc = ensure_pinned(e, 4096 + 8ull * (3 * n_shards + 1));
    if (rc) return rc;
    cudaStream_t s = e->stream;
    // the ring goes down through the mapped pinned block like every small header (no copy-engine traffic on this stream)
    memcpy(e->pin, ring, 4ull * n_shards);
    p.ring = reinterpret_cast<const uint32_t *>(e->route_ws + o_ring);
    p.totals = reinterpret_cast<unsigned long long *>(e->route_ws + o_tot);
    p.hist = reinterpret_cast<uint32_t *>(e->route_ws + o_hist);
    p.shard_of = shard_of ? shard_of : reinterpret_cast<uint32_t *>(e->route_ws + o_owner);
    p.out_index = static_cast<uint4 *>(out_index);
    p.hash64 = out_hash64 ? reinterpret_cast<unsigned long long *>(e->route_ws + o_h64) : nullptr;
    p.out_hash64 = static_cast<unsigned long long *>(out_hash64);
    p.stop = nullptr;
    CU(cudaEventRecord(e->ev[EV_START], s));
    k_copy_words<<<(n_shards + 255) / 256, 256, 0, s>>>(reinterpret_cast<uint32_t *>(e->route_ws + o_ring), reinterpret_cast<const uint32_t *>(e->pin_dev), n_shards);
    CU(cudaMemsetAsync(p.totals, 0, 8ull * 3 * n_shards, s));
    CU(cudaMemsetAsync(p.totals + 3 * n_shards, 0xFF, 8, s));
    k_route_hash<false><<<p.n_blocks, kRouteThreads, 0, s>>>(p);
    k_route_scan<<<n_shards, 1024, 0, s>>>(p);
    unsigned long long *host_tot = reinterpret_cast<unsigned long long *>(e->pin + 4096);
    k_route_starts<<<1, 256, 0, s>>>(p, reinterpret_cast<unsigned long long *>(e->pin_dev + 4096));
    k_route_scatter<<<p.n_blocks, kRouteThreads, 0, s>>>(p);
    CU(cudaEventRecord(e->ev[EV_GATHER], s));
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s));
    dbeel_stats &st = e->stats;
    memset(&st, 0, sizeof st);
    st.entries_in = n64;
    st.kernel_launches = 5;
    cudaEventElapsedTime(&st.ms_total, e->ev[EV_START], e->ev[EV_GATHER]);
    if (host_tot[3 * n_shards] != ~0ull) return fail(e, DBEEL_ERR_INVALID_ARG, "an arrival's index record does not frame an entry inside .data");
    for (uint32_t k = 0; k < n_shards; k++) {
        counts[k] = host_tot[k];
        if (bytes) bytes[k] = host_tot[n_shards + k];
    }
    st.entries_out = n64;
    st.input_bytes = n64 * 16;
    return DBEEL_OK;
}

// key_hash64: device; stream_starts / cuts / cut_starts: host
int cuts_entry(dbeel_engine *e, const void *key_hash64, const uint64_t *stream_starts, uint32_t n_streams, uint32_t capacity,
               uint32_t *cuts, uint32_t *cut_starts, uint32_t max_cuts_total) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!stream_starts || !cuts || !cut_starts || !n_streams) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (capacity < 1 || capacity > kCutMaxCapacity) return fail(e, DBEEL_ERR_INVALID_ARG, "capacity above what the device cut supports (use dbeel_memtable_cut)");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    // a stream of n arrivals has at most n / capacity full memtables
    std::vector<uint32_t> base(n_streams + 1, 0);
    for (uint32_t s = 0; s < n_streams; s++) {
        if (stream_starts[s + 1] < stream_starts[s] || stream_starts[s + 1] - stream_starts[s] >= 0xFFFFFFF0ull)
            return fail(e, DBEEL_ERR_INVALID_ARG, "stream_starts must ascend");
        base[s + 1] = base[s] + (uint32_t)((stream_starts[s + 1] - stream_starts[s]) / capacity);
    }
    const uint32_t total_max = base[n_streams];
    for (uint32_t s = 0; s <= n_streams; s++) cut_starts[s] = 0;
    if (stream_starts[n_streams] == stream_starts[0]) return DBEEL_OK;
    if (!key_hash64) return fail(e, DBEEL_ERR_INVALID_ARG, "null key identities");
    uint64_t off = 0;
    auto carve = [&](uint64_t b) { uint64_t o2 = off; off = align_up(off + b, kAlign); return o2; };
    const uint64_t o_starts = carve(8ull * (n_streams + 1)), o_base = carve(4ull * n_streams), o_n = carve(4ull * n_streams);
    const uint64_t o_cuts = carve(4ull * (total_max + 1));
    const uint64_t hdr = o_n; // starts | base go down, n_cuts | cuts come back
    int rc = ensure_device(e, &e->route_ws, &e->route_ws_cap, off);
    if (!rc) rc = ensure_pinned(e, off);
    if (rc) return rc;
    memcpy(e->pin + o_starts, stream_starts, 8ull * (n_streams + 1));
    memcpy(e->pin + o_base, base.data(), 4ull * n_streams);
    cudaStream_t s = e->stream;
    static bool attr_set = false;
    if (!attr_set) {
        CU(cudaFuncSetAttribute(k_memtable_cuts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(12ull * kCutSlots)));
        attr_set = true;
    }
    CU(cudaEventRecord(e->ev[EV_START], s));
    k_copy_words<<<(uint32_t)((hdr / 4 + 255) / 256), 256, 0, s>>>(reinterpret_cast<uint32_t *>(e->route_ws), reinterpret_cast<const uint32_t *>(e->pin_dev),
                                                                    (uint32_t)(hdr / 4));
    CutParams p;
    p.hash64 = static_cast<const unsigned long long *>(key_hash64);
    p.starts = reinterpret_cast<const unsigned long long *>(e->route_ws + o_starts);
    p.n_streams = n_streams;
    p.capacity = capacity;
    p.max_cuts = total_max;
    p.cut_base = reinterpret_cast<const uint32_t *>(e->route_ws + o_base);
    p.cuts = reinterpret_cast<uint32_t *>(e->route_ws + o_cuts);
    p.n_cuts = reinterpret_cast<uint32_t *>(e->route_ws + o_n);
    k_memtable_cuts<<<n_streams, 1024, 12ull * kCutSlots, s>>>(p);
    k_publish<<<1, 256, 0, s>>>(reinterpret_cast<uint32_t *>(e->pin_dev + o_n), p.n_cuts, n_streams, reinterpret_cast<uint32_t *>(e->pin_dev + o_cuts),
                                p.cuts, total_max);
    CU(cudaEventRecord(e->ev[EV_GATHER], s));
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s));
    dbeel_stats &st = e->stats;
    memset(&st, 0, sizeof st);
    st.kernel_launches = 3;
    st.entries_in = stream_starts[n_streams] - stream_starts[0];
    cudaEventElapsedTime(&st.ms_total, e->ev[EV_START], e->ev[EV_GATHER]);
    const uint32_t *hn = reinterpret_cast<const uint32_t *>(e->pin + o_n), *hc = reinterpret_cast<const uint32_t *>(e->pin + o_cuts);
    uint32_t w = 0;
    for (uint32_t k = 0; k < n_streams; k++) {
        cut_starts[k] = w;
        const uint32_t nc = hn[k] < base[k + 1] - base[k] ? hn[k] : base[k + 1] - base[k];
        if (w + nc > max_cuts_total) return fail(e, DBEEL_ERR_CAPACITY, "cuts array too small");
        for (uint32_t c = 0; c < nc; c++) cuts[w++] = hc[base[k] + c];
    }
    cut_starts[n_streams] = w;
    return DBEEL_OK;
}

// ------------------------------------------------------------------------------------ N4: WAL replay + flush

int wal_flush_entry(dbeel_engine *e, const void *wal, uint64_t wal_len, uint32_t capacity, dbeel_out *out, bool device) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!out || (wal_len && !wal)) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    e->err.clear();
    out->data_len = out->index_len = out->bloom_len = out->items_written = 0;
    const uint64_t n_pages64 = (wal_len + kWalPage - 1) / kWalPage;
    if (n_pages64 >= 0xFFFFFFF0ull) return fail(e, DBEEL_ERR_TOO_MANY_ENTRIES, "write-ahead log too large");
    if (wal_len == 0) { e->stats = dbeel_stats{}; return DBEEL_OK; }
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    cudaStream_t s = e->stream;
    const uint32_t n_pages = (uint32_t)n_pages64, nodes = n_pages + 1;
    uint32_t levels = 0;
    while ((1ull << levels) < nodes) levels++;

    const uint8_t *d_wal = static_cast<const uint8_t *>(wal);
    uint64_t data_cap_user = out->data_cap, index_cap_user = out->index_cap;
    void *user_data = out->data, *user_index = out->index;
    float ms_h2d = 0;
    const uint4 *d_index = nullptr;
    {
        BusyGuard g(e);
        if (!device) { // host log: stage it down (the flush below writes into staging too)
            int rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, align_up(wal_len + 32, kAlign));
            if (rc) return rc;
            CU(cudaEventRecord(e->ev[EV_H2D0], s));
            CU(cudaMemcpyAsync(e->stage_in, wal, wal_len, cudaMemcpyHostToDevice, s));
            CU(cudaEventRecord(e->ev[EV_H2D1], s));
            d_wal = e->stage_in;
        } else if ((uintptr_t)wal & 15) {
            return fail(e, DBEEL_ERR_INVALID_ARG, "device log buffer must be 16-byte aligned");
        }
        // scratch: jump / cnt tables, per-page sizes, the arrival index, 3 totals
        uint64_t off = 0;
        auto carve = [&](uint64_t bytes) { uint64_t o2 = off; off = align_up(off + bytes, kAlign); return o2; };
        const uint64_t o_jump = carve(4ull * (levels + 1) * nodes), o_cnt = carve(4ull * (levels + 1) * nodes);
        const uint64_t o_sizes = carve(8ull * n_pages), o_index = carve(16ull * n_pages), o_tot = carve(32);
        int rc = ensure_device(e, &e->wal_ws, &e->wal_ws_cap, off);
        if (!rc) rc = ensure_pinned(e, 4096);
        if (rc) return rc;
        WalParams w;
        w.wal = d_wal;
        w.len = wal_len;
        w.n_pages = n_pages;
        w.levels = levels;
        w.jump = reinterpret_cast<uint32_t *>(e->wal_ws + o_jump);
        w.cnt = reinterpret_cast<uint32_t *>(e->wal_ws + o_cnt);
        w.sizes = reinterpret_cast<uint2 *>(e->wal_ws + o_sizes);
        w.index = reinterpret_cast<uint4 *>(e->wal_ws + o_index);
        d_index = w.index;
        w.totals = reinterpret_cast<unsigned long long *>(e->wal_ws + o_tot);
        CU(cudaMemsetAsync(w.totals, 0, 32, s));
        const uint32_t grid = (nodes + 255) / 256;
        k_wal_parse<<<grid, 256, 0, s>>>(w);
        for (uint32_t k = 0; k < levels; k++) k_wal_double<<<grid, 256, 0, s>>>(w, k);
        k_wal_select<<<(n_pages + 255) / 256, 256, 0, s>>>(w);
        k_publish<<<1, 256, 0, s>>>(reinterpret_cast<uint32_t *>(e->pin_dev), reinterpret_cast<const uint32_t *>(w.totals), 6,
                                    nullptr, nullptr, 0);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(s));
        if (!device) cudaEventElapsedTime(&ms_h2d, e->ev[EV_H2D0], e->ev[EV_H2D1]);
    }
    unsigned long long totals[3];
    memcpy(totals, e->pin, sizeof totals);
    const uint64_t n_rec = totals[0], bytes = totals[1];
    const uint32_t wal_launches = levels + 3;
    if (totals[2] & kWalTooLarge) return fail(e, DBEEL_ERR_ITEM_TOO_LARGE, "a logged entry exceeds u32::MAX bytes");
    if (n_rec == 0) { e->stats = dbeel_stats{}; e->stats.kernel_launches = wal_launches; return DBEEL_OK; }

    // ---- the flush: the log is the batch's .data, the selected records its (sparse) .index
    dbeel_compact_opts o;
    default_opts(&o);
    JobExtra ex;
    ex.sparse_offsets = true;
    ex.data_bytes = bytes;
    dbeel_run batch{d_wal, wal_len, d_index, n_rec * 16};
    if (data_cap_user < bytes || index_cap_user < n_rec * 16) return fail(e, DBEEL_ERR_CAPACITY, "output buffer too small for the replayed entries");
    int rc;
    if (device) {
        BusyGuard g(e);
        e->stats.ms_h2d = 0;
        rc = run_job_device(e, &batch, 1, &o, true, out, true, &ex);
    } else {
        BusyGuard g(e);
        rc = ensure_device(e, &e->stage_out, &e->stage_out_cap, align_up(bytes + 16, kAlign) + align_up(n_rec * 16 + 16, kAlign));
        if (rc) return rc;
        dbeel_out dout = {};
        dout.data = e->stage_out;
        dout.data_cap = bytes;
        dout.index = e->stage_out + align_up(bytes + 16, kAlign);
        dout.index_cap = n_rec * 16;
        e->stats.ms_h2d = ms_h2d;
        rc = run_job_device(e, &batch, 1, &o, true, &dout, true, &ex);
        if (!rc && dout.items_written <= capacity) {
            if (dout.data_len) CU(cudaMemcpyAsync(user_data, dout.data, dout.data_len, cudaMemcpyDeviceToHost, s));
            if (dout.index_len) CU(cudaMemcpyAsync(user_index, dout.index, dout.index_len, cudaMemcpyDeviceToHost, s));
            CU(cudaStreamSynchronize(s));
        }
        out->data_len = dout.data_len;
        out->index_len = dout.index_len;
        out->items_written = dout.items_written;
    }
    if (rc) return rc;
    e->stats.kernel_launches += wal_launches;
    e->stats.input_bytes = wal_len;
    if (out->items_written > capacity) { // memtable.set(..)? -> ReachedCapacity (lsm_tree.rs:566, rbtree_arena lib.rs:458-461)
        out->data_len = out->index_len = out->items_written = 0;
        return fail(e, DBEEL_ERR_TREE_FULL, "the log holds more distinct keys than the memtable capacity");
    }
    return DBEEL_OK;
}


// ------------------------------------------------------------------------------------ N1: compact-many

struct JobShapes {
    std::vector<JobShape> shape;
    std::vector<uint64_t> bloom_off;
    uint64_t data = 0, index = 0, bloom = 0, entries = 0, runs = 0;
};

int job_shapes(dbeel_engine *e, const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size, double fp, JobShapes *js) {
    if (!(fp > 0.0 && fp < 1.0)) return e ? fail(e, DBEEL_ERR_INVALID_ARG, "bloom_fp must be in (0,1)") : DBEEL_ERR_INVALID_ARG;
    dbeel_compact_opts o;
    default_opts(&o);
    o.bloom_min_size = bloom_min_size;
    o.bloom_fp = fp;
    js->shape.assign(n_jobs, JobShape{});
    js->bloom_off.assign(n_jobs, 0);
    for (uint32_t g = 0; g < n_jobs; g++) {
        if (jobs[g].n_runs && !jobs[g].runs) return e ? fail(e, DBEEL_ERR_INVALID_ARG, "null run array") : DBEEL_ERR_INVALID_ARG;
        shape_of(jobs[g].runs, jobs[g].n_runs, &o, false, &js->shape[g]);
        js->data += js->shape[g].data_total;
        js->index += js->shape[g].n_total * 16;
        js->entries += js->shape[g].n_total;
        js->runs += jobs[g].n_runs;
        js->bloom_off[g] = js->bloom;
        js->bloom += align_up(js->shape[g].bloom_file, 16);
    }
    return DBEEL_OK;
}

int compact_many_entry(dbeel_engine *e, const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size, double fp, dbeel_out *out,
                       dbeel_job_result *results, bool device) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!out || (n_jobs && (!jobs || !results))) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g0(e);
    e->err.clear();
    out->data_len = out->index_len = out->bloom_len = out->items_written = 0;
    JobShapes js;
    int rc = job_shapes(e, jobs, n_jobs, bloom_min_size, fp, &js);
    if (rc) return rc;
    for (uint32_t g = 0; g < n_jobs; g++) results[g] = dbeel_job_result{0, 0, 0, 0, 0, 0, 0};
    if (js.runs > DBEEL_MAX_RUNS) return fail(e, DBEEL_ERR_TOO_MANY_RUNS, "more than DBEEL_MAX_RUNS runs over all jobs");
    if (js.entries >= 0xFFFFFFFEull) return fail(e, DBEEL_ERR_TOO_MANY_ENTRIES, "too many entries");
    if (out->data_cap < js.data || out->index_cap < js.index || out->bloom_cap < js.bloom)
        return fail(e, DBEEL_ERR_CAPACITY, "output buffer smaller than dbeel_compact_many_bound");
    if (n_jobs == 0 || js.entries == 0) { e->stats = dbeel_stats{}; return DBEEL_OK; }
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    cudaStream_t s = e->stream;

    // all runs back to back; host buffers are staged down first
    std::vector<dbeel_run> flat;
    std::vector<uint32_t> first(n_jobs + 1, 0);
    std::vector<int32_t> keep(n_jobs);
    for (uint32_t g = 0; g < n_jobs; g++) {
        first[g] = (uint32_t)flat.size();
        keep[g] = jobs[g].keep_tombstones;
        for (uint32_t r = 0; r < jobs[g].n_runs; r++) flat.push_back(jobs[g].runs[r]);
    }
    first[n_jobs] = (uint32_t)flat.size();
    dbeel_out dout = *out;
    if (!device) {
        uint64_t in_need = 0;
        for (auto &r : flat) {
            if ((r.data_len && !r.data) || (r.index_len && !r.index)) return fail(e, DBEEL_ERR_INVALID_ARG, "null run buffer");
            in_need += align_up(r.data_len + 32, kAlign) + align_up(r.index_len + 16, kAlign);
        }
        rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, in_need);
        if (!rc) rc = ensure_device(e, &e->stage_out, &e->stage_out_cap,
                                    align_up(js.data + 16, kAlign) + align_up(js.index + 16, kAlign) + align_up(js.bloom + 16, kAlign));
        if (rc) return rc;
        uint64_t pos = 0;
        for (auto &r : flat) {
            const void *hd = r.data, *hi = r.index;
            r.data = e->stage_in + pos;
            if (r.data_len) CU(cudaMemcpyAsync(e->stage_in + pos, hd, r.data_len, cudaMemcpyHostToDevice, s));
            pos += align_up(r.data_len + 32, kAlign);
            r.index = e->stage_in + pos;
            if (r.index_len) CU(cudaMemcpyAsync(e->stage_in + pos, hi, r.index_len, cudaMemcpyHostToDevice, s));
            pos += align_up(r.index_len + 16, kAlign);
        }
        dout.data = e->stage_out;
        dout.index = e->stage_out + align_up(js.data + 16, kAlign);
        dout.bloom = e->stage_out + align_up(js.data + 16, kAlign) + align_up(js.index + 16, kAlign);
    } else if ((uintptr_t)out->bloom & 15) {
        return fail(e, DBEEL_ERR_INVALID_ARG, "device output buffers must be 16-byte aligned");
    }
    // per-job filters
    std::vector<BloomParams> bloom(n_jobs);
    for (uint32_t g = 0; g < n_jobs; g++) {
        bloom[g] = BloomParams{};
        const JobShape &sh = js.shape[g];
        if (!sh.bloom_file) continue;
        uint8_t seed[32];
        if (jobs[g].bloom_seed) {
            memcpy(seed, jobs[g].bloom_seed, 32);
        } else {
            FILE *f = fopen("/dev/urandom", "rb");
            if (!f || fread(seed, 1, 32, f) != 32) {
                if (f) fclose(f);
                return fail(e, DBEEL_ERR_INVALID_ARG, "no entropy source for the bloom seed");
            }
            fclose(f);
        }
        bloom[g].words = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(dout.bloom) + js.bloom_off[g] + 8);
        bloom[g].bits = sh.bloom_bits;
        bloom[g].bits_magic = (uint64_t)((((unsigned __int128)1) << 64) / sh.bloom_bits);
        bloom[g].k_num = sh.bloom_k;
        for (int i = 0; i < 4; i++) memcpy(&bloom[g].sip[i], seed + 8 * i, 8);
    }
    if (js.bloom) CU(cudaMemsetAsync(dout.bloom, 0, js.bloom, s));
    dbeel_compact_opts o;
    default_opts(&o);
    o.bloom_min_size = bloom_min_size;
    o.bloom_fp = fp;
    JobExtra ex;
    ex.n_jobs = n_jobs;
    ex.job_first = first.data();
    ex.job_keep = keep.data();
    ex.job_bloom = bloom.data();
    ex.job_results = results;
    e->stats.ms_h2d = 0;
    rc = run_job_device(e, flat.data(), (uint32_t)flat.size(), &o, false, &dout, true, &ex);
    if (rc) return rc;
    for (uint32_t g = 0; g < n_jobs; g++) {
        results[g].bloom_off = js.bloom_off[g];
        results[g].bloom_len = js.shape[g].bloom_file;
    }
    if (!device) {
        if (dout.data_len) CU(cudaMemcpyAsync(out->data, dout.data, dout.data_len, cudaMemcpyDeviceToHost, s));
        if (dout.index_len) CU(cudaMemcpyAsync(out->index, dout.index, dout.index_len, cudaMemcpyDeviceToHost, s));
        if (js.bloom) CU(cudaMemcpyAsync(out->bloom, dout.bloom, js.bloom, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    out->data_len = dout.data_len;
    out->index_len = dout.index_len;
    out->bloom_len = js.bloom;
    out->items_written = dout.items_written;
    e->stats.output_bytes += js.bloom;
    return DBEEL_OK;
}

// ------------------------------------------------------------------------------------ hash-range scans (scan.cuh)

// The device-resident scan.  tables / out hold device pointers; ranges, per_range and stop live in the host's memory.
// data_bound / index_bound: what the selected entries can take at most (the scanned tables' .data bytes, 16 per record);
// the caller's caps above them change nothing.
int run_scan_device(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges, uint32_t n_ranges,
                    uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range, dbeel_scan_stop *stop) {
    dbeel_stats &st = e->stats;
    // the scan ends in front of the first table without a record: its first 16-byte index read hits EOF (lsm_tree.rs:250)
    uint32_t nt = 0;
    uint64_t n64 = 0, data_bound = 0, in_bytes = 0;
    while (nt < n_tables && tables[nt].index_len >= DBEEL_INDEX_ENTRY_SIZE) {
        n64 += tables[nt].index_len / DBEEL_INDEX_ENTRY_SIZE;
        data_bound += tables[nt].data_len;
        in_bytes += tables[nt].data_len + tables[nt].index_len;
        nt++;
    }
    const bool empty_stop = nt < n_tables;
    if (n64 >= 0xFFFFFFF0ull) return fail(e, DBEEL_ERR_TOO_MANY_ENTRIES, "more than 2^32 - 16 records in one scan");
    const uint32_t N = (uint32_t)n64;
    st.entries_in = N;
    st.input_bytes = in_bytes;
    *stop = empty_stop ? dbeel_scan_stop{(int32_t)nt, DBEEL_SCAN_READ, 0} : dbeel_scan_stop{-1, DBEEL_SCAN_END, 0};
    if (N == 0) return DBEEL_OK;

    // no ranges: one class that selects nothing, so the scan still finds its stop
    const uint32_t n_cls = n_ranges ? n_ranges : 1;
    const uint64_t data_cap = std::min<uint64_t>(out->data_cap, data_bound), index_cap = std::min<uint64_t>(out->index_cap, 16ull * N);
    const uint64_t gather_tiles = (data_cap + kGatherTileBytes - 1) / kGatherTileBytes;
    const uint32_t n_blocks = (N + kRouteThreads - 1) / kRouteThreads;
    const uint64_t res_tiles = (N + kResolveThreads - 1) / kResolveThreads, res_chunks = (res_tiles + 1023) / 1024;

    uint64_t off = 0;
    auto carve = [&](uint64_t b) { uint64_t o2 = off; off = align_up(off + b, kAlign); return o2; };
    // header block (host-initialised, goes down through the mapped pinned block): ctl | tables | ranges | mem_table, stop
    const uint64_t o_ctl = carve(sizeof(Ctl)), o_tab = carve(sizeof(ScanTable) * nt), o_rng = carve(8ull * n_cls);
    const uint64_t o_mt = carve(16ull * (n_cls + 1) + 8); // k_flush_table's rows, then the stop key: published together
    const uint64_t header_bytes = off;
    const uint64_t o_seg = carve(sizeof(Seg) * n_cls), o_tot = carve(8ull * (3 * n_cls + 1)), o_hist = carve(4ull * n_blocks * n_cls);
    const uint64_t o_cls = carve(4ull * N), o_rec = carve(16ull * N), o_res = carve(16ull * N), o_src = carve(8ull * N);
    const uint64_t o_tb = carve(8 * res_tiles), o_tc = carve(4 * res_tiles), o_cb = carve(8 * res_chunks), o_cc = carve(4 * res_chunks);
    const uint64_t o_tf = carve(4ull * (gather_tiles + 2));
    int rc = ensure_device(e, &e->ws, &e->ws_cap, off);
    const uint64_t o_hctl = header_bytes, o_hmt = o_hctl + align_up(sizeof(Ctl), 64), o_htot = o_hmt + align_up(16ull * (n_cls + 1) + 8, 64);
    if (!rc) rc = ensure_pinned(e, o_htot + 8ull * (3 * n_cls + 1));
    if (rc) return rc;
    uint8_t *ws = e->ws, *h = e->pin;

    memset(h, 0, header_bytes);
    ScanTable *ht = reinterpret_cast<ScanTable *>(h + o_tab);
    for (uint32_t t = 0, base = 0; t < nt; t++) {
        ht[t] = ScanTable{static_cast<const uint8_t *>(tables[t].data), tables[t].data_len, static_cast<const uint4 *>(tables[t].index), base,
                          (uint32_t)(tables[t].index_len / DBEEL_INDEX_ENTRY_SIZE)};
        base += ht[t].n;
    }
    uint2 *hr = reinterpret_cast<uint2 *>(h + o_rng);
    for (uint32_t r = 0; r < n_ranges; r++) hr[r] = make_uint2(ranges[r].start, ranges[r].end);
    if (!n_ranges) hr[0] = make_uint2(0, 0); // start == end holds for no hash in either mode
    unsigned long long *hstop = reinterpret_cast<unsigned long long *>(h + o_mt + 16ull * (n_cls + 1));
    *hstop = empty_stop ? (((unsigned long long)N << 2) | DBEEL_SCAN_READ) : ~0ull;

    ScanParams sp;
    sp.tables = reinterpret_cast<const ScanTable *>(ws + o_tab);
    sp.n_tables = nt;
    sp.n = N;
    sp.ranges = reinterpret_cast<const uint2 *>(ws + o_rng);
    sp.n_ranges = n_cls;
    sp.mode = mode;
    sp.cls = reinterpret_cast<uint32_t *>(ws + o_cls);
    sp.rec = reinterpret_cast<uint4 *>(ws + o_rec);
    sp.stop = reinterpret_cast<unsigned long long *>(ws + o_mt + 16ull * (n_cls + 1));
    sp.totals = reinterpret_cast<unsigned long long *>(ws + o_tot);
    sp.ctl = reinterpret_cast<Ctl *>(ws + o_ctl);
    sp.seg = reinterpret_cast<Seg *>(ws + o_seg);
    sp.data_cap = data_cap;
    sp.index_cap = index_cap;

    RouteParams rp;
    memset(&rp, 0, sizeof rp);
    rp.index = sp.rec; // the res record of every selected entry is what the split moves
    rp.n = N;
    rp.n_shards = n_cls;
    rp.n_blocks = n_blocks;
    rp.shard_of = sp.cls;
    rp.hist = reinterpret_cast<uint32_t *>(ws + o_hist);
    rp.totals = sp.totals;
    rp.out_index = reinterpret_cast<uint4 *>(ws + o_res);
    rp.stop = sp.stop;

    Params p;
    memset(&p, 0, sizeof p);
    p.n_total = N;
    p.ctl = sp.ctl;
    p.seg[0] = sp.seg; // n_levels 0: a range is a group, its first res position its segment start
    p.n_groups = n_cls;
    p.mem_table = reinterpret_cast<unsigned long long *>(ws + o_mt);
    p.tile_bytes = reinterpret_cast<unsigned long long *>(ws + o_tb);
    p.tile_count = reinterpret_cast<uint32_t *>(ws + o_tc);
    p.chunk_bytes = reinterpret_cast<unsigned long long *>(ws + o_cb);
    p.chunk_count = reinterpret_cast<uint32_t *>(ws + o_cc);
    p.src_ptr = reinterpret_cast<unsigned long long *>(ws + o_src);
    p.tile_first = reinterpret_cast<uint32_t *>(ws + o_tf);
    p.tile_first_n = (uint32_t)(gather_tiles + 2);
    p.out_data = static_cast<uint8_t *>(out->data);
    p.out_index = static_cast<uint4 *>(out->index);
    const uint4 *res = rp.out_index;

    cudaStream_t s = e->stream;
    uint32_t launches = 0;
    CU(cudaEventRecord(e->ev[EV_START], s));
    k_copy_words<<<(uint32_t)((header_bytes / 4 + 255) / 256), 256, 0, s>>>(reinterpret_cast<uint32_t *>(ws), reinterpret_cast<const uint32_t *>(e->pin_dev),
                                                                            (uint32_t)(header_bytes / 4));
    CU(cudaMemsetAsync(sp.totals, 0, 8ull * (3 * n_cls + 1), s));
    k_scan_classify<<<(N + 255) / 256, 256, 0, s>>>(sp);
    CU(cudaEventRecord(e->ev[EV_EXTRACT], s));
    k_route_hash<true><<<n_blocks, kRouteThreads, 0, s>>>(rp);
    k_route_scan<<<n_cls, 1024, 0, s>>>(rp);
    k_route_starts<<<1, 256, 0, s>>>(rp, reinterpret_cast<unsigned long long *>(e->pin_dev + o_htot));
    k_route_scatter<<<n_blocks, kRouteThreads, 0, s>>>(rp);
    k_scan_plan<<<1, 256, 0, s>>>(sp);
    k_scan_res_tiles<<<(uint32_t)res_tiles, kResolveThreads, 0, s>>>(p, res);
    k_scan_tiles<<<(uint32_t)res_chunks, 1024, 0, s>>>(p);
    k_scan_chunks<<<1, 1024, 0, s>>>(p);
    k_emit<<<(uint32_t)res_tiles, kResolveThreads, 0, s>>>(p, res);
    k_flush_table<<<(n_cls + 1 + 127) / 128, 128, 0, s>>>(p, res);
    CU(cudaEventRecord(e->ev[EV_RESOLVE], s));
    launches += 12;
    if (gather_tiles) {
        if (((uintptr_t)out->data & 31) == 0) k_gather32<false, false, false, true><<<(uint32_t)gather_tiles, kGatherThreads, 0, s>>>(p);
        else k_gather<<<(uint32_t)gather_tiles, kGatherThreads, 0, s>>>(p);
        launches++;
    }
    k_rebase_index<<<(N + 255) / 256, 256, 0, s>>>(p); // after the gather: it reads the offsets as stream offsets
    CU(cudaEventRecord(e->ev[EV_GATHER], s));
    k_publish<<<1, 256, 0, s>>>(reinterpret_cast<uint32_t *>(e->pin_dev + o_hctl), reinterpret_cast<const uint32_t *>(sp.ctl),
                                (uint32_t)(sizeof(Ctl) / 4), reinterpret_cast<uint32_t *>(e->pin_dev + o_hmt),
                                reinterpret_cast<const uint32_t *>(p.mem_table), (uint32_t)(4 * (n_cls + 1) + 2));
    launches += 2;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s));

    const Ctl *hc = reinterpret_cast<const Ctl *>(h + o_hctl);
    const unsigned long long *hmt = reinterpret_cast<const unsigned long long *>(h + o_hmt);
    const unsigned long long key = hmt[2 * (n_cls + 1)];
    st.kernel_launches = launches;
    cudaEventElapsedTime(&st.ms_total, e->ev[EV_START], e->ev[EV_GATHER]);
    cudaEventElapsedTime(&st.ms_extract, e->ev[EV_START], e->ev[EV_EXTRACT]);
    cudaEventElapsedTime(&st.ms_resolve, e->ev[EV_EXTRACT], e->ev[EV_RESOLVE]);
    cudaEventElapsedTime(&st.ms_gather, e->ev[EV_RESOLVE], e->ev[EV_GATHER]);
    st.entries_valid = key == ~0ull ? N : (uint32_t)(key >> 2);
    if (key != ~0ull && !(empty_stop && (key >> 2) == N)) {
        const uint32_t o = (uint32_t)(key >> 2);
        uint32_t t = 0;
        while (t + 1 < nt && ht[t + 1].base <= o) t++;
        *stop = dbeel_scan_stop{(int32_t)t, (uint32_t)(key & 3), (uint64_t)(o - ht[t].base)};
    }
    if (hc->flags & kScanOverCap) return fail(e, DBEEL_ERR_CAPACITY, "scan output larger than the output buffers");
    out->data_len = hc->out_data_len;
    out->items_written = hc->out_items;
    out->index_len = 16ull * hc->out_items;
    for (uint32_t r = 0; r < n_ranges; r++) {
        dbeel_flush_table &row = per_range[r];
        row.data_off = hmt[2 * r];
        row.data_len = hmt[2 * (r + 1)] - hmt[2 * r];
        row.items = hmt[2 * (r + 1) + 1] - hmt[2 * r + 1];
        row.index_off = hmt[2 * r + 1] * 16;
        row.index_len = row.items * 16;
    }
    st.entries_out = hc->out_items;
    st.output_bytes = out->data_len + out->index_len;
    st.gather_bytes = 2 * out->data_len + out->index_len + 8ull * hc->out_items;
    st.partitions = 1;
    return DBEEL_OK;
}

int scan_entry(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges, uint32_t n_ranges,
               uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range, dbeel_scan_stop *stop, bool device) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!out || !stop || (n_tables && !tables) || (n_ranges && (!ranges || !per_range))) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (mode > DBEEL_SCAN_EXACT) return fail(e, DBEEL_ERR_INVALID_ARG, "unknown scan mode");
    if (n_ranges > DBEEL_MAX_SCAN_RANGES) return fail(e, DBEEL_ERR_INVALID_ARG, "more than DBEEL_MAX_SCAN_RANGES ranges");
    for (uint32_t t = 0; t < n_tables; t++) {
        if ((tables[t].data_len && !tables[t].data) || (tables[t].index_len >= 16 && !tables[t].index)) return fail(e, DBEEL_ERR_INVALID_ARG, "null table buffer");
        if (device && ((uintptr_t)tables[t].index & 15)) return fail(e, DBEEL_ERR_INVALID_ARG, "device .index buffers must be 16-byte aligned");
    }
    if (device && (((uintptr_t)out->data | (uintptr_t)out->index) & 15)) return fail(e, DBEEL_ERR_INVALID_ARG, "device output buffers must be 16-byte aligned");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    e->stats = dbeel_stats{};
    out->data_len = out->index_len = out->bloom_len = out->items_written = 0;
    for (uint32_t r = 0; r < n_ranges; r++) per_range[r] = dbeel_flush_table{0, 0, 0, 0, 0};
    *stop = dbeel_scan_stop{-1, DBEEL_SCAN_END, 0};
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    if (device) {
        if ((out->data_cap && !out->data) || (out->index_cap && !out->index)) return fail(e, DBEEL_ERR_INVALID_ARG, "null output buffer");
        return run_scan_device(e, tables, n_tables, ranges, n_ranges, mode, out, per_range, stop);
    }
    // host buffers: every table goes down whole, the outputs come back (the tree must fit in device memory)
    uint64_t need = 0, data_bound = 0, n_rec = 0;
    for (uint32_t t = 0; t < n_tables; t++) {
        need += align_up(tables[t].data_len + 16, kAlign) + align_up(tables[t].index_len + 16, kAlign);
        data_bound += tables[t].data_len;
        n_rec += tables[t].index_len / DBEEL_INDEX_ENTRY_SIZE;
    }
    if ((out->data_cap && !out->data) || (out->index_cap && !out->index)) return fail(e, DBEEL_ERR_INVALID_ARG, "null output buffer");
    const uint64_t dcap = std::min<uint64_t>(out->data_cap, data_bound), icap = std::min<uint64_t>(out->index_cap, 16 * n_rec);
    int rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, std::max<uint64_t>(need, 256));
    if (!rc) rc = ensure_device(e, &e->stage_out, &e->stage_out_cap, align_up(dcap + 16, kAlign) + icap + 16);
    if (rc) return rc;
    cudaStream_t s = e->stream;
    CU(cudaEventRecord(e->ev[EV_H2D0], s));
    std::vector<dbeel_run> dt(n_tables);
    uint64_t pos = 0;
    for (uint32_t t = 0; t < n_tables; t++) {
        uint8_t *dd = e->stage_in + pos;
        pos += align_up(tables[t].data_len + 16, kAlign);
        uint8_t *di = e->stage_in + pos;
        pos += align_up(tables[t].index_len + 16, kAlign);
        if (tables[t].data_len) CU(cudaMemcpyAsync(dd, tables[t].data, tables[t].data_len, cudaMemcpyHostToDevice, s));
        if (tables[t].index_len) CU(cudaMemcpyAsync(di, tables[t].index, tables[t].index_len, cudaMemcpyHostToDevice, s));
        dt[t] = dbeel_run{dd, tables[t].data_len, di, tables[t].index_len};
    }
    CU(cudaEventRecord(e->ev[EV_H2D1], s));
    dbeel_out dout = {e->stage_out, dcap, 0, e->stage_out + align_up(dcap + 16, kAlign), icap, 0, nullptr, 0, 0, 0};
    rc = run_scan_device(e, dt.data(), n_tables, ranges, n_ranges, mode, &dout, per_range, stop);
    CU(cudaEventSynchronize(e->ev[EV_H2D1]));
    cudaEventElapsedTime(&e->stats.ms_h2d, e->ev[EV_H2D0], e->ev[EV_H2D1]);
    if (rc) return rc;
    CU(cudaEventRecord(e->ev[EV_D2H0], s));
    if (dout.data_len) CU(cudaMemcpyAsync(out->data, dout.data, dout.data_len, cudaMemcpyDeviceToHost, s));
    if (dout.index_len) CU(cudaMemcpyAsync(out->index, dout.index, dout.index_len, cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(e->ev[EV_D2H1], s));
    CU(cudaStreamSynchronize(s));
    cudaEventElapsedTime(&e->stats.ms_d2h, e->ev[EV_D2H0], e->ev[EV_D2H1]);
    out->data_len = dout.data_len;
    out->index_len = dout.index_len;
    out->items_written = dout.items_written;
    return DBEEL_OK;
}

// ------------------------------------------------------------------------------------ streamed hash-range scans
// dbeel_scan_ranges_stream: the tables come through the read callback one partition at a time (host/scan_plan.h), every
// range's output leaves through the write callback as its own stream.  Per partition c:
//   reader threads   c's .data spans -> pinned ring slot c mod R (the .index files are read whole first: the plan needs them)
//   engine thread    H2D of c's spans and index slices -> device buffer c & 1; the scan kernels over c's records; the
//                    exact-size D2H of c's range-major output -> pinned output slot c mod R, once c's header has arrived
//   writer threads   every range's piece of c -> the write callback, at the range's running stream offsets
// The engine enqueues c + 1's kernels before it waits for c's header, so the copies and the kernels keep overlapping; the
// stop word and the running per-range totals live on the device (k_scan_part_enter / _leave), so the kernels of c + 1
// never depend on the host having seen c.
int scan_stream_entry(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges, uint32_t n_ranges,
                      uint32_t mode, const dbeel_scan_io *io, uint64_t partition_bytes, dbeel_flush_table *per_range, dbeel_scan_stop *stop) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!stop || !io || !io->read || !io->write || (n_tables && !tables) || (n_ranges && (!ranges || !per_range)))
        return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (mode > DBEEL_SCAN_EXACT) return fail(e, DBEEL_ERR_INVALID_ARG, "unknown scan mode");
    if (n_ranges > DBEEL_MAX_SCAN_RANGES) return fail(e, DBEEL_ERR_INVALID_ARG, "more than DBEEL_MAX_SCAN_RANGES ranges");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    e->stats = dbeel_stats{};
    dbeel_stats &st = e->stats;
    for (uint32_t r = 0; r < n_ranges; r++) per_range[r] = dbeel_flush_table{0, 0, 0, 0, 0};
    *stop = dbeel_scan_stop{-1, DBEEL_SCAN_END, 0};
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    const uint64_t budget = partition_bytes ? partition_bytes : e->partition_bytes;

    // ---- 1. the .index files of the tables in front of the first one without a record, whole, into page-locked memory
    uint32_t nt = 0;
    uint64_t need = 0;
    std::vector<uint64_t> ioff, tbase; // pinned offset of table t's .index; ordinal of its record 0
    while (nt < n_tables && tables[nt].index_len >= DBEEL_INDEX_ENTRY_SIZE) {
        ioff.push_back(need);
        tbase.push_back(st.entries_in);
        need += align_up(tables[nt].index_len / 16 * 16 + 16, kAlign);
        st.entries_in += tables[nt].index_len / DBEEL_INDEX_ENTRY_SIZE;
        st.input_bytes += tables[nt].data_len + tables[nt].index_len;
        nt++;
    }
    int rc = ensure_host(e, &e->pin_index, &e->pin_index_cap, std::max<uint64_t>(need, 256));
    if (rc) return rc;
    {
        std::vector<StreamPump::ReadTask> rt;
        for (uint32_t t = 0; t < nt; t++)
            for (uint64_t d = 0, n = tables[t].index_len / 16 * 16; d < n; d += StreamPump::kPiece)
                rt.push_back(StreamPump::ReadTask{0, t, DBEEL_STREAM_INDEX, d, std::min<uint64_t>(StreamPump::kPiece, n - d), e->pin_index + ioff[t] + d});
        rc = parallel_pieces(rt.size(), [&](size_t k) { return io->read(io->ctx, rt[k].run, rt[k].kind, rt[k].off, rt[k].len, rt[k].dst); });
        if (rc) return fail(e, rc, "scan read callback failed (.index)");
    }

    // ---- 2. the plan (it schedules nothing at or after the first READ stop)
    std::vector<ScanPlanTable> pt(nt);
    for (uint32_t t = 0; t < nt; t++) pt[t] = ScanPlanTable{tables[t].data_len, e->pin_index + ioff[t], tables[t].index_len / DBEEL_INDEX_ENTRY_SIZE};
    const ScanPlan plan = scan_plan(pt.data(), nt, budget);
    // table t stops the scan at record r when the scan gets there: as nt < n_tables (an empty table) or the plan found
    if (plan.stopped) *stop = dbeel_scan_stop{(int32_t)plan.stop_table, DBEEL_SCAN_READ, plan.stop_record};
    else if (nt < n_tables) *stop = dbeel_scan_stop{(int32_t)nt, DBEEL_SCAN_READ, 0};
    st.entries_valid = plan.scheduled;
    const uint32_t np = (uint32_t)plan.parts.size();
    if (np == 0) return DBEEL_OK;

    // ---- 3. slot layouts: every piece's span (+32 bytes of slack for the narrow loads, aligned), then its index slice
    auto span_room = [](const ScanPiece &k) { return align_up(k.span_hi - k.span_lo + 32, kAlign); };
    auto slice_room = [](const ScanPiece &k) { return align_up(16 * (k.rec_hi - k.rec_lo) + 16, kAlign); };
    uint64_t max_in = 0, max_out = 0, max_n = 0, max_tiles = 0;
    for (const ScanPart &q : plan.parts) {
        uint64_t in = 0;
        for (uint32_t k = q.first_piece; k < q.first_piece + q.n_pieces; k++) in += span_room(plan.pieces[k]) + slice_room(plan.pieces[k]);
        max_in = std::max(max_in, in);
        max_out = std::max(max_out, align_up(q.data_bytes + 16, kAlign) + align_up(16 * q.records + 16, kAlign));
        max_n = std::max(max_n, q.records);
        max_tiles = std::max<uint64_t>(max_tiles, (q.data_bytes + kGatherTileBytes - 1) / kGatherTileBytes);
    }
    const uint32_t n_cls = n_ranges ? n_ranges : 1; // no ranges: one class that selects nothing, so the stop is still found
    const uint32_t NM = (uint32_t)max_n;
    const uint64_t blocks_max = (NM + kRouteThreads - 1) / kRouteThreads;
    const uint64_t tiles_max = (NM + kResolveThreads - 1) / kResolveThreads, chunks_max = (tiles_max + 1023) / 1024;
    uint64_t off = 0;
    auto carve = [&](uint64_t b) { uint64_t o2 = off; off = align_up(off + b, kAlign); return o2; };
    const uint64_t o_tab = carve(sizeof(ScanTable) * plan.pieces.size()), o_rng = carve(8ull * n_cls), o_ctl = carve(sizeof(Ctl));
    const uint64_t o_mt = carve(16ull * (n_cls + 1)), o_lstop = carve(8), o_gstop = carve(8), o_run = carve(16ull * n_cls);
    const uint64_t o_seg = carve(sizeof(Seg) * n_cls), o_tot = carve(8ull * (3 * n_cls + 1)), o_rtot = carve(8ull * (3 * n_cls + 1));
    const uint64_t o_hist = carve(4ull * blocks_max * n_cls);
    const uint64_t o_cls = carve(4ull * NM), o_rec = carve(16ull * NM), o_res = carve(16ull * NM), o_src = carve(8ull * NM);
    const uint64_t o_tb = carve(8 * tiles_max), o_tc = carve(4 * tiles_max), o_cb = carve(8 * chunks_max), o_cc = carve(4 * chunks_max);
    const uint64_t o_tf = carve(4ull * (max_tiles + 2));
    const uint64_t hdr_stride = align_up(8 + sizeof(ScanPieceRow) * n_cls, 64);
    const uint32_t R = (uint32_t)std::max(2, e->stream_ring);
    rc = ensure_device(e, &e->ws, &e->ws_cap, off);
    if (!rc) rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, max_in);
    if (!rc) rc = ensure_device(e, &e->stage_in2, &e->stage_in2_cap, max_in);
    if (!rc) rc = ensure_device(e, &e->stage_out, &e->stage_out_cap, max_out);
    if (!rc) rc = ensure_device(e, &e->stage_out2, &e->stage_out2_cap, max_out);
    if (!rc) rc = ensure_pinned(e, 2 * hdr_stride);
    if (!rc) rc = ensure_host(e, &e->ring_in, &e->ring_in_cap, (uint64_t)R * max_in);
    if (!rc) rc = ensure_host(e, &e->ring_out, &e->ring_out_cap, (uint64_t)R * max_out);
    if (rc) return rc;
    if (!e->s_h2d) {
        CU(cudaStreamCreateWithFlags(&e->s_h2d, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CU(cudaEventCreateWithFlags(&e->ev_h2d[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&e->ev_comp[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&e->ev_d2h[i], cudaEventDisableTiming));
        }
    }
    uint8_t *ws = e->ws, *sin[2] = {e->stage_in, e->stage_in2}, *sout[2] = {e->stage_out, e->stage_out2};
    cudaStream_t s = e->stream;

    // every partition's ScanTables (device input buffer c & 1 is known in advance), the ranges, the cross-partition state
    std::vector<ScanTable> ht(plan.pieces.size());
    std::vector<std::vector<uint64_t>> span_at(np); // slot offset of every piece's span
    for (uint32_t c = 0; c < np; c++) {
        const ScanPart &q = plan.parts[c];
        uint64_t pos = 0;
        for (uint32_t k = q.first_piece; k < q.first_piece + q.n_pieces; k++) {
            const ScanPiece &pc = plan.pieces[k];
            span_at[c].push_back(pos);
            const uint8_t *span = sin[c & 1] + pos;
            pos += span_room(pc);
            ht[k] = ScanTable{span - pc.span_lo, tables[pc.table].data_len, reinterpret_cast<const uint4 *>(sin[c & 1] + pos),
                              (uint32_t)(tbase[pc.table] + pc.rec_lo - q.first_ordinal), (uint32_t)(pc.rec_hi - pc.rec_lo)};
            pos += slice_room(pc);
        }
    }
    std::vector<uint2> hr(n_cls, make_uint2(0, 0)); // no ranges: start == end holds for no hash in either mode
    for (uint32_t r = 0; r < n_ranges; r++) hr[r] = make_uint2(ranges[r].start, ranges[r].end);
    CU(cudaMemcpyAsync(ws + o_tab, ht.data(), sizeof(ScanTable) * ht.size(), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(ws + o_rng, hr.data(), 8ull * n_cls, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(ws + o_gstop, 0xFF, 8, s));
    CU(cudaMemsetAsync(ws + o_run, 0, 16ull * n_cls, s));
    CU(cudaStreamSynchronize(s)); // ht / hr are pageable

    // the pump: R-slot pinned rings, one event per partition for the writer threads.  Declared in this order so that the
    // pump's threads are joined before the events they wait on are destroyed.
    struct EventList {
        std::vector<cudaEvent_t> ev;
        ~EventList() { for (auto &x : ev) if (x) cudaEventDestroy(x); }
    } ev_out;
    ev_out.ev.assign(np, nullptr);
    for (uint32_t c = 0; c < np; c++) CU(cudaEventCreateWithFlags(&ev_out.ev[c], cudaEventDisableTiming | cudaEventBlockingSync));
    // per device buffer: begin / end of the H2D copies, the kernels and the D2H copies of the partition that last used it
    EventList tev;
    tev.ev.assign(12, nullptr);
    for (auto &x : tev.ev) CU(cudaEventCreate(&x));
    enum { T_H2D = 0, T_KER = 4, T_D2H = 8 };
    auto stage_ms = [&](int stage, uint32_t slot) {
        float ms = 0;
        cudaEventElapsedTime(&ms, tev.ev[stage + 2 * slot], tev.ev[stage + 2 * slot + 1]);
        return ms;
    };
    const dbeel_stream_io rio{io->read, nullptr, io->ctx};
    const int dev = e->device;
    EventList *evl = &ev_out;
    std::unique_ptr<StreamPump> pump(new StreamPump(&rio, np, R, stream_threads(), [evl](uint32_t c) { cudaEventSynchronize(evl->ev[c]); },
                                                    [dev]() { cudaSetDevice(dev); }));
    pump->set_stream_write(io->write);
    for (uint32_t c = 0; c < np; c++) {
        const ScanPart &q = plan.parts[c];
        uint8_t *slot = e->ring_in + (uint64_t)(c % R) * max_in;
        for (uint32_t j = 0; j < q.n_pieces; j++) {
            const ScanPiece &pc = plan.pieces[q.first_piece + j];
            pump->add_read(c, pc.table, DBEEL_STREAM_DATA, pc.span_lo, pc.span_hi - pc.span_lo, slot + span_at[c][j]);
        }
    }
    pump->start();

    auto enqueue_h2d = [&](uint32_t c) -> int {
        const int prc = pump->wait_reads(c);
        if (prc) return fail(e, prc, "scan read callback failed (.data)");
        const ScanPart &q = plan.parts[c];
        const uint8_t *slot = e->ring_in + (uint64_t)(c % R) * max_in;
        CU(cudaEventRecord(tev.ev[T_H2D + 2 * (c & 1)], e->s_h2d));
        for (uint32_t j = 0; j < q.n_pieces; j++) {
            const ScanPiece &pc = plan.pieces[q.first_piece + j];
            const uint64_t sl = pc.span_hi - pc.span_lo, il = 16 * (pc.rec_hi - pc.rec_lo), at = span_at[c][j];
            CU(cudaMemcpyAsync(sin[c & 1] + at, slot + at, sl, cudaMemcpyHostToDevice, e->s_h2d));
            CU(cudaMemcpyAsync(sin[c & 1] + at + span_room(pc), e->pin_index + ioff[pc.table] + 16 * pc.rec_lo, il, cudaMemcpyHostToDevice, e->s_h2d));
        }
        CU(cudaEventRecord(tev.ev[T_H2D + 2 * (c & 1) + 1], e->s_h2d));
        CU(cudaEventRecord(e->ev_h2d[c & 1], e->s_h2d));
        return DBEEL_OK;
    };
    uint32_t launches = 0;
    auto enqueue_kernels = [&](uint32_t c) -> int {
        const ScanPart &q = plan.parts[c];
        const uint32_t N = (uint32_t)q.records;
        const uint32_t n_blocks = (N + kRouteThreads - 1) / kRouteThreads;
        const uint64_t res_tiles = (N + kResolveThreads - 1) / kResolveThreads, res_chunks = (res_tiles + 1023) / 1024;
        const uint64_t gather_tiles = (q.data_bytes + kGatherTileBytes - 1) / kGatherTileBytes;
        uint8_t *od = sout[c & 1], *oi = sout[c & 1] + align_up(q.data_bytes + 16, kAlign);
        ScanParams sp;
        sp.tables = reinterpret_cast<const ScanTable *>(ws + o_tab) + q.first_piece;
        sp.n_tables = q.n_pieces;
        sp.n = N;
        sp.ranges = reinterpret_cast<const uint2 *>(ws + o_rng);
        sp.n_ranges = n_cls;
        sp.mode = mode;
        sp.cls = reinterpret_cast<uint32_t *>(ws + o_cls);
        sp.rec = reinterpret_cast<uint4 *>(ws + o_rec);
        sp.stop = reinterpret_cast<unsigned long long *>(ws + o_lstop);
        sp.totals = reinterpret_cast<unsigned long long *>(ws + o_tot);
        sp.ctl = reinterpret_cast<Ctl *>(ws + o_ctl);
        sp.seg = reinterpret_cast<Seg *>(ws + o_seg);
        sp.data_cap = q.data_bytes;
        sp.index_cap = 16ull * N;
        RouteParams rp;
        memset(&rp, 0, sizeof rp);
        rp.index = sp.rec;
        rp.n = N;
        rp.n_shards = n_cls;
        rp.n_blocks = n_blocks;
        rp.shard_of = sp.cls;
        rp.hist = reinterpret_cast<uint32_t *>(ws + o_hist);
        rp.totals = sp.totals;
        rp.out_index = reinterpret_cast<uint4 *>(ws + o_res);
        rp.stop = sp.stop;
        Params p;
        memset(&p, 0, sizeof p);
        p.n_total = N;
        p.ctl = sp.ctl;
        p.seg[0] = sp.seg;
        p.n_groups = n_cls;
        p.mem_table = reinterpret_cast<unsigned long long *>(ws + o_mt);
        p.tile_bytes = reinterpret_cast<unsigned long long *>(ws + o_tb);
        p.tile_count = reinterpret_cast<uint32_t *>(ws + o_tc);
        p.chunk_bytes = reinterpret_cast<unsigned long long *>(ws + o_cb);
        p.chunk_count = reinterpret_cast<uint32_t *>(ws + o_cc);
        p.src_ptr = reinterpret_cast<unsigned long long *>(ws + o_src);
        p.tile_first = reinterpret_cast<uint32_t *>(ws + o_tf);
        p.tile_first_n = (uint32_t)(gather_tiles + 2);
        p.out_data = od;
        p.out_index = reinterpret_cast<uint4 *>(oi);
        const uint4 *res = rp.out_index;
        CU(cudaStreamWaitEvent(s, e->ev_h2d[c & 1], 0));
        if (c >= 2) CU(cudaStreamWaitEvent(s, e->ev_d2h[c & 1], 0)); // output buffer c & 1 drained by partition c - 2's D2H
        CU(cudaEventRecord(tev.ev[T_KER + 2 * (c & 1)], s));
        k_scan_part_enter<<<1, 1, 0, s>>>(sp.stop, reinterpret_cast<const unsigned long long *>(ws + o_gstop));
        CU(cudaMemsetAsync(sp.ctl, 0, sizeof(Ctl), s));
        CU(cudaMemsetAsync(sp.totals, 0, 8ull * (3 * n_cls + 1), s));
        k_scan_classify<<<(N + 255) / 256, 256, 0, s>>>(sp);
        k_route_hash<true><<<n_blocks, kRouteThreads, 0, s>>>(rp);
        k_route_scan<<<n_cls, 1024, 0, s>>>(rp);
        k_route_starts<<<1, 256, 0, s>>>(rp, reinterpret_cast<unsigned long long *>(ws + o_rtot));
        k_route_scatter<<<n_blocks, kRouteThreads, 0, s>>>(rp);
        k_scan_plan<<<1, 256, 0, s>>>(sp);
        k_scan_res_tiles<<<(uint32_t)res_tiles, kResolveThreads, 0, s>>>(p, res);
        k_scan_tiles<<<(uint32_t)res_chunks, 1024, 0, s>>>(p);
        k_scan_chunks<<<1, 1024, 0, s>>>(p);
        k_emit<<<(uint32_t)res_tiles, kResolveThreads, 0, s>>>(p, res);
        k_flush_table<<<(n_cls + 1 + 127) / 128, 128, 0, s>>>(p, res);
        launches += 13;
        if (gather_tiles) {
            if (((uintptr_t)od & 31) == 0) k_gather32<false, false, false, true><<<(uint32_t)gather_tiles, kGatherThreads, 0, s>>>(p);
            else k_gather<<<(uint32_t)gather_tiles, kGatherThreads, 0, s>>>(p);
            launches++;
        }
        k_scan_rebase_stream<<<(N + 255) / 256, 256, 0, s>>>(p, reinterpret_cast<const unsigned long long *>(ws + o_run)); // after the gather
        k_scan_part_leave<<<1, 256, 0, s>>>(p.mem_table, n_ranges, sp.stop, reinterpret_cast<unsigned long long *>(ws + o_gstop), q.first_ordinal,
                                            reinterpret_cast<unsigned long long *>(ws + o_run),
                                            reinterpret_cast<unsigned long long *>(e->pin_dev + (c & 1) * hdr_stride));
        launches += 2;
        CU(cudaGetLastError());
        CU(cudaEventRecord(tev.ev[T_KER + 2 * (c & 1) + 1], s));
        CU(cudaEventRecord(e->ev_comp[c & 1], s));
        return DBEEL_OK;
    };

    uint64_t out_data = 0, out_items = 0, gstop = ~0ull;
    uint32_t done = 0; // partitions whose output has been published
    std::vector<StreamPump::OutPiece> pieces;
    rc = enqueue_h2d(0);
    if (!rc && np > 1) rc = enqueue_h2d(1);
    if (!rc) rc = enqueue_kernels(0);
    for (uint32_t c = 0; c < np && !rc; c++) {
        if (c + 1 < np && (rc = enqueue_kernels(c + 1))) break;
        ce = cudaEventSynchronize(e->ev_comp[c & 1]);
        if (ce != cudaSuccess) { rc = fail(e, DBEEL_ERR_CUDA, "scan partition kernels", ce); break; }
        pump->release_input(c); // the kernels have read device buffer c & 1, which the H2D out of ring slot c mod R filled
        st.ms_h2d += stage_ms(T_H2D, c & 1);
        st.ms_total += stage_ms(T_KER, c & 1);
        if (c >= 2) { // partition c - 2's D2H (the kernels of c waited for it)
            CU(cudaEventSynchronize(tev.ev[T_D2H + 2 * (c & 1) + 1]));
            st.ms_d2h += stage_ms(T_D2H, c & 1);
        }
        const unsigned long long *hdr = reinterpret_cast<const unsigned long long *>(e->pin + (c & 1) * hdr_stride);
        const ScanPieceRow *rows = reinterpret_cast<const ScanPieceRow *>(hdr + 1);
        gstop = hdr[0];
        uint64_t dlen = 0, items = 0;
        for (uint32_t r = 0; r < n_ranges; r++) { dlen += rows[r].data_len; items += rows[r].items; }
        if ((rc = pump->wait_out_slot(c))) { fail(e, rc, "scan write callback failed"); break; }
        uint8_t *oslot = e->ring_out + (uint64_t)(c % R) * max_out, *oindex = oslot + align_up(dlen + 16, kAlign);
        const ScanPart &q = plan.parts[c];
        CU(cudaStreamWaitEvent(e->s_d2h, e->ev_comp[c & 1], 0));
        CU(cudaEventRecord(tev.ev[T_D2H + 2 * (c & 1)], e->s_d2h));
        if (dlen) CU(cudaMemcpyAsync(oslot, sout[c & 1], dlen, cudaMemcpyDeviceToHost, e->s_d2h));
        if (items) CU(cudaMemcpyAsync(oindex, sout[c & 1] + align_up(q.data_bytes + 16, kAlign), 16 * items, cudaMemcpyDeviceToHost, e->s_d2h));
        CU(cudaEventRecord(tev.ev[T_D2H + 2 * (c & 1) + 1], e->s_d2h));
        CU(cudaEventRecord(ev_out.ev[c], e->s_d2h));
        CU(cudaEventRecord(e->ev_d2h[c & 1], e->s_d2h));
        pieces.clear();
        for (uint32_t r = 0; r < n_ranges; r++) {
            const ScanPieceRow &w = rows[r];
            if (w.data_len) pieces.push_back(StreamPump::OutPiece{oslot + w.data_at, w.data_len, r, DBEEL_STREAM_DATA, w.stream_data_off});
            if (w.items) pieces.push_back(StreamPump::OutPiece{oindex + 16 * w.items_at, 16 * w.items, r, DBEEL_STREAM_INDEX, 16 * w.stream_items_off});
            per_range[r].data_len += w.data_len;
            per_range[r].items += w.items;
        }
        pump->publish_pieces(c, pieces);
        done = c + 1;
        out_data += dlen;
        out_items += items;
        if (gstop != ~0ull) { // the later partitions select nothing: read and write no more of them
            pump->end_at(c + 1);
            break;
        }
        if (c + 2 < np && (rc = enqueue_h2d(c + 2))) break;
    }
    cudaStreamSynchronize(s);
    cudaStreamSynchronize(e->s_h2d);
    cudaStreamSynchronize(e->s_d2h);
    if (rc) {
        pump->abort(rc); // its threads are joined when it goes out of scope
        return rc;
    }
    const int frc = pump->finish(); // every published piece has gone through the write callback
    if (frc) return fail(e, frc, "scan write callback failed");
    for (uint32_t c = done >= 2 ? done - 2 : 0; c < done; c++) st.ms_d2h += stage_ms(T_D2H, c & 1); // the last two D2H
    if (gstop != ~0ull) { // a DECODE stop (or a READ stop the device saw first) in front of the plan's
        const uint64_t o = gstop >> 2;
        uint32_t t = 0;
        while (t + 1 < nt && tbase[t + 1] <= o) t++;
        *stop = dbeel_scan_stop{(int32_t)t, (uint32_t)(gstop & 3), o - tbase[t]};
        st.entries_valid = o;
    }
    for (uint32_t r = 0; r < n_ranges; r++) per_range[r].index_len = 16 * per_range[r].items;
    st.entries_out = out_items;
    st.output_bytes = out_data + 16 * out_items;
    st.kernel_launches = launches;
    st.partitions = done;
    return DBEEL_OK;
}

} // namespace

// ------------------------------------------------------------------------------------ C ABI

extern "C" {

int dbeel_abi_version(void) { return DBEEL_ABI_VERSION; }

int dbeel_engine_create(int device, dbeel_engine **out) {
    if (!out) return DBEEL_ERR_INVALID_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return DBEEL_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return DBEEL_ERR_CUDA;
    if (prop.major != 10) return DBEEL_ERR_NO_DEVICE; // sm_100a SASS only: no fallback path
    if (cudaSetDevice(device) != cudaSuccess) return DBEEL_ERR_CUDA;
    dbeel_engine *e = new (std::nothrow) dbeel_engine();
    if (!e) return DBEEL_ERR_NOMEM;
    e->device = device;
    e->sm_count = prop.multiProcessorCount;
    if (const char *v = getenv("DBEEL_MERGE")) e->merge_variant = atoi(v);
    if (const char *v = getenv("DBEEL_PIPELINE")) e->pipeline = atoi(v);
    if (const char *v = getenv("DBEEL_PIPELINE_MIN_KB")) e->pipeline_min_bytes = (uint64_t)(atoi(v) > 0 ? atoi(v) : 1) << 10;
    if (const char *v = getenv("DBEEL_PARTITION_KB")) e->partition_bytes = (uint64_t)(atoi(v) > 0 ? atoi(v) : 1) << 10;
    if (const char *v = getenv("DBEEL_PARTITION_TAPER")) e->partition_taper = atoi(v) != 0;
    if (const char *v = getenv("DBEEL_STREAM_RING")) e->stream_ring = std::max(2, atoi(v));
    if (const char *v = getenv("DBEEL_PARTITION_MB")) e->partition_bytes = (uint64_t)(atoi(v) > 0 ? atoi(v) : 128) << 20;
    if (cudaFuncSetAttribute(k_merge_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * kMergeBufRecs * sizeof(Rec))) != cudaSuccess ||
        cudaFuncSetAttribute(k_gather_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGtSmem) != cudaSuccess) {
        dbeel_engine_destroy(e);
        return DBEEL_ERR_CUDA;
    }
    if (const char *v = getenv("DBEEL_NARROW")) e->narrow_loads = atoi(v);
    if (const char *v = getenv("DBEEL_GATHER")) e->gather_variant = atoi(v);
    if (const char *v = getenv("DBEEL_BLOOM_EXTRACT")) e->bloom_in_extract = atoi(v);
    if (const char *v = getenv("DBEEL_BLOOM_SIDE")) e->bloom_side = atoi(v);
    if (const char *v = getenv("DBEEL_FUSED_EMIT")) e->fused_emit = atoi(v);
    if (const char *v = getenv("DBEEL_FUSED_FINAL")) e->fused_final = atoi(v);
    if (const char *v = getenv("DBEEL_EXTRACT_PERSIST")) e->extract_persist = atoi(v);
    if (const char *v = getenv("DBEEL_PDL")) e->pdl = atoi(v);
    if (const char *v = getenv("DBEEL_STAGE_EVENTS")) e->stage_events = atoi(v);
    {
        int nb_t = 0, nb_f = 0;
        if (cudaFuncSetAttribute(k_merge_final<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFinSmem) == cudaSuccess &&
            cudaFuncSetAttribute(k_merge_final<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFinSmem) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_t, k_merge_final<true>, kFinThreads, kFinSmem) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_f, k_merge_final<false>, kFinThreads, kFinSmem) == cudaSuccess) {
            e->fin_ctas_per_sm = std::min(std::min(nb_t, nb_f), (int)DBEEL_FIN_CTAS);
        } else {
            cudaGetLastError();
            e->fin_ctas_per_sm = 0; // the five-kernel path
        }
        if (const char *v = getenv("DBEEL_FIN_CTAS_RT")) e->fin_ctas_per_sm = std::min(e->fin_ctas_per_sm, std::max(1, atoi(v)));
    }
    if (cudaStreamCreateWithFlags(&e->s_side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess) {
        dbeel_engine_destroy(e);
        return DBEEL_ERR_CUDA;
    }
    if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) { delete e; return DBEEL_ERR_CUDA; }
    for (int i = 0; i < EV_COUNT; i++)
        if (cudaEventCreate(&e->ev[i]) != cudaSuccess) { dbeel_engine_destroy(e); return DBEEL_ERR_CUDA; }
    *out = e;
    return DBEEL_OK;
}

void *dbeel_engine_stream(dbeel_engine *e) { return e ? static_cast<void *>(e->stream) : nullptr; }

void dbeel_engine_destroy(dbeel_engine *e) {
    if (!e) return;
    if (e->worker.joinable()) e->worker.join();
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (int i = 0; i < EV_COUNT; i++)
        if (e->ev[i]) cudaEventDestroy(e->ev[i]);
    if (e->ws) cudaFree(e->ws);
    if (e->stage_in) cudaFree(e->stage_in);
    if (e->stage_out) cudaFree(e->stage_out);
    if (e->stage_in2) cudaFree(e->stage_in2);
    if (e->stage_out2) cudaFree(e->stage_out2);
    if (e->bloom_dev) cudaFree(e->bloom_dev);
    if (e->wal_ws) cudaFree(e->wal_ws);
    if (e->route_ws) cudaFree(e->route_ws);
    for (int i = 0; i < 2; i++) {
        if (e->ev_h2d[i]) cudaEventDestroy(e->ev_h2d[i]);
        if (e->ev_comp[i]) cudaEventDestroy(e->ev_comp[i]);
        if (e->ev_d2h[i]) cudaEventDestroy(e->ev_d2h[i]);
    }
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    if (e->s_side) cudaStreamDestroy(e->s_side);
    if (e->s_h2d) cudaStreamDestroy(e->s_h2d);
    if (e->s_d2h) cudaStreamDestroy(e->s_d2h);
    if (e->pin) cudaFreeHost(e->pin);
    if (e->ring_in) cudaFreeHost(e->ring_in);
    if (e->ring_out) cudaFreeHost(e->ring_out);
    if (e->pin_index) cudaFreeHost(e->pin_index);
    if (e->pin_bloom) cudaFreeHost(e->pin_bloom);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

// Bloom::compute_bitmap_size (bloomfilter 1.0.12): ceil(n * ln(p) / (-8 * ln2^2)) in f64
uint64_t dbeel_bloom_bitmap_bytes(uint64_t items, double fp) {
    const double ln2 = 0.693147180559945309417232121458176568; // core::f64::consts::LN_2
    return (uint64_t)ceil((double)items * log(fp) / (-8.0 * (ln2 * ln2)));
}

// Bloom::optimal_k_num: max(1, ceil(m / n * ln(2.0)))
uint32_t dbeel_bloom_k_num(uint64_t bitmap_bits, uint64_t items) {
    uint32_t k = (uint32_t)ceil((double)bitmap_bits / (double)items * log(2.0));
    return k < 1 ? 1 : k;
}

uint64_t dbeel_bloom_file_size(uint64_t items, double fp) {
    uint64_t bits = dbeel_bloom_bitmap_bytes(items, fp) * 8;
    return 8 + 4 * ((bits + 31) / 32) + 8 + 8 + 4 + 144;
}

int dbeel_compact_bound(const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts, uint64_t *data_cap,
                        uint64_t *index_cap, uint64_t *bloom_cap) {
    if (n_runs && !runs) return DBEEL_ERR_INVALID_ARG;
    dbeel_compact_opts o;
    default_opts(&o);
    if (opts) o = *opts;
    if (!(o.bloom_fp > 0.0 && o.bloom_fp < 1.0)) return DBEEL_ERR_INVALID_ARG;
    JobShape sh;
    shape_of(runs, n_runs, &o, false, &sh);
    if (data_cap) *data_cap = sh.data_total;
    if (index_cap) *index_cap = sh.n_total * 16;
    if (bloom_cap) *bloom_cap = sh.bloom_file;
    return DBEEL_OK;
}

// While an asynchronous job runs, the worker thread owns e->err and e->stats: a refused call returns the code without
// touching either (BUSY is an expected answer for a reactor that polls).
#define REFUSE_WHILE_ASYNC(e)                                                                  \
    if ((e) && (e)->async_state.load(std::memory_order_acquire) != 0) return DBEEL_ERR_BUSY

int dbeel_compact(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts,
                  dbeel_out *out) {
    REFUSE_WHILE_ASYNC(e);
    return entry(e, runs, n_runs, opts, out, false, false);
}

int dbeel_compact_stream(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts,
                         const dbeel_stream_io *io, dbeel_out *out) {
    return stream_entry(e, runs, n_runs, opts, io, out);
}

int dbeel_compact_device(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts,
                         dbeel_out *out) {
    REFUSE_WHILE_ASYNC(e);
    return entry(e, runs, n_runs, opts, out, false, true);
}

int dbeel_compact_submit(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts,
                         dbeel_out *out) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!out || (n_runs && !runs)) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    int expected = 0;
    if (!e->async_state.compare_exchange_strong(expected, 1)) return DBEEL_ERR_BUSY; // the worker owns e->err
    if (e->worker.joinable()) e->worker.join();
    e->async_runs.assign(runs, runs + n_runs); // the descriptors are copied; the buffers they point to are not
    default_opts(&e->async_opts);
    if (opts) e->async_opts = *opts;
    if (e->async_opts.bloom_seed) {
        memcpy(e->async_seed, e->async_opts.bloom_seed, 32);
        e->async_opts.bloom_seed = e->async_seed;
    }
    e->worker = std::thread([e, out]() {
        e->async_status = entry(e, e->async_runs.data(), (uint32_t)e->async_runs.size(), &e->async_opts, out, false, false);
        e->async_state.store(2, std::memory_order_release);
    });
    return DBEEL_OK;
}

int dbeel_poll(dbeel_engine *e, int *status) {
    if (!e) return 0;
    if (e->async_state.load(std::memory_order_acquire) != 2) return 0;
    if (e->worker.joinable()) e->worker.join();
    if (status) *status = e->async_status;
    e->async_state.store(0, std::memory_order_release);
    return 1;
}

int dbeel_wait(dbeel_engine *e) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (e->async_state.load(std::memory_order_acquire) == 0) return fail(e, DBEEL_ERR_INVALID_ARG, "no job in flight");
    if (e->worker.joinable()) e->worker.join();
    const int st = e->async_status;
    e->async_state.store(0, std::memory_order_release);
    return st;
}

int dbeel_flush(dbeel_engine *e, const dbeel_run *batch, dbeel_out *out) {
    REFUSE_WHILE_ASYNC(e);
    return entry(e, batch, batch ? 1 : 0, nullptr, out, true, false);
}

static int flush_many_entry(dbeel_engine *e, const dbeel_run *batches, uint32_t n, dbeel_out *out, dbeel_flush_table *table,
                            bool device, bool sparse = false, uint64_t payload_bound = 0) {
    if (!e) return DBEEL_ERR_INVALID_ARG;
    if (!out || !table || (n && !batches)) return fail(e, DBEEL_ERR_INVALID_ARG, "null argument");
    if (e->busy) return fail(e, DBEEL_ERR_BUSY, "engine busy");
    BusyGuard g(e);
    e->err.clear();
    dbeel_compact_opts o;
    default_opts(&o);
    cudaError_t ce = cudaSetDevice(e->device);
    if (ce != cudaSuccess) return fail(e, DBEEL_ERR_CUDA, "cudaSetDevice", ce);
    for (uint32_t i = 0; i < n; i++) table[i] = dbeel_flush_table{0, 0, 0, 0, 0};
    JobExtra ex;
    ex.flush_table = table;
    if (sparse) { // the batches' index records point into shared .data (routed streams): no running-offset check
        ex.sparse_offsets = true;
        ex.data_bytes = payload_bound;
    }
    if (device) return run_job_device(e, batches, n, &o, true, out, true, &ex);
    // host buffers: stage everything down, run, bring the concatenated SSTables back
    uint64_t in_need = 0, dsum = 0, isum = 0;
    for (uint32_t r = 0; r < n; r++) {
        if ((batches[r].data_len && !batches[r].data) || (batches[r].index_len && !batches[r].index))
            return fail(e, DBEEL_ERR_INVALID_ARG, "null batch buffer");
        in_need += align_up(batches[r].data_len + 32, kAlign) + align_up(batches[r].index_len + 16, kAlign);
        dsum += batches[r].data_len;
        isum += batches[r].index_len / DBEEL_INDEX_ENTRY_SIZE * 16;
    }
    if (out->data_cap < dsum || out->index_cap < isum) return fail(e, DBEEL_ERR_CAPACITY, "output buffer too small");
    int rc = ensure_device(e, &e->stage_in, &e->stage_in_cap, in_need);
    if (!rc) rc = ensure_device(e, &e->stage_out, &e->stage_out_cap, align_up(dsum + 16, kAlign) + align_up(isum + 16, kAlign));
    if (rc) return rc;
    std::vector<dbeel_run> dr(n);
    uint64_t pos = 0;
    for (uint32_t r = 0; r < n; r++) {
        dr[r] = dbeel_run{e->stage_in + pos, batches[r].data_len, nullptr, batches[r].index_len};
        if (batches[r].data_len) CU(cudaMemcpyAsync(e->stage_in + pos, batches[r].data, batches[r].data_len, cudaMemcpyHostToDevice, e->stream));
        pos += align_up(batches[r].data_len + 32, kAlign);
        dr[r].index = e->stage_in + pos;
        if (batches[r].index_len) CU(cudaMemcpyAsync(e->stage_in + pos, batches[r].index, batches[r].index_len, cudaMemcpyHostToDevice, e->stream));
        pos += align_up(batches[r].index_len + 16, kAlign);
    }
    dbeel_out dout = *out;
    dout.data = e->stage_out;
    dout.index = e->stage_out + align_up(dsum + 16, kAlign);
    dout.bloom = nullptr;
    dout.bloom_cap = 0;
    rc = run_job_device(e, dr.data(), n, &o, true, &dout, true, &ex);
    if (rc) return rc;
    if (dout.data_len) CU(cudaMemcpyAsync(out->data, dout.data, dout.data_len, cudaMemcpyDeviceToHost, e->stream));
    if (dout.index_len) CU(cudaMemcpyAsync(out->index, dout.index, dout.index_len, cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    out->data_len = dout.data_len;
    out->index_len = dout.index_len;
    out->bloom_len = 0;
    out->items_written = dout.items_written;
    return DBEEL_OK;
}

int dbeel_flush_many(dbeel_engine *e, const dbeel_run *batches, uint32_t n_batches, dbeel_out *out, dbeel_flush_table *table) {
    REFUSE_WHILE_ASYNC(e);
    return flush_many_entry(e, batches, n_batches, out, table, false);
}

int dbeel_flush_many_device(dbeel_engine *e, const dbeel_run *batches, uint32_t n_batches, dbeel_out *out,
                            dbeel_flush_table *table) {
    REFUSE_WHILE_ASYNC(e);
    return flush_many_entry(e, batches, n_batches, out, table, true);
}

int dbeel_flush_many_sparse_device(dbeel_engine *e, const dbeel_run *batches, uint32_t n_batches, uint64_t payload_bound,
                                   dbeel_out *out, dbeel_flush_table *table) {
    REFUSE_WHILE_ASYNC(e);
    return flush_many_entry(e, batches, n_batches, out, table, true, true, payload_bound);
}

int dbeel_route_device(dbeel_engine *e, const dbeel_run *batch, const uint32_t *ring_hashes, uint32_t n_shards, void *out_index,
                       uint64_t out_index_cap, uint32_t *shard_of, void *out_key_hash64, uint64_t *counts, uint64_t *payload_bytes) {
    REFUSE_WHILE_ASYNC(e);
    return route_entry(e, batch, ring_hashes, n_shards, out_index, out_index_cap, shard_of, out_key_hash64, counts, payload_bytes);
}

int dbeel_memtable_cuts_device(dbeel_engine *e, const void *key_hash64, const uint64_t *stream_starts, uint32_t n_streams,
                               uint32_t capacity, uint32_t *cuts, uint32_t *cut_starts, uint32_t max_cuts_total) {
    REFUSE_WHILE_ASYNC(e);
    return cuts_entry(e, key_hash64, stream_starts, n_streams, capacity, cuts, cut_starts, max_cuts_total);
}

int dbeel_flush_device(dbeel_engine *e, const dbeel_run *batch, dbeel_out *out) {
    REFUSE_WHILE_ASYNC(e);
    return entry(e, batch, batch ? 1 : 0, nullptr, out, true, true);
}

int dbeel_get_many(dbeel_engine *e, const dbeel_table *tables, uint32_t n_tables, const void *keys, const uint64_t *key_offsets,
                   uint64_t n_keys, uint32_t mode, dbeel_lookup_result *results) {
    REFUSE_WHILE_ASYNC(e);
    return lookup_entry(e, tables, n_tables, keys, key_offsets, n_keys, mode, results, false);
}

int dbeel_get_many_device(dbeel_engine *e, const dbeel_table *tables, uint32_t n_tables, const void *keys,
                          const uint64_t *key_offsets, uint64_t n_keys, uint32_t mode, dbeel_lookup_result *results) {
    REFUSE_WHILE_ASYNC(e);
    return lookup_entry(e, tables, n_tables, keys, key_offsets, n_keys, mode, results, true);
}

int dbeel_compact_many_bound(const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size, double bloom_fp, uint64_t *data_cap,
                             uint64_t *index_cap, uint64_t *bloom_cap) {
    if (n_jobs && !jobs) return DBEEL_ERR_INVALID_ARG;
    JobShapes js;
    int rc = job_shapes(nullptr, jobs, n_jobs, bloom_min_size, bloom_fp, &js);
    if (rc) return rc;
    if (data_cap) *data_cap = js.data;
    if (index_cap) *index_cap = js.index;
    if (bloom_cap) *bloom_cap = js.bloom;
    return DBEEL_OK;
}

int dbeel_compact_many(dbeel_engine *e, const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size, double bloom_fp,
                       dbeel_out *out, dbeel_job_result *results) {
    REFUSE_WHILE_ASYNC(e);
    return compact_many_entry(e, jobs, n_jobs, bloom_min_size, bloom_fp, out, results, false);
}

int dbeel_compact_many_device(dbeel_engine *e, const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size, double bloom_fp,
                              dbeel_out *out, dbeel_job_result *results) {
    REFUSE_WHILE_ASYNC(e);
    return compact_many_entry(e, jobs, n_jobs, bloom_min_size, bloom_fp, out, results, true);
}

int dbeel_wal_flush(dbeel_engine *e, const void *wal, uint64_t wal_len, uint32_t capacity, dbeel_out *out) {
    REFUSE_WHILE_ASYNC(e);
    return wal_flush_entry(e, wal, wal_len, capacity, out, false);
}

int dbeel_wal_flush_device(dbeel_engine *e, const void *wal, uint64_t wal_len, uint32_t capacity, dbeel_out *out) {
    REFUSE_WHILE_ASYNC(e);
    return wal_flush_entry(e, wal, wal_len, capacity, out, true);
}

int dbeel_scan_ranges(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges, uint32_t n_ranges,
                      uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range, dbeel_scan_stop *stop) {
    REFUSE_WHILE_ASYNC(e);
    return scan_entry(e, tables, n_tables, ranges, n_ranges, mode, out, per_range, stop, false);
}

int dbeel_scan_ranges_device(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges,
                             uint32_t n_ranges, uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range, dbeel_scan_stop *stop) {
    REFUSE_WHILE_ASYNC(e);
    return scan_entry(e, tables, n_tables, ranges, n_ranges, mode, out, per_range, stop, true);
}

int dbeel_scan_ranges_stream(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges,
                             uint32_t n_ranges, uint32_t mode, const dbeel_scan_io *io, uint64_t partition_bytes,
                             dbeel_flush_table *per_range, dbeel_scan_stop *stop) {
    REFUSE_WHILE_ASYNC(e);
    return scan_stream_entry(e, tables, n_tables, ranges, n_ranges, mode, io, partition_bytes, per_range, stop);
}

void *dbeel_host_alloc(uint64_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void dbeel_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// Stats and the error text of an asynchronous job belong to its worker thread until dbeel_poll / dbeel_wait has joined it.
int dbeel_last_stats(const dbeel_engine *e, dbeel_stats *out) {
    if (!e || !out) return DBEEL_ERR_INVALID_ARG;
    if (e->async_state.load(std::memory_order_acquire) != 0) return DBEEL_ERR_BUSY;
    *out = e->stats;
    return DBEEL_OK;
}

const char *dbeel_last_error(const dbeel_engine *e) {
    if (!e) return "null engine";
    if (e->async_state.load(std::memory_order_acquire) != 0) return "an asynchronous job is in flight";
    return e->err.c_str();
}

const char *dbeel_strerror(int code) {
    switch (code) {
    case DBEEL_OK: return "ok";
    case DBEEL_ERR_INVALID_ARG: return "invalid argument";
    case DBEEL_ERR_CAPACITY: return "output buffer too small";
    case DBEEL_ERR_ITEM_TOO_LARGE: return "item too large";
    case DBEEL_ERR_CUDA: return "CUDA error";
    case DBEEL_ERR_NOMEM: return "out of memory";
    case DBEEL_ERR_TOO_MANY_RUNS: return "too many runs";
    case DBEEL_ERR_TOO_MANY_ENTRIES: return "too many entries";
    case DBEEL_ERR_UNSORTED_RUN: return "input run not strictly ascending";
    case DBEEL_ERR_NO_DEVICE: return "no sm_100 CUDA device";
    case DBEEL_ERR_BUSY: return "engine busy";
    case DBEEL_ERR_BAD_BLOOM: return "malformed .bloom file";
    case DBEEL_ERR_TREE_FULL: return "memtable capacity reached";
    default: return "unknown error";
    }
}

} // extern "C"
