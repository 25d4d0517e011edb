/*
 * dbeel_compact.h -- C ABI of the B200 compaction engine (libdbeel_compact.so).
 *
 * This is the drop-in boundary for ONE hot path of tontinton/dbeel's storage engine: the
 * merge core of LSMTree::compact, the memtable flush that feeds level 0, and the
 * bloom / per-entry index build on the output run.  Everything else (file open/create,
 * the CompactionAction journal, renames, the sstables swap, the page cache, the WAL)
 * stays with the caller.  The library never touches the filesystem.
 *
 * Reference interfaces replaced (paths under /root/reference):
 *
 *   dbeel_compact*      <- the body of LSMTree::compact between opening the inputs and
 *                          writing the bloom file: src/storage_engine/lsm_tree.rs:1002-1076
 *                          (BinaryHeap<CompactionItem> merge :52-71,:1038-1066,
 *                          read_next_entry :1158-1170, EntryWriter::write/close
 *                          src/storage_engine/entry_writer.rs:71-160, Bloom::set + dump
 *                          lsm_tree.rs:1026-1034,:1049-1051,:1070-1076)
 *   dbeel_flush*        <- RedBlackTree::set semantics (rbtree_arena/src/lib.rs:497-534) +
 *                          LSMTree::flush_memtable_to_disk (lsm_tree.rs:925-946)
 *   dbeel_flush_many*   <- the same for many memtables at once (several collections / shards, or a backlog)
 *   dbeel_compact_many* <- compact_tree's loop over the groups its picker produced: one LSMTree::compact per
 *                          group (src/tasks/compaction.rs:82-101), all groups in one launch sequence
 *   dbeel_compact_stream<- the same merge core with the reference's file edge around it: the DmaStreamReaders of the
 *                          inputs (lsm_tree.rs:984-991) and EntryWriter's DMA files (entry_writer.rs:30-69) become
 *                          read / write callbacks feeding a pinned ring                 ["next" row N3]
 *   dbeel_get_many*     <- the SSTable loop of LSMTree::get_entry: Bloom::check + binary_search
 *                          (lsm_tree.rs:605-670, 686-719) for a batch of keys        ["next" row N2]
 *   dbeel_wal_flush*    <- read_memtable_from_wal_file + the recovery flush of open_or_create_ex
 *                          (lsm_tree.rs:552-574, 478-513)                            ["next" row N4]
 *   dbeel_bloom_*       <- Bloom::new_for_fp_rate sizing (lsm_tree.rs:1028-1031)
 *   error codes         <- src/error.rs:8-74 (only the variants this path can raise)
 *
 * Byte formats are the reference's own (bincode fixint little-endian, mod.rs:45-73):
 *   .data  record = klen:u64 | key | dlen:u64 | data | ts:i128      (dlen == 0: tombstone)
 *   .index record = offset:u64 | key_size:u32 (=8+klen) | full_size:u32   (16 bytes)
 *   .bloom        = bincode(bloomfilter::Bloom) -- see DESIGN.md for the field order
 *
 * Plain pointers and sizes only; no C++ or torch types cross this boundary.
 */
#ifndef DBEEL_COMPACT_H
#define DBEEL_COMPACT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBEEL_ABI_VERSION 1

/* status codes (0 = ok).  No exception or panic ever crosses the ABI. */
enum {
    DBEEL_OK = 0,
    DBEEL_ERR_INVALID_ARG = 1,     /* null pointer, misaligned device buffer, bad option    */
    DBEEL_ERR_CAPACITY = 2,        /* an output buffer is smaller than dbeel_compact_bound  */
    DBEEL_ERR_ITEM_TOO_LARGE = 3,  /* Error::ItemTooLarge, entry_writer.rs:72-74            */
    DBEEL_ERR_CUDA = 4,            /* a CUDA call failed; dbeel_last_error() has the text   */
    DBEEL_ERR_NOMEM = 5,           /* device or pinned-host allocation failed               */
    DBEEL_ERR_TOO_MANY_RUNS = 6,   /* more than DBEEL_MAX_RUNS inputs                       */
    DBEEL_ERR_TOO_MANY_ENTRIES = 7,/* more than 2^32-2 input entries in one job             */
    DBEEL_ERR_UNSORTED_RUN = 8,    /* an input run violates "keys strictly ascending"       */
    DBEEL_ERR_NO_DEVICE = 9,       /* no CUDA device / not an sm_100 part                   */
    DBEEL_ERR_BUSY = 10,           /* engine already has a job in flight                    */
    DBEEL_ERR_BAD_BLOOM = 11,      /* a .bloom file is not a bincode bloomfilter::Bloom      */
    DBEEL_ERR_TREE_FULL = 12       /* rbtree_arena ReachedCapacity (lib.rs:458-461)          */
};

#define DBEEL_MAX_RUNS 1024u
#define DBEEL_INDEX_ENTRY_SIZE 16u            /* mod.rs:33 */
#define DBEEL_DEFAULT_BLOOM_MIN_SIZE 1048576u /* mod.rs:19 */
#define DBEEL_DEFAULT_BLOOM_FP 0.01           /* lsm_tree.rs:48 */
#define DBEEL_DEFAULT_TREE_CAPACITY 8192u     /* mod.rs:18 */

/* One input SSTable: the bytes of its .data and .index files.
 * For the *_device entry points both are device pointers; `index` must be aligned to 16 bytes, `data` may start anywhere
 * (the SSTables dbeel_flush_many / dbeel_compact_many leave back to back in one output stream are valid inputs as they lie). */
typedef struct dbeel_run {
    const void *data;
    uint64_t data_len;
    const void *index;
    uint64_t index_len; /* entries = index_len / 16 (lsm_tree.rs:978-979); a ragged tail is ignored */
} dbeel_run;

/* Output SSTable buffers, owned by the caller.  *_cap in, *_len out. */
typedef struct dbeel_out {
    void *data;
    uint64_t data_cap, data_len;
    void *index;
    uint64_t index_cap, index_len;
    void *bloom;         /* may be NULL when bloom_cap == 0 (no bloom will be produced) */
    uint64_t bloom_cap, bloom_len; /* bloom_len == 0: no .bloom file (lsm_tree.rs:1026-1034) */
    uint64_t items_written;        /* lsm_tree.rs:1053 */
} dbeel_out;

#define DBEEL_FLAG_VERIFY_SORTED 0x1u /* full adjacent-key check of every input run */
/* Decode the input runs exactly like the reference's sequential reader (read_next_entry, lsm_tree.rs:1158-1170):
 *   - an index record's `offset` and `key_size` are IGNORED -- the entry is the next full_size bytes of the .data stream
 *     and its key length is the bincode length prefix found there (the output .index carries the recomputed values,
 *     entry_writer.rs:76-86);
 *   - an i128 timestamp outside `time`'s +-9999-year range fails the decode (utils/timestamp_nanos.rs:15-24) and, like
 *     every decode error, ends that run (lsm_tree.rs:1014,1063).
 * Without the flag the engine is stricter about the index (a wrong offset / key_size ends the run) and does not range-
 * check timestamps; on files the reference's own writer produced both modes give byte-identical output.
 * dbeel_compact / dbeel_compact_device / dbeel_compact_submit only. */
#define DBEEL_FLAG_REFERENCE_READER 0x2u

typedef struct dbeel_compact_opts {
    int32_t keep_tombstones;   /* LSMTree::compact's third argument (lsm_tree.rs:954)      */
    uint32_t flags;            /* DBEEL_FLAG_*                                             */
    uint64_t bloom_min_size;   /* --sstable-bloom-min-size, strict '>' (lsm_tree.rs:1027)  */
    double bloom_fp;           /* BLOOM_MAX_ALLOWED_ERROR                                  */
    const uint8_t *bloom_seed; /* 32 bytes (host memory), or NULL = random like getrandom  */
} dbeel_compact_opts;

/* What the last job did.  Times are CUDA-event milliseconds on the engine's stream. */
typedef struct dbeel_stats {
    uint64_t input_bytes;      /* sum(len(.data)+len(.index))                              */
    uint64_t output_bytes;     /* len(out.data)+len(out.index)+len(out.bloom)              */
    uint64_t entries_in;       /* sum(index_len/16)                                        */
    uint64_t entries_valid;    /* after run truncation at the first undecodable record     */
    uint64_t entries_out;      /* items_written                                            */
    uint32_t runs_truncated;   /* runs that ended early (lsm_tree.rs:1014,1063)            */
    uint32_t key_prefix_len;   /* common key prefix skipped by the comparison window        */
    uint32_t merge_passes;
    uint32_t kernel_launches;  /* kernels launched by this job                             */
    float ms_total;            /* first kernel .. last kernel (device-resident part)       */
    float ms_extract;          /* validate + key-window extraction                         */
    float ms_merge;            /* all merge passes                                         */
    float ms_resolve;          /* winner / tombstone resolution + offsets scan + .index    */
    float ms_gather;           /* .data gather + bloom (the roofline kernel)               */
    float ms_h2d, ms_d2h;      /* host entry points only                                   */
    uint64_t gather_bytes;     /* algorithmic bytes of the gather kernel (read + written)  */
    uint32_t partitions;       /* host entry points: key-range partitions pipelined (1 = single shot) */
    uint32_t index_repaired;   /* DBEEL_FLAG_REFERENCE_READER: 1 = an input index disagreed with its .data and the job ran on the canonical index */
} dbeel_stats;

typedef struct dbeel_engine dbeel_engine;

/* One engine per calling thread / shard, bound to one GPU and one stream. */
int dbeel_engine_create(int device, dbeel_engine **out);
void dbeel_engine_destroy(dbeel_engine *e);
/* The engine's CUDA stream (a cudaStream_t): every kernel of its jobs is launched there.  For callers that want to record
 * their own events around jobs or order other work against them.  Several engines on one GPU run their jobs concurrently. */
void *dbeel_engine_stream(dbeel_engine *e);

/* Host placement.  dbeel pins one executor thread per core (src/main.rs:51-60); with one GPU per shard that thread and
 * the pinned buffers it stages through should sit on the GPU's NUMA node, or every byte crosses the socket interconnect on
 * its way to the PCIe root complex.  dbeel_bind_to_gpu moves the CALLING thread onto the CPUs of `device`'s NUMA node
 * (within the process's allowed set) and prefers that node for its future page allocations; call it before
 * dbeel_host_alloc / before touching the buffers.  numa_node / n_cpus (nullable) report what was applied (-1 / 0 when the
 * machine exposes no NUMA topology: not an error). */
int dbeel_gpu_numa_node(int device);
int dbeel_bind_to_gpu(int device, int *numa_node, int *n_cpus);

/* Upper bounds for the output buffers of a compaction of `runs` (host-side arithmetic only):
 * data_cap = sum(data_len), index_cap = 16 * sum(index_len/16), bloom_cap = size of the
 * .bloom file or 0 when sum(data_len) <= bloom_min_size. */
int dbeel_compact_bound(const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts,
                        uint64_t *data_cap, uint64_t *index_cap, uint64_t *bloom_cap);

/* Merge `runs` (runs[i] is position i in indices_to_compact: the final tie-break) into one
 * SSTable.  Host buffers in, host buffers out; copies are part of the call. */
int dbeel_compact(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs,
                  const dbeel_compact_opts *opts, dbeel_out *out);

/* The same compaction fed from files ["next" row N3: the storage edge].  The reference reads its inputs through
 * DmaStreamReaders (lsm_tree.rs:984-991) and writes through EntryWriter's buffered DMA files (entry_writer.rs:30-69); here
 * the caller hands over two callbacks instead of buffers, and the engine moves the bytes
 *     file -> read() -> pinned ring -> H2D -> kernels -> D2H -> pinned ring -> write() -> file
 * one key-range partition at a time, so file reads, both PCIe directions and file writes overlap and the page-locked
 * memory is a few partitions however large the SSTables are.  runs[i].data / .index are ignored (lengths only).
 *   read : fill dst with [offset, offset + len) of run `run`'s .data (DBEEL_STREAM_DATA) or .index (DBEEL_STREAM_INDEX)
 *   write: store len bytes at `offset` of the output's .data / .index / .bloom (DBEEL_STREAM_BLOOM: one call, offset 0)
 * Both are called from several engine threads at once (pread / pwrite are fine) and return 0 or an error code of the
 * caller's, which dbeel_compact_stream returns unchanged.  Output pieces arrive in no particular order; when an input turns
 * out to need the one-piece path (a run that ends early, lsm_tree.rs:1014,1063) the outputs are written again from offset
 * 0, so the caller truncates each output to out->*_len afterwards (bloom_len == 0: no .bloom file).  `out` returns
 * lengths only; its pointers are ignored.  Same bytes as dbeel_compact. */
#define DBEEL_STREAM_DATA 1u  /* = FileTypeKind::Data  (mod.rs:36-42) */
#define DBEEL_STREAM_INDEX 2u /* = FileTypeKind::Index */
#define DBEEL_STREAM_BLOOM 3u /* = FileTypeKind::Bloom */
typedef struct dbeel_stream_io {
    int (*read)(void *ctx, uint32_t run, uint32_t kind, uint64_t offset, uint64_t len, void *dst);
    int (*write)(void *ctx, uint32_t kind, uint64_t offset, const void *src, uint64_t len);
    void *ctx;
} dbeel_stream_io;
int dbeel_compact_stream(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs, const dbeel_compact_opts *opts,
                         const dbeel_stream_io *io, dbeel_out *out);

/* Same, inputs and outputs resident in device memory (16-byte aligned).  Returns after the
 * job has completed on the engine's stream. */
int dbeel_compact_device(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs,
                         const dbeel_compact_opts *opts, dbeel_out *out);

/* Memtable flush: `batch` holds writes in ARRIVAL order in run layout (keys may repeat, not
 * sorted).  Output = what flush_memtable_to_disk writes for the memtable those writes
 * build: ascending keys, last arrival per key, tombstones kept, no bloom.  The caller cuts
 * batches at memtable boundaries (dbeel_memtable_cut helps). */
int dbeel_flush(dbeel_engine *e, const dbeel_run *batch, dbeel_out *out);
int dbeel_flush_device(dbeel_engine *e, const dbeel_run *batch, dbeel_out *out);

/* Many memtables in one launch sequence (the flush side of a write-heavy shard produces a memtable every few
 * milliseconds; one job per memtable is launch-bound).  batches[i] is memtable i's arrivals (same layout as
 * dbeel_flush).  The n SSTables are written back to back into out->data / out->index; table[i] says where
 * SSTable i lives.  Every SSTable's .index offsets are relative to its own .data start, exactly what n separate
 * dbeel_flush calls would have produced. */
typedef struct dbeel_flush_table {
    uint64_t data_off, data_len;   /* bytes of out->data holding this memtable's .data file   */
    uint64_t index_off, index_len; /* bytes of out->index holding its .index file             */
    uint64_t items;                /* entries written (distinct keys of the memtable)          */
} dbeel_flush_table;
int dbeel_flush_many(dbeel_engine *e, const dbeel_run *batches, uint32_t n_batches, dbeel_out *out,
                     dbeel_flush_table *table /* n_batches rows, host memory */);
int dbeel_flush_many_device(dbeel_engine *e, const dbeel_run *batches, uint32_t n_batches, dbeel_out *out,
                            dbeel_flush_table *table);

/* ---- cfg5: shard routing + flushes of routed streams ---------------------------------------------------------------
 * A dbeel node runs one shard per core; a key belongs to the shard that owns murmur3_32(key bytes, seed 0) on the
 * consistent-hash ring of shard names "<node name>-<cpu id>" (hash_bytes / hash_string, src/shards.rs:95-101; names
 * :213-214).  MyShard::owns_key with replica_index 0 (shards.rs:586-598, checked per request in
 * src/tasks/db_server.rs:119-122): shard s owns the hashes in [hash of the previous shard on the ring, hash of s), wrapping
 * -- i.e. the first shard whose hash is GREATER than the key's.  (dbeel_client picks the first shard with hash >= the key's,
 * dbeel_client/src/lib.rs:344; the two differ only for a key whose hash equals a shard's, which that shard refuses.) */
#define DBEEL_MAX_SHARDS 256u
uint32_t dbeel_murmur3_32(const void *bytes, uint64_t len, uint32_t seed);                 /* host arithmetic */
uint32_t dbeel_ring_owner(const uint32_t *ring_hashes, uint32_t n_shards, uint32_t key_hash); /* host arithmetic: ring position */
/* Build the ring of `n_shards` shards of node `node_name` (NULL = "dbeel", args.rs): ring_hashes[] ascending,
 * ring_ids[p] = cpu id of the shard at ring position p.  Returns 0, or DBEEL_ERR_INVALID_ARG on a hash collision. */
int dbeel_shard_ring(const char *node_name, uint32_t n_shards, uint32_t *ring_hashes, uint32_t *ring_ids);

/* Route an arrival batch (run layout, arrival order; device pointers, 16-byte aligned) to the ring's shards on the GPU.
 * out_index (device, >= batch->index_len bytes) receives the batch's index records split into one stream per ring
 * position: position p's arrivals, in arrival order, are records [sum(counts[0..p)), +counts[p]).  The records are
 * unchanged -- they still point into batch->data -- so a shard's stream is an arrival batch with sparse offsets (below).
 * shard_of (device, n u32, or NULL) receives every arrival's ring position; counts / payload_bytes (host, n_shards each;
 * payload_bytes may be NULL) the arrivals and the sum of full_size per position.
 * out_key_hash64 (device, n u64, or NULL): a 64-bit identity of every arrival's key, in the same shard-major order as
 * out_index -- the input of dbeel_memtable_cuts_device. */
int dbeel_route_device(dbeel_engine *e, const dbeel_run *batch, const uint32_t *ring_hashes /* host, ascending */,
                       uint32_t n_shards, void *out_index, uint64_t out_index_cap, uint32_t *shard_of, void *out_key_hash64,
                       uint64_t *counts, uint64_t *payload_bytes);

/* The memtable-full trigger (lsm_tree.rs:747-765, 600-603: a flush starts right after the insert that makes the tree hold
 * `capacity` keys) for whole streams at once, on the device.  Stream s = key identities [stream_starts[s],
 * stream_starts[s+1]) of key_hash64 (arrival order).  cuts[cut_starts[s] .. cut_starts[s+1]) receive, for every FULL memtable
 * of stream s, the number of the stream's arrivals consumed up to and including it; what follows the last cut is the
 * memtable still filling.  capacity <= 9216 (shared-memory set); max_cuts_total >= sum(len(s) / capacity).
 * The identities are 64-bit hashes: a collision inside one memtable would cut one key late.  The flush reports every
 * SSTable's exact entry count -- a full memtable must yield exactly `capacity` -- so callers check that and fall back to the
 * exact host function dbeel_memtable_cut (dbeel_tree.h) on a mismatch. */
int dbeel_memtable_cuts_device(dbeel_engine *e, const void *key_hash64, const uint64_t *stream_starts /* host */,
                               uint32_t n_streams, uint32_t capacity, uint32_t *cuts /* host */, uint32_t *cut_starts /* host */,
                               uint32_t max_cuts_total);

/* dbeel_flush_many_device for batches whose index records do not abut in .data (slices of a routed stream: every batch's
 * `data` is the shared arrival buffer, `index` a slice of dbeel_route_device's out_index).  payload_bound >= the sum of
 * full_size over all batches (e.g. from payload_bytes above); out->data_cap >= payload_bound.  DBEEL_ERR_CAPACITY if the
 * bound turns out too low (nothing is written past it). */
int dbeel_flush_many_sparse_device(dbeel_engine *e, const dbeel_run *batches, uint32_t n_batches, uint64_t payload_bound,
                                   dbeel_out *out, dbeel_flush_table *table);

/* ---- N1: many independent compactions in one launch sequence ---------------------------------------------------
 * compact_tree (src/tasks/compaction.rs:82-101) issues one LSMTree::compact per group of SSTables it picked, and a node
 * runs one such loop per collection and shard; small level-0 merges are launch-bound one at a time.  Every job here is
 * exactly one dbeel_compact: its own runs (tie-break = position inside the job), its own keep_tombstones, its own bloom
 * filter (enabled and sized from ITS inputs, its own 32-byte seed).  Outputs land back to back in out->data /
 * out->index (file-relative .index offsets per job) and in out->bloom at 16-byte aligned offsets; results[j] says where.
 * Each job's three files are byte-identical to a separate dbeel_compact with the same arguments. */
typedef struct dbeel_job {
    const dbeel_run *runs;     /* in the order of indices_to_compact */
    uint32_t n_runs;
    int32_t keep_tombstones;
    const uint8_t *bloom_seed; /* 32 bytes, or NULL = fresh random seed */
} dbeel_job;
typedef struct dbeel_job_result {
    uint64_t data_off, data_len;
    uint64_t index_off, index_len;
    uint64_t bloom_off, bloom_len; /* bloom_len == 0: no filter for this job (lsm_tree.rs:1026-1034) */
    uint64_t items_written;
} dbeel_job_result;
int dbeel_compact_many_bound(const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size, double bloom_fp,
                             uint64_t *data_cap, uint64_t *index_cap, uint64_t *bloom_cap);
int dbeel_compact_many(dbeel_engine *e, const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size, double bloom_fp,
                       dbeel_out *out, dbeel_job_result *results);
int dbeel_compact_many_device(dbeel_engine *e, const dbeel_job *jobs, uint32_t n_jobs, uint64_t bloom_min_size,
                              double bloom_fp, dbeel_out *out, dbeel_job_result *results);

/* Asynchronous form of dbeel_compact for callers that must not block their reactor (dbeel's
 * compaction task runs on a glommio executor, src/tasks/compaction.rs:139-153): submit returns at
 * once, the job runs on an engine-owned worker thread, poll / wait report its status.  All
 * buffers (runs, the 32-byte seed, out) must stay valid until the job has been reaped by a
 * dbeel_wait() or a dbeel_poll() that returned 1.  One job per engine at a time (DBEEL_ERR_BUSY). */
int dbeel_compact_submit(dbeel_engine *e, const dbeel_run *runs, uint32_t n_runs,
                         const dbeel_compact_opts *opts, dbeel_out *out);
int dbeel_poll(dbeel_engine *e, int *status); /* returns 1 when finished (then *status = the job's code), else 0 */
int dbeel_wait(dbeel_engine *e);              /* blocks; returns the job's status code */

/* ---- N2: batched point lookups on the files this engine writes ------------------------------------------------
 * Replaces the SSTable loop of LSMTree::get_entry (src/storage_engine/lsm_tree.rs:686-719) for a batch of keys:
 * tables[] is the tree's `sstables` vector (oldest first; the loop walks it newest first, :688), every table is its
 * three files' bytes.  Per key: Bloom::check on the .bloom bytes (:691-696), then binary_search over .index / .data
 * (:605-670).  The memtable look-ups in front of it (:677-684) stay on the host.
 *
 *   DBEEL_LOOKUP_REFERENCE  binary_search restated step for step.  Its loop leaves right after probing index record 0
 *                           (`if half == 0 ... break`, :660), so a few present keys are reported absent -- this mode
 *                           reports exactly what the reference reports.
 *   DBEEL_LOOKUP_EXACT      lower-bound search: every present key is found.                                        */
#define DBEEL_LOOKUP_REFERENCE 0u
#define DBEEL_LOOKUP_EXACT 1u
#define DBEEL_LOOKUP_CORRUPT 0x80000000u /* in bloom_rejects: an index record pointed outside its .data file (the
                                            reference's read_at fails there and the whole get returns Err) */
typedef struct dbeel_table {
    const void *data;  uint64_t data_len;
    const void *index; uint64_t index_len;  /* multiple of 16 */
    const void *bloom; uint64_t bloom_len;  /* the .bloom file, or NULL / 0 when the table has none (:94-101) */
} dbeel_table;
typedef struct dbeel_lookup_result {
    int32_t table;          /* position in tables[] of the SSTable that answered, -1 = key not found      */
    uint32_t bloom_rejects; /* tables skipped by their filter before the answer (| DBEEL_LOOKUP_CORRUPT)    */
    uint64_t record;        /* index record number inside that table: its EntryOffset locates the entry    */
} dbeel_lookup_result;
/* keys: the query keys back to back; key_offsets: n_keys + 1 byte offsets (key i = keys[key_offsets[i] ..
 * key_offsets[i+1])).  dbeel_get_many takes host pointers everywhere and uploads the tables for the call (tests,
 * small tables); dbeel_get_many_device takes device pointers everywhere (tables resident in HBM, e.g. straight
 * from dbeel_compact_device) -- only the 172-byte trailer of each .bloom is read back to parse its parameters. */
int dbeel_get_many(dbeel_engine *e, const dbeel_table *tables, uint32_t n_tables, const void *keys,
                   const uint64_t *key_offsets, uint64_t n_keys, uint32_t mode, dbeel_lookup_result *results);
int dbeel_get_many_device(dbeel_engine *e, const dbeel_table *tables, uint32_t n_tables, const void *keys,
                          const uint64_t *key_offsets, uint64_t n_keys, uint32_t mode, dbeel_lookup_result *results);

/* ---- N4: write-ahead-log replay + flush ------------------------------------------------------------------------
 * Replaces LSMTree::read_memtable_from_wal_file (lsm_tree.rs:552-574) followed by flush_memtable_to_disk, i.e. the
 * recovery of an unflushed memtable in open_or_create_ex (:478-513).  `wal` is the whole `.memtable` file: bincode
 * Entries at 4096-aligned offsets, each padded to `size + 4096 - size % 4096` (:740-744).  Replay rules kept:
 * the cursor moves to the first page boundary strictly after every record; an entry whose timestamp does not
 * deserialize is skipped; a record that runs past the end of the file ends the replay; an all-zero page is the entry
 * (key = [], data = [], timestamp = 0).  `capacity` is the memtable's (DEFAULT_TREE_CAPACITY, mod.rs:18): more distinct
 * keys than that fail the reference's replay with ReachedCapacity -> DBEEL_ERR_TREE_FULL.  out->data / out->index
 * receive the SSTable; caps: the sum of the logged entries' sizes (<= wal_len) and 16 bytes per logged entry
 * (<= 16 * ceil(wal_len / 4096)).  No bloom (lsm_tree.rs:908). */
int dbeel_wal_flush(dbeel_engine *e, const void *wal, uint64_t wal_len, uint32_t capacity, dbeel_out *out);
int dbeel_wal_flush_device(dbeel_engine *e, const void *wal, uint64_t wal_len, uint32_t capacity, dbeel_out *out);

/* ---- hash-range scans: the iterator behind shard migration -----------------------------------------------------
 * Replaces the scan of migrate_actions (src/tasks/migration.rs:62-131): LSMTree::iter_filter (lsm_tree.rs:133-282) over
 * the whole tree, keeping every entry whose murmur3_32(key bytes, seed 0) lies in one of `ranges` and assigning it to the
 * FIRST range that holds (between_cmp, migration.rs:54-60; `position`, :98-104).  Range planning, the sends and the
 * deletes stay with the caller.
 *
 * tables[] lists the tables in iteration order: for a live tree its SSTables oldest first (ascending file index), then
 * the flushing memtable and then the active memtable, each as a sorted run-layout buffer (what dbeel_flush would write
 * for it).  Every table's records are visited 0 .. index_len/16 - 1 (a ragged tail is ignored); nothing is deduplicated,
 * so old versions and tombstones are yielded wherever they lie.  Every record is read the way AsyncIter::read_one reads
 * it: the full_size bytes at its `offset` (key_size is ignored) must deserialize as exactly one Entry, timestamp in range.
 *
 * The scan ends at the first record it cannot yield, like the reference's `while let Ok(Some(entry))` (:96): nothing
 * after it -- later tables and memtables included -- is selected.  *stop says where:
 *   DBEEL_SCAN_DECODE  a bincode or timestamp failure (the reference's loop ends silently there);
 *   DBEEL_SCAN_READ    full_size == 0, bytes past the end of .data, or a table with no record (its first index read hits
 *                      EOF; leave EMPTY MEMTABLES out of tables[] -- the reference iterates them without reading).  The
 *                      reference panics on these; whether a read past EOF panics there depends on whether the zero-padded
 *                      last page is in its page cache, and this engine always stops.
 *
 *   DBEEL_SCAN_REFERENCE  between_cmp read literally: a wrapped range (end < start) holds for every hash, start == end
 *                         for none.  Node removal and step 1 of node addition pass (previous shard, this shard), which
 *                         wraps for the lowest shard on the ring.
 *   DBEEL_SCAN_EXACT      a wrapped range is [start, 2^32) u [0, end).
 *
 * Output: range r's entries, in iteration order, back to back in out->data / out->index at per_range[r] (n_ranges rows,
 * host memory).  Every range's .index carries offsets relative to its own .data (key_size = 8 + klen, full_size), so
 * every range's output is both a valid SSTable-layout run and a valid arrival batch for dbeel_flush on the receiving
 * shard.  No bloom (bloom_cap is ignored).  data_cap >= sum(data_len) and index_cap >= 16 * records always suffice;
 * smaller caps that the selection does not fit give DBEEL_ERR_CAPACITY (nothing is written) with *stop filled in.
 * n_ranges > DBEEL_MAX_SCAN_RANGES: DBEEL_ERR_INVALID_ARG.  Zero tables or zero ranges: empty outputs.
 * dbeel_last_stats: ms_extract = classify, ms_resolve = split by range + offsets, ms_gather = payload copy.
 *
 * dbeel_scan_ranges takes host buffers and uploads every table whole (the tree must fit in device memory; nothing is
 * streamed); dbeel_scan_ranges_device takes tables and out in device memory (.index and outputs 16-byte aligned), ranges /
 * per_range / stop in host memory. */
#define DBEEL_SCAN_REFERENCE 0u
#define DBEEL_SCAN_EXACT 1u
#define DBEEL_MAX_SCAN_RANGES 256u
#define DBEEL_SCAN_END 0u    /* ran to the end of the last table          */
#define DBEEL_SCAN_DECODE 1u /* stopped: the reference's loop ends here   */
#define DBEEL_SCAN_READ 2u   /* stopped: the reference panics here        */
typedef struct dbeel_hash_range {
    uint32_t start, end;
} dbeel_hash_range;
typedef struct dbeel_scan_stop {
    int32_t table;   /* position in tables[] of the record that stopped the scan, -1: DBEEL_SCAN_END */
    uint32_t reason; /* DBEEL_SCAN_*                                                              */
    uint64_t record; /* its record number inside that table                                       */
} dbeel_scan_stop;
int dbeel_scan_ranges(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges,
                      uint32_t n_ranges, uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range, dbeel_scan_stop *stop);
int dbeel_scan_ranges_device(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges,
                             uint32_t n_ranges, uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range,
                             dbeel_scan_stop *stop);

/* The same scan fed from files, one output stream per range (shard migration sends every range's entries to another
 * shard, over a socket or a channel).  The engine moves the bytes
 *     file -> read() -> pinned ring -> H2D -> kernels -> D2H -> pinned ring -> write(range) -> the range's stream
 * one partition at a time, so the page-locked and device memory is a few partitions however large the tree is.  A
 * partition is a run of consecutive records in iteration order (it may span tables) whose index slices and .data spans
 * take at most partition_bytes (0 = the engine's partition size); a single record larger than that gets a partition of
 * its own.  tables[i].data / .index are ignored (lengths only); every table's .index is read whole first (16 bytes per
 * record), the .data files partition by partition.
 *   read : fill dst with [offset, offset + len) of table `table`'s .data (DBEEL_STREAM_DATA) or .index (DBEEL_STREAM_INDEX)
 *   write: store len bytes at `offset` of range `range`'s .data (DBEEL_STREAM_DATA) or .index (DBEEL_STREAM_INDEX) stream
 * Both are called from several engine threads at once and return 0 or an error code of the caller's, which
 * dbeel_scan_ranges_stream returns unchanged; the engine stays usable after one.  Pieces arrive in no particular order;
 * a range that selects nothing gets no write call.
 *
 * Range r's stream is byte for byte what dbeel_scan_ranges puts at per_range[r] for the same tables, ranges and mode: its
 * .data bytes, and its .index records with offsets relative to the range's own .data.  per_range[r] has data_off ==
 * index_off == 0 (every range is its own stream) and the lengths and items of dbeel_scan_ranges.  *stop is the same, and
 * nothing after the stop is ever written.  There is no output capacity (no DBEEL_ERR_CAPACITY).  The 2^32-record limit
 * of dbeel_scan_ranges applies per partition, not per call.  dbeel_last_stats fills partitions (partitions scanned), the
 * entries_* counts, input_bytes and output_bytes; ms_h2d, ms_total and ms_d2h are the sums over the partitions of the
 * H2D copies, the kernels and the D2H copies (they overlap each other and the callbacks). */
typedef struct dbeel_scan_io {
    int (*read)(void *ctx, uint32_t table, uint32_t kind, uint64_t offset, uint64_t len, void *dst);
    int (*write)(void *ctx, uint32_t range, uint32_t kind, uint64_t offset, const void *src, uint64_t len);
    void *ctx;
} dbeel_scan_io;
int dbeel_scan_ranges_stream(dbeel_engine *e, const dbeel_run *tables, uint32_t n_tables, const dbeel_hash_range *ranges,
                             uint32_t n_ranges, uint32_t mode, const dbeel_scan_io *io, uint64_t partition_bytes,
                             dbeel_flush_table *per_range, dbeel_scan_stop *stop);

/* Bloom::new_for_fp_rate arithmetic (bloomfilter 1.0.12). */
uint64_t dbeel_bloom_bitmap_bytes(uint64_t items, double fp);
uint32_t dbeel_bloom_k_num(uint64_t bitmap_bits, uint64_t items);
uint64_t dbeel_bloom_file_size(uint64_t items, double fp);

/* Pinned host memory for the host entry points (optional; any host pointer is accepted). */
void *dbeel_host_alloc(uint64_t bytes);
void dbeel_host_free(void *p);

int dbeel_last_stats(const dbeel_engine *e, dbeel_stats *out);
const char *dbeel_last_error(const dbeel_engine *e);
const char *dbeel_strerror(int code);
int dbeel_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* DBEEL_COMPACT_H */
