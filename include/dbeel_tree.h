/*
 * dbeel_tree.h -- host-side mirror of the file protocol AROUND the GPU path, C ABI.
 *
 * The reference is Rust (compiled code) and no Rust toolchain exists here, so the host side
 * above the engine's C ABI is C++ (dbeel_b200/csrc/host/lsm_tree_host.cc), mirroring the
 * reference's own interface for this path -- same names, argument meaning, error behaviour:
 *
 *   dbeel_tree_open        <- LSMTree::open_or_create_ex: journal replay + SSTable discovery
 *                             (src/storage_engine/lsm_tree.rs:424-465)
 *   dbeel_tree_recover_wal <- the rest of open_or_create_ex: an unflushed memtable's log is replayed and flushed
 *                             (lsm_tree.rs:466-513, read_memtable_from_wal_file :552-574) through dbeel_wal_flush()
 *   dbeel_tree_compact     <- LSMTree::compact(indices_to_compact, output_index, keep_tombstones)
 *                             (lsm_tree.rs:950-1156): same files, same CompactionAction journal
 *                             (:73-77, :1078-1111), same renames / deletes; the merge core
 *                             (:1002-1076) is dbeel_compact()
 *   dbeel_tree_flush       <- LSMTree::flush's SSTable part (lsm_tree.rs:875-915): writes the
 *                             next even index through dbeel_flush(), no bloom
 *   dbeel_tree_sstables    <- LSMTree::sstable_indices_and_sizes (lsm_tree.rs:592-598)
 *   dbeel_tree_get_many    <- the SSTable loop of LSMTree::get_entry (lsm_tree.rs:686-719) through dbeel_get_many()
 *   dbeel_tree_scan_ranges <- migrate_actions' scan over iter_filter (src/tasks/migration.rs:62-131) through
 *                             dbeel_scan_ranges()
 *   dbeel_tree_scan_ranges_to_dir <- the same scan streamed from the tree's files through dbeel_scan_ranges_stream(),
 *                             one pair of files per range
 *   dbeel_memtable_cut     <- RedBlackTree::set + active_memtable_full (rbtree_arena lib.rs:497-534,
 *                             lsm_tree.rs:600-603,757-765): how many arrivals fill one memtable
 *   dbeel_plan_compactions <- compact_tree's size-tiered picker (src/tasks/compaction.rs:35-102),
 *                             made deterministic (the reference enumerates a HashMap)
 */
#ifndef DBEEL_TREE_H
#define DBEEL_TREE_H

#include <stdint.h>

#include "dbeel_compact.h"

#ifdef __cplusplus
extern "C" {
#endif

#define DBEEL_ERR_IO 20        /* a filesystem call failed; dbeel_tree_last_error() has errno text */
#define DBEEL_ERR_NO_SSTABLE 21 /* an index in indices_to_compact has no .data/.index files */

typedef struct dbeel_tree dbeel_tree;

/* EntryWriter's page-cache write-through (src/storage_engine/entry_writer.rs:94-156): while it writes an SSTable the
 * reference mirrors both streams into the shard's page cache in 4 KiB pages keyed by ((FileTypeKind, files_index), page
 * address), the last page of each stream zero-padded at close().  dbeel_out_pages replays exactly those `set` calls -- same
 * pages, same order -- for an SSTable the engine produced (host buffers), so the Rust side can warm its PartitionPageCache
 * from the returned buffers.  Not on-disk state: skipping it can never serve stale bytes (the keys carry the fresh index). */
#define DBEEL_FILE_DATA 1u  /* FileTypeKind::Data  (mod.rs:36-42: Memtable, Data, Index, Bloom) */
#define DBEEL_FILE_INDEX 2u /* FileTypeKind::Index */
typedef void (*dbeel_page_sink)(void *ctx, uint32_t file_kind, uint64_t files_index, uint64_t address, const uint8_t *page /* 4096 bytes */);
int dbeel_out_pages(const void *data, uint64_t data_len, const void *index, uint64_t index_len, uint64_t files_index,
                    dbeel_page_sink sink, void *ctx);
/* A tree with a sink installed calls it for every SSTable dbeel_tree_compact / _compact_many / _flush / _recover_wal write. */
void dbeel_tree_set_page_sink(dbeel_tree *t, dbeel_page_sink sink, void *ctx);

int dbeel_tree_open(const char *dir, dbeel_engine *engine, uint64_t sstable_bloom_min_size, dbeel_tree **out);
void dbeel_tree_close(dbeel_tree *t);

/* (index, size = entries) of every SSTable, ascending by index.  Returns the count; fills up to cap. */
uint32_t dbeel_tree_sstables(const dbeel_tree *t, uint64_t *indices, uint64_t *sizes, uint32_t cap);
uint64_t dbeel_tree_write_sstable_index(const dbeel_tree *t); /* next even index a flush will use */

int dbeel_tree_compact(dbeel_tree *t, const uint64_t *indices_to_compact, uint32_t n, uint64_t output_index,
                       int keep_tombstones, const uint8_t *bloom_seed /* 32 bytes or NULL */);

/* compact_tree's loop (tasks/compaction.rs:82-101) in one go: all groups of a dbeel_plan_compactions() result (same
 * flattened layout) are merged by ONE dbeel_compact_many() call, then committed group by group exactly like
 * dbeel_tree_compact.  bloom_seeds: 32 bytes per group back to back, or NULL. */
int dbeel_tree_compact_many(dbeel_tree *t, const uint64_t *members, const uint32_t *group_start, uint32_t n_groups,
                            const uint64_t *output_index, const int32_t *keep_tombstones, const uint8_t *bloom_seeds);

/* Flush one memtable's arrivals (host buffers, arrival order) to the next even index. */
int dbeel_tree_flush(dbeel_tree *t, const dbeel_run *batch, uint64_t *written_index, uint64_t *items_written);

/* The SSTable loop of LSMTree::get_entry (lsm_tree.rs:686-719) for a batch of keys, over the tree's files (each table
 * with its .bloom if the file exists): results[i].table is a position in dbeel_tree_sstables() order.  Keys / modes /
 * rows as in dbeel_get_many.  The memtable look-ups in front of it (:677-684) are the caller's. */
int dbeel_tree_get_many(dbeel_tree *t, const void *keys, const uint64_t *key_offsets, uint64_t n_keys, uint32_t mode,
                        dbeel_lookup_result *results);

/* The scan of migrate_actions (src/tasks/migration.rs:62-131) over this tree through dbeel_scan_ranges(): the tree's
 * SSTables in dbeel_tree_sstables() order, then the caller's memtables (the flushing one, then the active one, each as a
 * sorted run: this mirror keeps no memtable; empty ones are skipped).  stop->table is a position in that combined order
 * (SSTables first, then memtables[]).  Ranges / modes / outputs as in dbeel_scan_ranges. */
int dbeel_tree_scan_ranges(dbeel_tree *t, const dbeel_run *memtables, uint32_t n_memtables, const dbeel_hash_range *ranges,
                           uint32_t n_ranges, uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range,
                           dbeel_scan_stop *stop);

/* The same scan, streamed: the SSTables are read from their files with pread, partition by partition, the memtables from
 * the caller's memory, through dbeel_scan_ranges_stream() (the tree's files are never held whole in memory).  Range r goes
 * to <out_dir>/<r>.data and <out_dir>/<r>.index (out_dir is created if missing): the bytes of range r's slice of
 * dbeel_tree_scan_ranges, its .index offsets relative to <r>.data.  Every file is cut to its final length; a range that
 * selects nothing leaves two empty files.  per_range rows have data_off == index_off == 0; stop as in
 * dbeel_tree_scan_ranges.  On an error every file this call created is removed. */
int dbeel_tree_scan_ranges_to_dir(dbeel_tree *t, const dbeel_run *memtables, uint32_t n_memtables, const dbeel_hash_range *ranges,
                                  uint32_t n_ranges, uint32_t mode, const char *out_dir, dbeel_flush_table *per_range,
                                  dbeel_scan_stop *stop);

/* WAL recovery step of open_or_create_ex.  0 logs: *wal_file_index = 0; 1 log: its index; 2 logs: the older one is
 * replayed (memtable of `tree_capacity` entries, DBEEL_ERR_TREE_FULL like the reference's ReachedCapacity), flushed
 * to `<newer index>.data / .index` exactly as the reference does, and removed; more than 2: error (the reference
 * panics).  *items_written = entries of the recovered SSTable (0 if nothing was recovered). */
int dbeel_tree_recover_wal(dbeel_tree *t, uint32_t tree_capacity, uint64_t *wal_file_index, uint64_t *items_written);

const char *dbeel_tree_last_error(const dbeel_tree *t);

/* Number of arrivals, starting at `first_record`, that a memtable of `capacity` distinct keys
 * absorbs before it is full (the insert that fills it included); the rest of the batch if it
 * never fills. */
uint64_t dbeel_memtable_cut(const dbeel_run *batch, uint64_t first_record, uint32_t capacity);

/* compact_tree's picker.  In: n SSTables (index, size).  Out: groups to compact, flattened:
 * group g covers members[group_start[g] .. group_start[g+1]) (SSTable indices, in the order they
 * must be passed as indices_to_compact), writes output_index[g], with keep_tombstones[g].
 * Groups are ordered largest tables first, so only the final level drops tombstones
 * (compaction.rs:91-92).  Returns the number of groups (<= n / 2). */
uint32_t dbeel_plan_compactions(const uint64_t *indices, const uint64_t *sizes, uint32_t n,
                                uint32_t compaction_factor, uint64_t *members, uint32_t *group_start,
                                uint64_t *output_index, int32_t *keep_tombstones);

#ifdef __cplusplus
}
#endif
#endif /* DBEEL_TREE_H */
