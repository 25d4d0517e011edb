/*
 * scan_oracle.c -- CPU restatement of the scan shard migration runs over a tree: migrate_actions
 * (src/tasks/migration.rs:62-131) over LSMTree::iter_filter / AsyncIter (src/storage_engine/lsm_tree.rs:133-282).
 *
 * TEST INFRASTRUCTURE ONLY, like oracle/dbeel_oracle.c: nothing under dbeel_b200/ links or imports it.  It compiles the
 * compaction oracle into itself and reuses its restatements of the on-disk records (entry_decode: bincode with
 * reject_trailing_bytes + the timestamp range) and of murmur3_32; the compaction oracle's own source stays as it is.
 *
 * Functions below restate, in order:
 *   between_cmp ........ migration.rs:54-60 (mode 1 = the exact reading of a wrapped range, see dbeel_compact.h)
 *   filter + position .. migration.rs:86-104 (the iter_filter closure, then `position` on the yielded entry)
 *   read_one ........... lsm_tree.rs:213-282 (UnreadSSTable -> ReadingSSTable -> Memtable), with the read failures of
 *                        CachedFileReader (cached_file_reader.rs:65-68, 82) and the index read past EOF of an empty table
 *   migrate_actions .... migration.rs:96 `while let Ok(Some(entry))`: the first Err ends the scan
 */
#include "../oracle/dbeel_oracle.c"

#define SCAN_END 0u
#define SCAN_DECODE 1u
#define SCAN_READ 2u

static int between_cmp(uint32_t hash, uint32_t start, uint32_t end, uint32_t mode) {
    if (end < start) {
        if (mode) return hash >= start || hash < end;
        return hash < start || hash >= end; /* hash.cmp(start) == Less || hash.cmp(end) != Less */
    }
    return hash >= start && hash < end; /* hash.cmp(start) != Less && hash.cmp(end) == Less */
}

/* position(): the first range that holds, or -1 (the iter_filter closure's `any` is position() >= 0) */
static int32_t range_of(const uint8_t *key, uint64_t klen, const uint32_t *ranges, uint32_t n_ranges, uint32_t mode) {
    const uint32_t hash = orc_murmur3_32(key, klen, 0); /* hash_bytes, shards.rs:95-101 */
    for (uint32_t r = 0; r < n_ranges; r++)
        if (between_cmp(hash, ranges[2 * r], ranges[2 * r + 1], mode)) return (int32_t)r;
    return -1;
}

typedef struct {
    uint32_t table;     /* IterState: table i, or n_tables = Memtable (nothing left: the memtables are tables here) */
    uint64_t record;    /* index_offset / 16 */
} scan_iter;

/* One read_one step that reads a record.  Returns 1 with the entry's location, 0 at the end, or -(reason) on Err. */
static int read_one(const orc_run *tables, uint32_t n_tables, scan_iter *it, const uint8_t **entry, uint64_t *klen, uint32_t *full_size) {
    if (it->table >= n_tables) return 0;
    const orc_run *t = &tables[it->table];
    const uint64_t size = t->index_len / INDEX_ENTRY_SIZE; /* sstable.size (:451-453) */
    if (size == 0) return -(int)SCAN_READ;                 /* read_at_into(0, 16 bytes) hits EOF */
    const uint8_t *rec = t->index + it->record * INDEX_ENTRY_SIZE;
    const uint64_t offset = rd_u64(rec);
    const uint32_t fs = rd_u32(rec + 12); /* EntryOffset { offset, key_size (unused), full_size } */
    if (fs == 0) return -(int)SCAN_READ;  /* assert_ne!(size, 0), cached_file_reader.rs:82 */
    if (offset > t->data_len || fs > t->data_len - offset) return -(int)SCAN_READ; /* page[start..end] past EOF */
    orc_entry e;
    if (!entry_decode(t->data + offset, fs, &e)) return -(int)SCAN_DECODE;
    *entry = t->data + offset;
    *klen = e.klen;
    *full_size = fs;
    entry_free(&e);
    it->record++;
    if (it->record >= size) { it->table++; it->record = 0; } /* the next table, or the memtable state */
    return 1;
}

/* out->data / out->index: range-major, iteration order inside a range, every range's offsets relative to its own start.
 * per_range: 5 u64 per range {data_off, data_len, index_off, index_len, items}.  Returns 0 or ORC_ERR_*. */
int orc_scan_ranges(const orc_run *tables, uint32_t n_tables, const uint32_t *ranges, uint32_t n_ranges, uint32_t mode,
                    orc_out *out, uint64_t *per_range, int32_t *stop_table, uint32_t *stop_reason, uint64_t *stop_record) {
    uint64_t total = 0;
    for (uint32_t t = 0; t < n_tables; t++) total += tables[t].index_len / INDEX_ENTRY_SIZE;
    const uint8_t **sel = (const uint8_t **)malloc(sizeof(*sel) * (total ? total : 1));
    uint64_t *sel_kl = (uint64_t *)malloc(8 * (total ? total : 1));
    uint32_t *sel_fs = (uint32_t *)malloc(4 * (total ? total : 1)), *sel_r = (uint32_t *)malloc(4 * (total ? total : 1));
    if (!sel || !sel_kl || !sel_fs || !sel_r) { free(sel); free(sel_kl); free(sel_fs); free(sel_r); return ORC_ERR_NOMEM; }
    scan_iter it = {0, 0};
    *stop_table = -1;
    *stop_reason = SCAN_END;
    *stop_record = 0;
    uint64_t n_sel = 0;
    for (;;) {
        const uint8_t *ent;
        uint64_t klen;
        uint32_t fs;
        const scan_iter at = it;
        const int rc = read_one(tables, n_tables, &it, &ent, &klen, &fs);
        if (rc == 0) break;
        if (rc < 0) {
            *stop_table = (int32_t)at.table;
            *stop_reason = (uint32_t)-rc;
            *stop_record = at.record;
            break;
        }
        const int32_t r = range_of(ent + 8, klen, ranges, n_ranges, mode);
        if (r < 0) continue; /* the filter said no: read_one returns Continue */
        sel[n_sel] = ent;
        sel_kl[n_sel] = klen;
        sel_fs[n_sel] = fs;
        sel_r[n_sel] = (uint32_t)r;
        n_sel++;
    }
    uint64_t data_total = 0;
    for (uint32_t r = 0; r < n_ranges; r++) memset(per_range + 5 * r, 0, 40);
    for (uint64_t k = 0; k < n_sel; k++) {
        per_range[5 * sel_r[k] + 1] += sel_fs[k];
        per_range[5 * sel_r[k] + 4] += 1;
        data_total += sel_fs[k];
    }
    int ret = ORC_OK;
    if (data_total > out->data_cap || 16 * n_sel > out->index_cap) {
        ret = ORC_ERR_CAPACITY;
    } else {
        uint64_t d = 0, i = 0;
        for (uint32_t r = 0; r < n_ranges; r++) {
            per_range[5 * r] = d;
            per_range[5 * r + 2] = i * 16;
            per_range[5 * r + 3] = per_range[5 * r + 4] * 16;
            d += per_range[5 * r + 1];
            i += per_range[5 * r + 4];
        }
        uint64_t *dcur = (uint64_t *)calloc(n_ranges ? n_ranges : 1, 8), *icur = (uint64_t *)calloc(n_ranges ? n_ranges : 1, 8);
        if (!dcur || !icur) {
            ret = ORC_ERR_NOMEM;
        } else {
            for (uint64_t k = 0; k < n_sel; k++) { /* the receiving end of range r sees its entries in iteration order */
                const uint32_t r = sel_r[k];
                uint8_t *irec = out->index + per_range[5 * r + 2] + 16 * icur[r];
                memcpy(out->data + per_range[5 * r] + dcur[r], sel[k], sel_fs[k]);
                wr_u64(irec, dcur[r]);
                wr_u32(irec + 8, (uint32_t)(8 + sel_kl[k]));
                wr_u32(irec + 12, sel_fs[k]);
                dcur[r] += sel_fs[k];
                icur[r]++;
            }
            out->data_len = d;
            out->index_len = 16 * i;
            out->items_written = i;
        }
        free(dcur);
        free(icur);
    }
    free(sel); free(sel_kl); free(sel_fs); free(sel_r);
    return ret;
}

int orc_between_cmp(uint32_t hash, uint32_t start, uint32_t end, uint32_t mode) { return between_cmp(hash, start, end, mode); }
