// scan_plan.h -- the partition plan of a streamed hash-range scan (dbeel_scan_ranges_stream).  Plain C++: no CUDA in
// here, so the plan is tested on a box without a GPU (tests/scan_plan_shim.cc, tests/test_scan_plan.py).
//
// The scan visits the tables' records in iteration order (tables in order, records in order).  The plan cuts that order
// into partitions: runs of consecutive records, possibly spanning tables.  A partition holds one PIECE per table it
// touches: the piece's index slice and one contiguous .data span that covers every record of the slice.  The engine
// moves a partition's spans and slices into a ring slot and runs the scan kernels over its records.
//
// Rules:
//   - the records at and after the first READ stop (entry_readable fails, or a table without a record) are not scheduled:
//     the reference panics there, and nothing after it may be selected; stopped / stop_table / stop_record say where;
//   - every scheduled record is readable, so its bytes [offset, offset + full_size) lie inside its piece's span;
//   - a partition's index bytes plus span bytes stay within `budget`, unless it holds a single record that alone exceeds
//     it; scattered offsets (a damaged or hand-made index) only make the spans, and so the partitions, smaller;
//   - a partition holds fewer than kScanPartMaxRecords records (the kernels count records in 32 bits).
#pragma once
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../device_fns.cuh"

namespace dbeel {

constexpr uint64_t kScanPartMaxRecords = 0xFFFFFFF0ull;

struct ScanPiece {
    uint32_t table;
    uint64_t rec_lo, rec_hi;   // index records [rec_lo, rec_hi) of the table
    uint64_t span_lo, span_hi; // .data bytes [span_lo, span_hi) of the table
};

struct ScanPart {
    uint32_t first_piece, n_pieces; // pieces[first_piece, first_piece + n_pieces)
    uint64_t first_ordinal;         // global ordinal of the partition's first record
    uint64_t records;
    uint64_t span_bytes;            // sum of the pieces' spans
    uint64_t data_bytes;            // sum of the records' full_size: what the partition can select at most
};

struct ScanPlanTable {
    uint64_t data_len;  // the .data file's length
    const uint8_t *index; // the whole .index file (16-byte records, little-endian)
    uint64_t n;           // index_len / 16
};

struct ScanPlan {
    std::vector<ScanPiece> pieces;
    std::vector<ScanPart> parts;
    uint64_t scheduled = 0; // records scheduled = ordinal of the READ stop when there is one
    bool stopped = false;   // a READ stop lies in front of the end of the last table
    uint32_t stop_table = 0;
    uint64_t stop_record = 0;
};

inline void scan_plan_record(const uint8_t *index, uint64_t r, uint64_t *off, uint32_t *fs) {
    memcpy(off, index + 16 * r, 8);
    memcpy(fs, index + 16 * r + 12, 4);
}

inline ScanPlan scan_plan(const ScanPlanTable *tables, uint32_t n_tables, uint64_t budget) {
    ScanPlan p;
    bool open = false;       // a partition is being filled
    bool piece_open = false; // ... and its last piece belongs to the current table
    uint64_t cost = 0;       // index bytes + span bytes of the open partition
    auto close_part = [&]() {
        if (open) {
            ScanPart &q = p.parts.back();
            q.n_pieces = (uint32_t)(p.pieces.size() - q.first_piece);
        }
        open = false;
        piece_open = false;
        cost = 0;
    };
    for (uint32_t t = 0; t < n_tables && !p.stopped; t++) {
        piece_open = false;
        if (tables[t].n == 0) { // its first 16-byte index read hits EOF
            p.stopped = true;
            p.stop_table = t;
            p.stop_record = 0;
            break;
        }
        for (uint64_t r = 0; r < tables[t].n; r++) {
            uint64_t off;
            uint32_t fs;
            scan_plan_record(tables[t].index, r, &off, &fs);
            if (!entry_readable(off, fs, tables[t].data_len)) {
                p.stopped = true;
                p.stop_table = t;
                p.stop_record = r;
                break;
            }
            // what the open partition would cost with this record in it
            uint64_t grow = 16 + fs;
            if (open && piece_open) {
                const ScanPiece &k = p.pieces.back();
                const uint64_t lo = off < k.span_lo ? off : k.span_lo, hi = off + fs > k.span_hi ? off + fs : k.span_hi;
                grow = 16 + (hi - lo) - (k.span_hi - k.span_lo);
            }
            if (open && (cost + grow > budget || p.parts.back().records + 1 >= kScanPartMaxRecords)) {
                close_part();
                grow = 16 + fs;
            }
            if (!open) {
                p.parts.push_back(ScanPart{(uint32_t)p.pieces.size(), 0, p.scheduled, 0, 0, 0});
                open = true;
            }
            ScanPart &q = p.parts.back();
            if (!piece_open) {
                p.pieces.push_back(ScanPiece{t, r, r + 1, off, off + fs});
                piece_open = true;
            } else {
                ScanPiece &k = p.pieces.back();
                k.rec_hi = r + 1;
                q.span_bytes -= k.span_hi - k.span_lo;
                if (off < k.span_lo) k.span_lo = off;
                if (off + fs > k.span_hi) k.span_hi = off + fs;
            }
            q.span_bytes += p.pieces.back().span_hi - p.pieces.back().span_lo;
            q.records++;
            q.data_bytes += fs;
            cost += grow;
            p.scheduled++;
        }
    }
    close_part();
    return p;
}

} // namespace dbeel
