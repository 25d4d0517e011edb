// Host build of the streamed scan's partition planner (dbeel_b200/csrc/host/scan_plan.h, the code the engine runs),
// exported with a C ABI so tests/test_scan_plan.py can check its plans against a Python restatement without a GPU.
#include <stdint.h>

#include "../dbeel_b200/csrc/host/scan_plan.h"

using namespace dbeel;

extern "C" {

// pieces: 6 words per piece {part, table, rec_lo, rec_hi, span_lo, span_hi}; parts: 4 words per partition {first_ordinal,
// records, span_bytes, data_bytes}; summary: {pieces, partitions, scheduled, stopped, stop_table, stop_record}.
// Returns -1 when the arrays are too small.
int shim_scan_plan(uint32_t n_tables, const uint64_t *data_len, const uint8_t *const *index, const uint64_t *n, uint64_t budget,
                   uint64_t *pieces, uint64_t max_pieces, uint64_t *parts, uint64_t max_parts, uint64_t *summary) {
    std::vector<ScanPlanTable> t(n_tables);
    for (uint32_t i = 0; i < n_tables; i++) t[i] = ScanPlanTable{data_len[i], index[i], n[i]};
    const ScanPlan p = scan_plan(t.data(), n_tables, budget);
    if (p.pieces.size() > max_pieces || p.parts.size() > max_parts) return -1;
    for (size_t c = 0; c < p.parts.size(); c++) {
        const ScanPart &q = p.parts[c];
        parts[4 * c] = q.first_ordinal;
        parts[4 * c + 1] = q.records;
        parts[4 * c + 2] = q.span_bytes;
        parts[4 * c + 3] = q.data_bytes;
        for (uint32_t k = q.first_piece; k < q.first_piece + q.n_pieces; k++) {
            const ScanPiece &s = p.pieces[k];
            uint64_t *w = pieces + 6 * k;
            w[0] = c; w[1] = s.table; w[2] = s.rec_lo; w[3] = s.rec_hi; w[4] = s.span_lo; w[5] = s.span_hi;
        }
    }
    summary[0] = p.pieces.size();
    summary[1] = p.parts.size();
    summary[2] = p.scheduled;
    summary[3] = p.stopped;
    summary[4] = p.stop_table;
    summary[5] = p.stop_record;
    return 0;
}
}
