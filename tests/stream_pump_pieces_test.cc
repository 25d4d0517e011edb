// stream_pump_pieces_test.cc -- the multi-stream side of dbeel_b200/csrc/host/stream_pump.h (publish_pieces, end_at), the
// flow of the streamed hash-range scan, without a GPU.
//
// A fake engine walks the partitions like scan_stream_entry does: it waits for a partition's reads, "runs its kernels"
// (the output is a function of the partition's input bytes), fills the partition's output ring slot from a thread standing
// in for the D2H copy and publishes one piece per (stream, kind) the partition feeds, at the stream's running offset.
// Checks: every byte of every stream arrives exactly once, at its offset, with the right value; nothing is written for the
// partitions behind end_at; errors of either callback stop the pump with their code.
//
//   g++ -O1 -g -std=c++17 -pthread -fsanitize=thread tests/stream_pump_pieces_test.cc -o /tmp/t && /tmp/t
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <map>
#include <random>

#include "../dbeel_b200/csrc/host/stream_pump.h"

using dbeel::StreamPump;

namespace {

struct Files {
    std::vector<uint8_t> input; // one input "table"
    uint32_t n_streams = 0;
    std::vector<std::vector<uint8_t>> out;  // [2 s + kind - 1]
    std::vector<std::vector<uint8_t>> hits; // how often each byte was written
    std::atomic<int> reads{0}, writes{0};
    int fail_read_at = -1, fail_write_at = -1;
    std::mutex mu;
};

int rd(void *ctx, uint32_t table, uint32_t kind, uint64_t off, uint64_t len, void *dst) {
    Files *f = static_cast<Files *>(ctx);
    const int k = f->reads.fetch_add(1);
    if (k == f->fail_read_at) return 77;
    if (table != 0 || kind != DBEEL_STREAM_DATA || off + len > f->input.size()) return 78;
    if ((k & 7) == 0) std::this_thread::sleep_for(std::chrono::microseconds(150));
    memcpy(dst, f->input.data() + off, len);
    return 0;
}

int wr(void *ctx, uint32_t stream, uint32_t kind, uint64_t off, const void *src, uint64_t len) {
    Files *f = static_cast<Files *>(ctx);
    const int k = f->writes.fetch_add(1);
    if (k == f->fail_write_at) return 88;
    if (stream >= f->n_streams || (kind != DBEEL_STREAM_DATA && kind != DBEEL_STREAM_INDEX)) return 89;
    if ((k & 3) == 0) std::this_thread::sleep_for(std::chrono::microseconds(200));
    std::lock_guard<std::mutex> lk(f->mu);
    std::vector<uint8_t> &dst = f->out[2 * stream + kind - 1];
    std::vector<uint8_t> &h = f->hits[2 * stream + kind - 1];
    if (dst.size() < off + len) { dst.resize(off + len); h.resize(off + len); }
    memcpy(dst.data() + off, src, len);
    for (uint64_t i = 0; i < len; i++) h[off + i]++;
    return 0;
}

int legacy_write(void *, uint32_t, uint64_t, const void *, uint64_t) { return 90; } // publish_pieces must not call it

// The byte at `pos` of a partition's piece for (stream, kind): derived from the partition's input, so a misread ring slot shows.
uint8_t value(uint8_t in, uint32_t stream, uint32_t kind, uint64_t pos) { return (uint8_t)(in * 3 + stream * 7 + kind + pos); }

int scenario(uint32_t np, uint32_t n_streams, uint32_t ring, int threads, uint64_t max_len, unsigned seed, int fail_read_at,
             int fail_write_at, uint32_t end) {
    std::mt19937_64 rng(seed);
    Files f;
    f.fail_read_at = fail_read_at;
    f.fail_write_at = fail_write_at;
    f.n_streams = n_streams;
    f.out.resize(2 * n_streams);
    f.hits.resize(2 * n_streams);
    // per partition: its input length and, per (stream, kind), how many bytes it feeds (0 often: a range that selects nothing)
    std::vector<uint64_t> in_len(np), in_off(np + 1, 0);
    std::vector<std::vector<uint64_t>> plen(np, std::vector<uint64_t>(2 * n_streams));
    uint64_t max_in = 1, max_out = 1;
    for (uint32_t c = 0; c < np; c++) {
        in_len[c] = 1 + rng() % max_len;
        in_off[c + 1] = in_off[c] + in_len[c];
        uint64_t o = 0;
        for (auto &l : plen[c]) { l = rng() % 3 == 0 ? 0 : rng() % max_len; o += l; }
        max_in = std::max(max_in, in_len[c]);
        max_out = std::max(max_out, o);
    }
    f.input.resize(in_off[np]);
    for (auto &b : f.input) b = (uint8_t)rng();
    std::vector<uint8_t> ring_in((uint64_t)ring * max_in), ring_out((uint64_t)ring * max_out);
    std::vector<std::atomic<int>> d2h_done(np);
    for (auto &x : d2h_done) x.store(0);
    dbeel_stream_io io{rd, legacy_write, &f};
    StreamPump pump(&io, np, ring, threads, [&](uint32_t c) {
        while (!d2h_done[c].load(std::memory_order_acquire)) std::this_thread::yield();
    });
    pump.set_stream_write(wr);
    for (uint32_t c = 0; c < np; c++) pump.add_read(c, 0, DBEEL_STREAM_DATA, in_off[c], in_len[c], ring_in.data() + (uint64_t)(c % ring) * max_in);
    pump.start();
    std::vector<uint64_t> run(2 * n_streams, 0); // running stream offsets
    std::vector<std::thread> copiers;
    int rc = 0;
    uint32_t published = 0;
    for (uint32_t c = 0; c < np && !rc; c++) {
        if ((rc = pump.wait_reads(c))) break;
        const uint8_t *slot = ring_in.data() + (uint64_t)(c % ring) * max_in;
        if (memcmp(slot, f.input.data() + in_off[c], in_len[c]) != 0) { fprintf(stderr, "partition %u: ring slot misread\n", c); return -1; }
        const uint8_t first = slot[0];
        pump.release_input(c);
        if ((rc = pump.wait_out_slot(c))) break;
        uint8_t *oslot = ring_out.data() + (uint64_t)(c % ring) * max_out;
        std::vector<StreamPump::OutPiece> pieces;
        std::vector<uint8_t> img;
        for (uint32_t k = 0; k < 2 * n_streams; k++) {
            const uint32_t s = k / 2, kind = k % 2 + 1;
            for (uint64_t i = 0; i < plen[c][k]; i++) img.push_back(value(first, s, kind, run[k] + i));
            if (plen[c][k]) pieces.push_back(StreamPump::OutPiece{oslot + img.size() - plen[c][k], plen[c][k], s, kind, run[k]});
            run[k] += plen[c][k];
        }
        copiers.emplace_back([&, c, oslot, img]() { // the "D2H", a little later
            std::this_thread::sleep_for(std::chrono::microseconds(80 + 40 * (c % 4)));
            memcpy(oslot, img.data(), img.size());
            d2h_done[c].store(1, std::memory_order_release);
        });
        pump.publish_pieces(c, pieces);
        published = c + 1;
        if (c + 1 == end) { pump.end_at(end); break; }
    }
    if (rc) pump.abort(rc);
    const int frc = rc ? rc : pump.finish();
    for (auto &t : copiers) t.join();
    if (frc) return frc;
    // every stream: exactly the bytes of the published partitions, each once
    for (uint32_t k = 0; k < 2 * n_streams; k++) {
        const uint32_t s = k / 2, kind = k % 2 + 1;
        uint64_t want = 0, pos = 0;
        for (uint32_t c = 0; c < published; c++) want += plen[c][k];
        if (f.out[k].size() != want) { fprintf(stderr, "stream %u kind %u: %zu bytes, want %llu\n", s, kind, f.out[k].size(), (unsigned long long)want); return -2; }
        for (uint32_t c = 0; c < published; c++) {
            const uint8_t first = f.input[in_off[c]];
            for (uint64_t i = 0; i < plen[c][k]; i++, pos++)
                if (f.out[k][pos] != value(first, s, kind, pos) || f.hits[k][pos] != 1) {
                    fprintf(stderr, "stream %u kind %u byte %llu wrong (hits %u)\n", s, kind, (unsigned long long)pos, f.hits[k][pos]);
                    return -3;
                }
        }
    }
    return 0;
}

} // namespace

int main() {
    int bad = 0;
    unsigned seed = 1;
    for (uint32_t np : {1u, 2u, 5u, 17u})
        for (uint32_t ring : {2u, 3u, 4u})
            for (int threads : {1, 3, 8}) {
                const int rc = scenario(np, 1 + seed % 6, ring, threads, 700, seed, -1, -1, np);
                seed++;
                if (rc) { fprintf(stderr, "scenario np=%u ring=%u threads=%d -> %d\n", np, ring, threads, rc); bad++; }
            }
    // pieces larger than kPiece: one piece becomes several callback calls
    if (const int rc = scenario(3, 2, 2, 4, 18ull << 20, 999, -1, -1, 3)) { fprintf(stderr, "large -> %d\n", rc); bad++; }
    // end_at: the partitions behind it are never read past the ring's lead, published or written
    for (uint32_t end : {1u, 4u, 9u})
        if (const int rc = scenario(12, 3, 3, 4, 500, 700 + end, -1, -1, end)) { fprintf(stderr, "end_at(%u) -> %d\n", end, rc); bad++; }
    // error injection: the pump stops with the callback's code, never hangs
    for (int at : {0, 2, 9, 20}) {
        int rc = scenario(10, 4, 3, 4, 500, 500 + at, at % 10, -1, 10); // one read per partition
        if (rc != 77) { fprintf(stderr, "read failure at %d -> %d (want 77)\n", at, rc); bad++; }
        rc = scenario(10, 4, 3, 4, 500, 600 + at, -1, at, 10);
        if (rc != 88) { fprintf(stderr, "write failure at %d -> %d (want 88)\n", at, rc); bad++; }
    }
    printf(bad ? "FAILED %d\n" : "ok\n", bad);
    return bad ? 1 : 0;
}
