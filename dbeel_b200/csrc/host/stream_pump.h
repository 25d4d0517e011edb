// stream_pump.h -- the threads between a file (the caller's read / write callbacks) and the pinned rings of the streaming
// host path (dbeel_compact_stream, row N3: the storage edge).  Plain C++: no CUDA in here, so the flow control is
// exercised on a box without a GPU (tests/stream_pump_test.cc); the engine supplies "wait until partition c's D2H has
// landed" as a callable.
//
// The pipeline of dbeel_compact.cu walks the key-range partitions of a compaction in order.  With files on both sides:
//
//   reader threads   pull partition c's slices of every run into ring slot c mod R of the pinned INPUT ring -- as soon
//                    as the partition that used the slot before (c - R) has been consumed (its kernels are done)
//   engine thread    waits for partition c's reads, enqueues its H2D / kernels / D2H (into slot c mod R of the pinned
//                    OUTPUT ring, once partition c - R has left it), publishes what the D2H will deliver
//   writer threads   walk the partitions in order: wait for the D2H, push the slot's bytes through the write callback
//                    in pieces, hand the slot back
//
// so file reads, both PCIe directions and file writes all overlap, and the pinned memory is R slots however large the
// SSTables are.  Any callback error aborts the pump; the first error code is what every wait returns from then on.
//
// A partition's output is either one .data and one .index piece of a single output (publish_out, the compaction) or any
// number of pieces that each name an output stream, a kind and an offset (publish_pieces, the streamed scan: one output
// stream per hash range, written through the stream-write callback).  end_at(n) ends the walk after partition n - 1: the
// later partitions are never read, published or written (the scan stops there).
#pragma once
#include <stdint.h>

#include <atomic>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "../../../include/dbeel_compact.h"

namespace dbeel {

class StreamPump {
  public:
    struct ReadTask {
        uint32_t part, run, kind;
        uint64_t off, len;
        uint8_t *dst;
    };
    struct OutPart { // where partition c's output sits in the pinned ring and where it goes in the files
        const uint8_t *data = nullptr;
        uint64_t data_len = 0, data_off = 0;
        const uint8_t *index = nullptr;
        uint64_t index_len = 0, index_off = 0;
    };
    struct OutPiece { // one piece of a multi-stream partition: len bytes at src go to offset `off` of (stream, kind)
        const uint8_t *src = nullptr;
        uint64_t len = 0;
        uint32_t stream = 0, kind = 0;
        uint64_t off = 0;
    };
    typedef int (*StreamWriteFn)(void *ctx, uint32_t stream, uint32_t kind, uint64_t offset, const void *src, uint64_t len);
    static constexpr uint64_t kPiece = 8ull << 20; // bytes per callback call

    // wait_out(c): blocks until partition c's output has arrived in host memory (the engine: cudaEventSynchronize).
    // thread_init(): run once on every pump thread (the engine: cudaSetDevice).
    StreamPump(const dbeel_stream_io *io, uint32_t n_parts, uint32_t ring, int n_threads, std::function<void(uint32_t)> wait_out,
               std::function<void()> thread_init = nullptr)
        : io_(io), np_(n_parts), ring_(ring ? ring : 1), nt_(n_threads > 0 ? n_threads : 1), wait_out_(std::move(wait_out)),
          thread_init_(std::move(thread_init)), r_left_(n_parts, 0), w_left_(n_parts, 0), w_next_(new std::atomic<uint64_t>[n_parts ? n_parts : 1]),
          chunks_(n_parts), end_(n_parts) {
        for (uint32_t c = 0; c < n_parts; c++) w_next_[c].store(0);
    }
    StreamPump(const StreamPump &) = delete;
    StreamPump &operator=(const StreamPump &) = delete;
    ~StreamPump() {
        abort(DBEEL_ERR_INVALID_ARG); // no-op for the error code when the pump finished cleanly
        join();
    }

    // Before start(), in partition order.  A slice longer than kPiece becomes several tasks.
    void add_read(uint32_t part, uint32_t run, uint32_t kind, uint64_t off, uint64_t len, uint8_t *dst) {
        for (uint64_t done = 0; done < len; done += kPiece) {
            const uint64_t n = len - done < kPiece ? len - done : kPiece;
            tasks_.push_back(ReadTask{part, run, kind, off + done, n, dst + done});
            r_left_[part]++;
        }
    }

    // Before start(): the callback publish_pieces writes through (ctx = the read callback's).
    void set_stream_write(StreamWriteFn fn) { stream_write_ = fn; }

    void start() {
        started_ = true;
        for (int i = 0; i < nt_; i++) threads_.emplace_back([this] { reader(); });
        for (int i = 0; i < nt_; i++) threads_.emplace_back([this] { writer(); });
    }

    int wait_reads(uint32_t part) {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return failed_ || r_left_[part] == 0; });
        return failed_ ? err_ : 0;
    }

    void release_input(uint32_t part) {
        std::lock_guard<std::mutex> lk(mu_);
        if (part + 1 > consumed_) consumed_ = part + 1;
        cv_.notify_all();
    }

    // The output ring slot of `part` is free once partition part - ring has been written out.
    int wait_out_slot(uint32_t part) {
        if (part < ring_) return 0;
        const uint32_t prev = part - ring_;
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return failed_ || (published_ > prev && w_left_[prev] == 0); });
        return failed_ ? err_ : 0;
    }

    void publish_out(uint32_t part, const OutPart &o) {
        std::vector<Chunk> ch;
        split(&ch, o.data, o.data_len, 0, DBEEL_STREAM_DATA, o.data_off, false);
        split(&ch, o.index, o.index_len, 0, DBEEL_STREAM_INDEX, o.index_off, false);
        publish(part, std::move(ch));
    }

    void publish_pieces(uint32_t part, const std::vector<OutPiece> &ps) {
        std::vector<Chunk> ch;
        for (const OutPiece &q : ps) split(&ch, q.src, q.len, q.stream, q.kind, q.off, true);
        publish(part, std::move(ch));
    }

    // Partitions [n, n_parts) will not be published: their reads are skipped and finish() does not wait for them.
    void end_at(uint32_t n) {
        std::lock_guard<std::mutex> lk(mu_);
        if (n < end_) end_ = n;
        cv_.notify_all();
    }

    // Everything published has been written (or the pump failed).  Joins the threads.
    int finish() {
        {
            std::unique_lock<std::mutex> lk(mu_);
            cv_.wait(lk, [&] {
                if (failed_) return true;
                if (published_ < end_) return false;
                for (uint32_t c = 0; c < end_; c++)
                    if (w_left_[c]) return false;
                return true;
            });
            done_ = true;
            cv_.notify_all();
        }
        join();
        return failed_ ? err_ : 0;
    }

    void abort(int code) {
        std::lock_guard<std::mutex> lk(mu_);
        if (!failed_ && !done_) {
            failed_ = true;
            err_ = code;
        }
        cv_.notify_all();
    }

  private:
    struct Chunk { // one write callback call
        const uint8_t *src;
        uint64_t len;
        uint32_t stream, kind;
        uint64_t off;
        bool multi; // through stream_write_
    };

    static void split(std::vector<Chunk> *ch, const uint8_t *src, uint64_t len, uint32_t stream, uint32_t kind, uint64_t off, bool multi) {
        for (uint64_t done = 0; done < len; done += kPiece)
            ch->push_back(Chunk{src + done, len - done < kPiece ? len - done : kPiece, stream, kind, off + done, multi});
    }

    void publish(uint32_t part, std::vector<Chunk> ch) {
        std::lock_guard<std::mutex> lk(mu_);
        chunks_[part] = std::move(ch);
        w_left_[part] = chunks_[part].size();
        published_ = part + 1;
        cv_.notify_all();
    }

    void join() {
        for (auto &t : threads_)
            if (t.joinable()) t.join();
        threads_.clear();
    }

    void fail_locked(int code) {
        if (!failed_) {
            failed_ = true;
            err_ = code ? code : DBEEL_ERR_INVALID_ARG;
        }
    }

    void reader() {
        if (thread_init_) thread_init_();
        while (true) {
            const size_t k = r_next_.fetch_add(1);
            if (k >= tasks_.size()) return;
            const ReadTask &t = tasks_[k];
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return failed_ || t.part >= end_ || t.part < consumed_ + ring_; });
                if (failed_) return;
                if (t.part >= end_) continue;
            }
            const int rc = io_->read(io_->ctx, t.run, t.kind, t.off, t.len, t.dst);
            std::lock_guard<std::mutex> lk(mu_);
            if (rc) fail_locked(rc);
            r_left_[t.part]--;
            cv_.notify_all();
            if (failed_) return;
        }
    }

    void writer() {
        if (thread_init_) thread_init_();
        for (uint32_t c = 0; c < np_; c++) {
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return failed_ || c >= end_ || published_ > c; });
                if (failed_ || c >= end_) return;
            }
            const std::vector<Chunk> &ch = chunks_[c]; // not modified once published
            const uint64_t total = ch.size();
            if (total == 0) continue;
            if (wait_out_) wait_out_(c);
            while (true) {
                const uint64_t k = w_next_[c].fetch_add(1);
                if (k >= total) break;
                const Chunk &q = ch[k];
                const int rc = q.multi ? stream_write_(io_->ctx, q.stream, q.kind, q.off, q.src, q.len)
                                       : io_->write(io_->ctx, q.kind, q.off, q.src, q.len);
                std::lock_guard<std::mutex> lk(mu_);
                if (rc) fail_locked(rc);
                w_left_[c]--;
                cv_.notify_all();
                if (failed_) return;
            }
        }
    }

    const dbeel_stream_io *io_;
    const uint32_t np_, ring_;
    const int nt_;
    std::function<void(uint32_t)> wait_out_;
    std::function<void()> thread_init_;
    std::vector<ReadTask> tasks_;
    std::atomic<size_t> r_next_{0};
    std::mutex mu_;
    std::condition_variable cv_;
    // all below under mu_
    std::vector<uint32_t> r_left_;
    std::vector<uint64_t> w_left_;
    std::unique_ptr<std::atomic<uint64_t>[]> w_next_;
    std::vector<std::vector<Chunk>> chunks_;
    StreamWriteFn stream_write_ = nullptr;
    uint32_t end_;           // partitions [end_, np_) are skipped
    uint32_t consumed_ = 0;  // partitions [0, consumed_) have released their input slot
    uint32_t published_ = 0; // partitions [0, published_) have their output described
    bool failed_ = false, done_ = false, started_ = false;
    int err_ = 0;
    std::vector<std::thread> threads_;
};

} // namespace dbeel
