// lsm_tree_host.cc -- the host side of the drop-in: file protocol around the GPU merge core.
// See include/dbeel_tree.h for the reference functions each entry point mirrors.
#include <errno.h>
#include <fcntl.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/statvfs.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <filesystem>
#include <thread>
#include <map>
#include <string>
#include <string_view>
#include <unordered_set>
#include <vector>

#include "../../../include/dbeel_tree.h"
#include "../device_fns.cuh" // the scalar arithmetic the kernels use, compiled for the host here (murmur3_32, ring_owner)

namespace fs = std::filesystem;

namespace {

constexpr int kIndexPadding = 20; // mod.rs:21
const char *kData = "data", *kIndex = "index", *kBloom = "bloom", *kMemtable = "memtable";
const char *kCompactData = "compact_data", *kCompactIndex = "compact_index", *kCompactBloom = "compact_bloom",
           *kCompactAction = "compact_action";

struct SSTable {
    uint64_t index;
    uint64_t size; // entries
};

std::string file_path(const std::string &dir, uint64_t index, const char *ext) { // lsm_tree.rs:284-288
    char name[64];
    snprintf(name, sizeof name, "%0*llu.%s", kIndexPadding, (unsigned long long)index, ext);
    return (fs::path(dir) / name).string();
}

// "^(\d+)\.<ext>$" (lsm_tree.rs:306-310)
bool parse_name(const std::string &name, const char *ext, uint64_t *index) {
    size_t dot = name.find('.');
    if (dot == std::string::npos || dot == 0 || name.substr(dot + 1) != ext) return false;
    uint64_t v = 0;
    for (size_t i = 0; i < dot; i++) {
        if (name[i] < '0' || name[i] > '9') return false;
        v = v * 10 + (uint64_t)(name[i] - '0');
    }
    *index = v;
    return true;
}

struct PinnedBuf { // dbeel_host_alloc'ed: PCIe transfers at full speed
    uint8_t *p = nullptr;
    uint64_t len = 0;
    PinnedBuf() = default;
    explicit PinnedBuf(uint64_t n) : p(static_cast<uint8_t *>(dbeel_host_alloc(n ? n : 1))), len(n) {}
    PinnedBuf(const PinnedBuf &) = delete;
    PinnedBuf &operator=(const PinnedBuf &) = delete;
    PinnedBuf(PinnedBuf &&o) noexcept : p(o.p), len(o.len) { o.p = nullptr; }
    PinnedBuf &operator=(PinnedBuf &&o) noexcept {
        if (this != &o) { dbeel_host_free(p); p = o.p; len = o.len; o.p = nullptr; }
        return *this;
    }
    ~PinnedBuf() { dbeel_host_free(p); }
};

// bincode (fixint, little-endian) writers for the CompactionAction journal (lsm_tree.rs:73-77)
void put_u64(std::string &b, uint64_t v) { b.append(reinterpret_cast<const char *>(&v), 8); }
void put_path(std::string &b, const std::string &p) { put_u64(b, p.size()); b += p; } // PathBuf serializes as str

bool get_u64(const std::string &b, size_t &pos, uint64_t *v) {
    if (b.size() - pos < 8) return false;
    memcpy(v, b.data() + pos, 8);
    pos += 8;
    return true;
}
bool get_path(const std::string &b, size_t &pos, std::string *p) {
    uint64_t n;
    if (!get_u64(b, pos, &n) || b.size() - pos < n) return false;
    p->assign(b, pos, n);
    pos += n;
    return true;
}

} // namespace

struct dbeel_tree {
    std::string dir;
    dbeel_engine *engine = nullptr;
    uint64_t bloom_min_size = DBEEL_DEFAULT_BLOOM_MIN_SIZE;
    std::vector<SSTable> sstables; // ascending by index (lsm_tree.rs:1136)
    uint64_t write_sstable_index = 0;
    std::string err;
    dbeel_page_sink page_sink = nullptr; // EntryWriter's page-cache write-through (entry_writer.rs:94-156), if the caller wants it
    void *page_ctx = nullptr;
};

namespace {

int io_fail(dbeel_tree *t, const std::string &what) {
    t->err = what + ": " + strerror(errno);
    return DBEEL_ERR_IO;
}

// File <-> pinned memory in 32 MiB pieces spread over a few threads (pread / pwrite): one thread moves a RAM-resident
// file at memcpy speed, which is a fraction of what the PCIe link behind the pinned buffer takes (N3: the storage edge).
constexpr uint64_t kIoChunk = 32ull << 20;

int io_threads() {
    static const int n = [] {
        if (const char *v = getenv("DBEEL_IO_THREADS")) return std::max(1, atoi(v));
        const unsigned hw = std::thread::hardware_concurrency();
        return (int)std::min(8u, std::max(1u, hw / 2));
    }();
    return n;
}

// moves [0, len) between fd and mem; returns 0 or an errno
int move_chunks(int fd, uint8_t *mem, uint64_t len, bool reading) {
    const uint64_t n_chunks = (len + kIoChunk - 1) / kIoChunk;
    std::atomic<uint64_t> next{0};
    std::atomic<int> err{0};
    auto work = [&]() {
        for (uint64_t c = next.fetch_add(1); c < n_chunks && !err.load(); c = next.fetch_add(1)) {
            uint64_t pos = c * kIoChunk;
            const uint64_t end = std::min(len, pos + kIoChunk);
            while (pos < end) {
                const ssize_t r = reading ? pread(fd, mem + pos, end - pos, (off_t)pos) : pwrite(fd, mem + pos, end - pos, (off_t)pos);
                if (r < 0 && errno == EINTR) continue;
                if (r <= 0) { err.store(r < 0 ? errno : EIO); return; }
                pos += (uint64_t)r;
            }
        }
    };
    const int nt = (int)std::min<uint64_t>((uint64_t)io_threads(), n_chunks);
    std::vector<std::thread> pool;
    for (int i = 1; i < nt; i++) pool.emplace_back(work);
    work();
    for (auto &th : pool) th.join();
    return err.load();
}

int read_file(dbeel_tree *t, const std::string &path, PinnedBuf *out) {
    int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) return io_fail(t, "open " + path);
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); return io_fail(t, "fstat " + path); }
    PinnedBuf buf((uint64_t)st.st_size);
    if (!buf.p) { close(fd); t->err = "dbeel_host_alloc failed"; return DBEEL_ERR_NOMEM; }
    const int e = move_chunks(fd, buf.p, buf.len, true);
    close(fd);
    if (e) { errno = e; return io_fail(t, "read " + path); }
    *out = std::move(buf);
    return DBEEL_OK;
}

int write_file(dbeel_tree *t, const std::string &path, const void *data, uint64_t len) {
    int fd = open(path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return io_fail(t, "create " + path);
    const int e = move_chunks(fd, const_cast<uint8_t *>(static_cast<const uint8_t *>(data)), len, false);
    if (e) { close(fd); errno = e; return io_fail(t, "write " + path); }
    if (close(fd) != 0) return io_fail(t, "close " + path);
    return DBEEL_OK;
}

bool exists(const std::string &p) { struct stat st; return stat(p.c_str(), &st) == 0; }

struct CompactionAction {
    std::vector<std::pair<std::string, std::string>> renames;
    std::vector<std::string> deletes;
};

std::string encode_action(const CompactionAction &a) {
    std::string b;
    put_u64(b, a.renames.size());
    for (auto &r : a.renames) { put_path(b, r.first); put_path(b, r.second); }
    put_u64(b, a.deletes.size());
    for (auto &d : a.deletes) put_path(b, d);
    return b;
}

bool decode_action(const std::string &b, CompactionAction *a) {
    size_t pos = 0;
    uint64_t n;
    if (!get_u64(b, pos, &n)) return false;
    for (uint64_t i = 0; i < n; i++) {
        std::string s, d;
        if (!get_path(b, pos, &s) || !get_path(b, pos, &d)) return false;
        a->renames.emplace_back(std::move(s), std::move(d));
    }
    if (!get_u64(b, pos, &n)) return false;
    for (uint64_t i = 0; i < n; i++) {
        std::string d;
        if (!get_path(b, pos, &d)) return false;
        a->deletes.push_back(std::move(d));
    }
    return pos == b.size(); // reject_trailing_bytes
}

// run_compaction_action (lsm_tree.rs:576-590): deletes first, then the renames whose source exists
int run_action(dbeel_tree *t, const CompactionAction &a) {
    for (auto &d : a.deletes)
        if (exists(d)) unlink(d.c_str()); // remove_file_log_on_err: failure is not fatal
    for (auto &r : a.renames)
        if (exists(r.first) && rename(r.first.c_str(), r.second.c_str()) != 0) return io_fail(t, "rename " + r.first);
    return DBEEL_OK;
}

} // namespace

extern "C" {

int dbeel_tree_open(const char *dir, dbeel_engine *engine, uint64_t bloom_min_size, dbeel_tree **out) {
    if (!dir || !engine || !out) return DBEEL_ERR_INVALID_ARG;
    *out = nullptr;
    auto *t = new (std::nothrow) dbeel_tree();
    if (!t) return DBEEL_ERR_NOMEM;
    t->dir = dir;
    t->engine = engine;
    t->bloom_min_size = bloom_min_size;
    std::error_code ec;
    fs::create_directories(t->dir, ec); // lsm_tree.rs:415-420
    // replay compaction journals (lsm_tree.rs:424-438).  The reference re-creates its reader on
    // every loop iteration and would spin on a valid journal; each journal holds one action.
    std::vector<std::string> journals, names;
    for (auto &de : fs::directory_iterator(t->dir, ec)) names.push_back(de.path().filename().string());
    uint64_t idx;
    for (auto &n : names)
        if (parse_name(n, kCompactAction, &idx)) journals.push_back((fs::path(t->dir) / n).string());
    for (auto &j : journals) {
        std::string buf; // journals are tiny: plain memory, no pinned allocation (works without a GPU)
        {
            int fd = open(j.c_str(), O_RDONLY);
            if (fd < 0) { int rc = io_fail(t, "open " + j); delete t; return rc; }
            char tmp[4096];
            ssize_t r;
            while ((r = read(fd, tmp, sizeof tmp)) > 0) buf.append(tmp, (size_t)r);
            close(fd);
        }
        CompactionAction a;
        if (decode_action(buf, &a)) {
            int rc = run_action(t, a);
            if (rc) { delete t; return rc; }
        }
        unlink(j.c_str());
    }
    // discover SSTables (lsm_tree.rs:440-459): size = len(.index) / 16
    names.clear();
    for (auto &de : fs::directory_iterator(t->dir, ec)) names.push_back(de.path().filename().string());
    std::vector<uint64_t> indices;
    for (auto &n : names)
        if (parse_name(n, kData, &idx)) indices.push_back(idx);
    std::sort(indices.begin(), indices.end());
    for (uint64_t i : indices) {
        struct stat st;
        std::string ip = file_path(t->dir, i, kIndex);
        if (stat(ip.c_str(), &st) != 0) { int rc = io_fail(t, "stat " + ip); delete t; return rc; }
        t->sstables.push_back({i, (uint64_t)st.st_size / DBEEL_INDEX_ENTRY_SIZE});
    }
    // lsm_tree.rs:461-465
    t->write_sstable_index = indices.empty() ? 0 : indices.back() + 2 - (indices.back() & 1);
    *out = t;
    return DBEEL_OK;
}

void dbeel_tree_close(dbeel_tree *t) { delete t; }

uint32_t dbeel_tree_sstables(const dbeel_tree *t, uint64_t *indices, uint64_t *sizes, uint32_t cap) {
    if (!t) return 0;
    for (uint32_t i = 0; i < t->sstables.size() && i < cap; i++) {
        if (indices) indices[i] = t->sstables[i].index;
        if (sizes) sizes[i] = t->sstables[i].size;
    }
    return (uint32_t)t->sstables.size();
}

uint64_t dbeel_tree_write_sstable_index(const dbeel_tree *t) { return t ? t->write_sstable_index : 0; }

const char *dbeel_tree_last_error(const dbeel_tree *t) { return t ? t->err.c_str() : "null tree"; }

// EntryWriter's write-through (entry_writer.rs:94-156) for a finished SSTable: the page-cache `set` calls the reference makes
// while it writes the same entries one by one, in the same order.  After entry i the .data stream holds off_i + full_size_i
// bytes and the .index stream 16 (i + 1): a 4 KiB page is handed over the moment its last byte is written (write_to_cache,
// :115-137), data before index inside one write(); close() hands over the two zero-padded tail pages, data first (:140-156).
int dbeel_out_pages(const void *data, uint64_t data_len, const void *index, uint64_t index_len, uint64_t files_index, dbeel_page_sink sink,
                    void *ctx) {
    if (!sink || (data_len && !data) || (index_len && !index)) return DBEEL_ERR_INVALID_ARG;
    constexpr uint64_t kPage = 4096;
    const uint8_t *d = static_cast<const uint8_t *>(data), *ix = static_cast<const uint8_t *>(index);
    const uint64_t n = index_len / DBEEL_INDEX_ENTRY_SIZE;
    uint64_t dw = 0, iw = 0; // data_written / index_written
    for (uint64_t i = 0; i < n; i++) {
        uint32_t fs;
        memcpy(&fs, ix + 16 * i + 12, 4);
        const uint64_t dend = dw + fs;
        if (dend > data_len) return DBEEL_ERR_INVALID_ARG;
        for (uint64_t pg = dw / kPage; (pg + 1) * kPage <= dend; pg++) sink(ctx, DBEEL_FILE_DATA, files_index, pg * kPage, d + pg * kPage);
        dw = dend;
        const uint64_t iend = iw + 16;
        if (iend % kPage == 0) sink(ctx, DBEEL_FILE_INDEX, files_index, iend - kPage, ix + iend - kPage);
        iw = iend;
    }
    uint8_t tail[kPage];
    if (dw % kPage) {
        memset(tail, 0, kPage);
        memcpy(tail, d + dw - dw % kPage, dw % kPage);
        sink(ctx, DBEEL_FILE_DATA, files_index, dw - dw % kPage, tail);
    }
    if (iw % kPage) {
        memset(tail, 0, kPage);
        memcpy(tail, ix + iw - iw % kPage, iw % kPage);
        sink(ctx, DBEEL_FILE_INDEX, files_index, iw - iw % kPage, tail);
    }
    return DBEEL_OK;
}

void dbeel_tree_set_page_sink(dbeel_tree *t, dbeel_page_sink sink, void *ctx) {
    if (!t) return;
    t->page_sink = sink;
    t->page_ctx = ctx;
}

// Everything LSMTree::compact does once the compact_* files are complete (lsm_tree.rs:1078-1155): the CompactionAction
// journal, the renames, the sstable-list swap, the deletes.
static int commit_written(dbeel_tree *t, const uint64_t *indices_to_compact, uint32_t n, uint64_t output_index, uint64_t items_written) {
    int rc;
    const std::string cdata = file_path(t->dir, output_index, kCompactData), cindex = file_path(t->dir, output_index, kCompactIndex),
                      cbloom = file_path(t->dir, output_index, kCompactBloom);
    // lsm_tree.rs:1078-1105: journal
    CompactionAction action;
    action.renames = {{cdata, file_path(t->dir, output_index, kData)},
                      {cindex, file_path(t->dir, output_index, kIndex)},
                      {cbloom, file_path(t->dir, output_index, kBloom)}};
    for (uint32_t i = 0; i < n; i++)
        for (const char *ext : {kData, kIndex, kBloom}) action.deletes.push_back(file_path(t->dir, indices_to_compact[i], ext));
    const std::string journal = file_path(t->dir, output_index, kCompactAction);
    const std::string enc = encode_action(action);
    rc = write_file(t, journal, enc.data(), enc.size());
    if (rc) return rc;
    // lsm_tree.rs:1107-1111: renames whose source exists (no bloom -> that rename is skipped)
    for (auto &r : action.renames)
        if (exists(r.first) && rename(r.first.c_str(), r.second.c_str()) != 0) return io_fail(t, "rename " + r.first);
    // lsm_tree.rs:1113-1139: swap the sstable list
    std::vector<SSTable> next;
    for (auto &s : t->sstables)
        if (std::find(indices_to_compact, indices_to_compact + n, s.index) == indices_to_compact + n) next.push_back(s);
    next.push_back({output_index, items_written});
    std::sort(next.begin(), next.end(), [](const SSTable &a, const SSTable &b) { return a.index < b.index; });
    t->sstables.swap(next);
    // lsm_tree.rs:1147-1153: delete the inputs, then the journal
    for (auto &d : action.deletes)
        if (exists(d)) unlink(d.c_str());
    unlink(journal.c_str());
    return DBEEL_OK;
}

// ... for a job whose output sits in host buffers: the compact_* files first (lsm_tree.rs:995-1000,1068-1076), then the rest.
static int commit_compaction(dbeel_tree *t, const uint64_t *indices_to_compact, uint32_t n, uint64_t output_index, const void *data,
                             uint64_t data_len, const void *index, uint64_t index_len, const void *bloom, uint64_t bloom_len,
                             uint64_t items_written) {
    const std::string cdata = file_path(t->dir, output_index, kCompactData), cindex = file_path(t->dir, output_index, kCompactIndex),
                      cbloom = file_path(t->dir, output_index, kCompactBloom);
    int rc = write_file(t, cdata, data, data_len);
    if (!rc) rc = write_file(t, cindex, index, index_len);
    if (!rc && bloom_len) rc = write_file(t, cbloom, bloom, bloom_len);
    if (rc) return rc;
    // entry_writer.rs:94-95: the writer mirrors what it writes into the shard's page cache under the NEW files_index
    if (t->page_sink) dbeel_out_pages(data, data_len, index, index_len, output_index, t->page_sink, t->page_ctx);
    return commit_written(t, indices_to_compact, n, output_index, items_written);
}

// The file edge of a streamed compaction (dbeel_compact_stream): the inputs' descriptors stand where the reference holds
// DmaStreamReaders (lsm_tree.rs:984-991), the compact_* descriptors where it holds EntryWriter's DMA files (:995-1000).
namespace {
// Output side: several threads pwrite()-ing into ONE file take turns on its inode lock (measured on tmpfs: 3.2 GB/s however
// many writers -- a cfg2 job's 2 GB then cost 0.45 s of a 0.52 s call), so each output is sized to its upper bound, mapped
// shared, and the writer threads copy into the mapping: page faults of different threads proceed in parallel.  The file is cut
// to its final length afterwards.  (A file system that refuses the mapping falls back to pwrite.)
struct StreamFiles {
    std::vector<int> data_fd, index_fd;
    int out_fd[4] = {-1, -1, -1, -1}; // by DBEEL_STREAM_* kind
    uint8_t *out_map[4] = {nullptr, nullptr, nullptr, nullptr};
    uint64_t out_cap[4] = {0, 0, 0, 0};
    std::atomic<int> saved_errno{0};
    void unmap() {
        for (int k = 0; k < 4; k++)
            if (out_map[k]) { munmap(out_map[k], out_cap[k]); out_map[k] = nullptr; }
    }
    ~StreamFiles() {
        unmap();
        for (int fd : data_fd) if (fd >= 0) close(fd);
        for (int fd : index_fd) if (fd >= 0) close(fd);
        for (int fd : out_fd) if (fd >= 0) close(fd);
    }
};

int stream_read(void *ctx, uint32_t run, uint32_t kind, uint64_t off, uint64_t len, void *dst) {
    auto *f = static_cast<StreamFiles *>(ctx);
    const int fd = kind == DBEEL_STREAM_DATA ? f->data_fd[run] : f->index_fd[run];
    uint8_t *p = static_cast<uint8_t *>(dst);
    while (len) {
        const ssize_t r = pread(fd, p, len, (off_t)off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) { f->saved_errno.store(r < 0 ? errno : EIO); return DBEEL_ERR_IO; }
        p += r; off += (uint64_t)r; len -= (uint64_t)r;
    }
    return 0;
}

int stream_write(void *ctx, uint32_t kind, uint64_t off, const void *src, uint64_t len) {
    auto *f = static_cast<StreamFiles *>(ctx);
    if (kind < 1 || kind > 3) return DBEEL_ERR_INVALID_ARG;
    if (f->out_map[kind]) {
        if (off > f->out_cap[kind] || len > f->out_cap[kind] - off) return DBEEL_ERR_CAPACITY;
        memcpy(f->out_map[kind] + off, src, len);
        return 0;
    }
    const uint8_t *p = static_cast<const uint8_t *>(src);
    while (len) {
        const ssize_t r = pwrite(f->out_fd[kind], p, len, (off_t)off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) { f->saved_errno.store(r < 0 ? errno : EIO); return DBEEL_ERR_IO; }
        p += r; off += (uint64_t)r; len -= (uint64_t)r;
    }
    return 0;
}

bool stream_maps() { // DBEEL_STREAM_MMAP=0: outputs through pwrite (A/B switch)
    const char *v = getenv("DBEEL_STREAM_MMAP");
    return !v || atoi(v) != 0;
}

bool tree_streams() { // DBEEL_TREE_STREAM=0: every compaction takes the whole-buffer path (A/B switch, read per call)
    const char *v = getenv("DBEEL_TREE_STREAM");
    return !v || atoi(v) != 0;
}
} // namespace

// dbeel_tree_compact, files streamed through the engine's pinned rings: nothing is held whole in memory
static int tree_compact_streamed(dbeel_tree *t, const uint64_t *indices_to_compact, uint32_t n, uint64_t output_index, int keep_tombstones,
                                 const uint8_t *bloom_seed) {
    StreamFiles f;
    f.data_fd.assign(n, -1);
    f.index_fd.assign(n, -1);
    std::vector<dbeel_run> runs(n);
    for (uint32_t i = 0; i < n; i++) { // lsm_tree.rs:956-993: open the inputs
        const std::string dp = file_path(t->dir, indices_to_compact[i], kData), ip = file_path(t->dir, indices_to_compact[i], kIndex);
        if (!exists(dp) || !exists(ip)) { t->err = "no such sstable: " + dp; return DBEEL_ERR_NO_SSTABLE; }
        f.data_fd[i] = open(dp.c_str(), O_RDONLY);
        f.index_fd[i] = open(ip.c_str(), O_RDONLY);
        struct stat sd, si;
        if (f.data_fd[i] < 0 || f.index_fd[i] < 0 || fstat(f.data_fd[i], &sd) != 0 || fstat(f.index_fd[i], &si) != 0) return io_fail(t, "open " + dp);
        runs[i] = dbeel_run{nullptr, (uint64_t)sd.st_size, nullptr, (uint64_t)si.st_size};
    }
    // lsm_tree.rs:995-1000: the compact_* files
    const std::string cpath[4] = {"", file_path(t->dir, output_index, kCompactData), file_path(t->dir, output_index, kCompactIndex),
                                  file_path(t->dir, output_index, kCompactBloom)};
    auto drop_outputs = [&]() { for (int k = 1; k <= 3; k++) unlink(cpath[k].c_str()); };
    for (int k = 1; k <= 3; k++) {
        f.out_fd[k] = open(cpath[k].c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644); // read-write: a shared writable mapping needs it
        if (f.out_fd[k] < 0) { const int rc = io_fail(t, "create " + cpath[k]); drop_outputs(); return rc; }
    }
    dbeel_compact_opts opts;
    opts.keep_tombstones = keep_tombstones;
    opts.flags = 0;
    opts.bloom_min_size = t->bloom_min_size;
    opts.bloom_fp = DBEEL_DEFAULT_BLOOM_FP;
    opts.bloom_seed = bloom_seed;
    if (stream_maps()) { // size every output to its bound and map it (see StreamFiles)
        uint64_t cap[4] = {0, 0, 0, 0};
        // A store into a mapped page the file system cannot back raises SIGBUS where pwrite would return ENOSPC: only map when
        // the volume has room for the bounds (plus slack); otherwise the writers go through pwrite and a full disk is an error code.
        struct statvfs vfs;
        bool room = false;
        if (dbeel_compact_bound(runs.data(), n, &opts, &cap[1], &cap[2], &cap[3]) == DBEEL_OK && fstatvfs(f.out_fd[1], &vfs) == 0)
            room = (uint64_t)vfs.f_bavail * (uint64_t)vfs.f_frsize >= cap[1] + cap[2] + cap[3] + (64ull << 20);
        if (room) {
            for (int k = 1; k <= 3; k++) {
                if (!cap[k] || ftruncate(f.out_fd[k], (off_t)cap[k]) != 0) continue;
                void *m = mmap(nullptr, cap[k], PROT_READ | PROT_WRITE, MAP_SHARED, f.out_fd[k], 0);
                if (m == MAP_FAILED) { if (ftruncate(f.out_fd[k], 0) != 0) {} continue; }
                f.out_map[k] = static_cast<uint8_t *>(m);
                f.out_cap[k] = cap[k];
            }
        }
    }
    dbeel_stream_io io{stream_read, stream_write, &f};
    dbeel_out out = {};
    // lsm_tree.rs:1002-1076 -- the merge core, on the GPU
    int rc = dbeel_compact_stream(t->engine, runs.data(), n, &opts, &io, &out);
    if (rc) {
        if (rc == DBEEL_ERR_IO) { errno = f.saved_errno.load(); io_fail(t, "streamed compaction"); }
        else t->err = dbeel_last_error(t->engine);
        drop_outputs();
        return rc;
    }
    f.unmap();
    const uint64_t lens[4] = {0, out.data_len, out.index_len, out.bloom_len};
    for (int k = 1; k <= 3; k++) { // cut to the final length (the files were sized to their bounds; a redone job may have written past it)
        const bool cut = ftruncate(f.out_fd[k], (off_t)lens[k]) == 0;
        const bool closed = close(f.out_fd[k]) == 0;
        f.out_fd[k] = -1;
        if (!cut || !closed) { rc = io_fail(t, "close " + cpath[k]); drop_outputs(); return rc; }
    }
    if (!out.bloom_len) unlink(cpath[3].c_str()); // no filter: no .bloom file (lsm_tree.rs:1068-1076)
    return commit_written(t, indices_to_compact, n, output_index, out.items_written);
}


int dbeel_tree_compact(dbeel_tree *t, const uint64_t *indices_to_compact, uint32_t n, uint64_t output_index,
                       int keep_tombstones, const uint8_t *bloom_seed) {
    if (!t || (n && !indices_to_compact)) return DBEEL_ERR_INVALID_ARG;
    t->err.clear();
    // The default: stream the files through the engine.  A page sink needs the finished SSTable in memory (dbeel_out_pages
    // replays the writer's `set` calls in entry order), so a tree with one installed takes the whole-buffer path below.
    if (tree_streams() && !t->page_sink) return tree_compact_streamed(t, indices_to_compact, n, output_index, keep_tombstones, bloom_seed);
    // lsm_tree.rs:956-993: open the inputs (here: read them whole into pinned memory)
    std::vector<PinnedBuf> data(n), index(n);
    std::vector<dbeel_run> runs(n);
    for (uint32_t i = 0; i < n; i++) {
        std::string dp = file_path(t->dir, indices_to_compact[i], kData), ip = file_path(t->dir, indices_to_compact[i], kIndex);
        if (!exists(dp) || !exists(ip)) { t->err = "no such sstable: " + dp; return DBEEL_ERR_NO_SSTABLE; }
        int rc = read_file(t, dp, &data[i]);
        if (!rc) rc = read_file(t, ip, &index[i]);
        if (rc) return rc;
        runs[i] = dbeel_run{data[i].p, data[i].len, index[i].p, index[i].len};
    }
    dbeel_compact_opts opts;
    opts.keep_tombstones = keep_tombstones;
    opts.flags = 0;
    opts.bloom_min_size = t->bloom_min_size;
    opts.bloom_fp = DBEEL_DEFAULT_BLOOM_FP;
    opts.bloom_seed = bloom_seed;
    uint64_t dc, ic, bc;
    int rc = dbeel_compact_bound(runs.data(), n, &opts, &dc, &ic, &bc);
    if (rc) return rc;
    PinnedBuf od(dc), oi(ic), ob(bc);
    if (!od.p || !oi.p || !ob.p) { t->err = "dbeel_host_alloc failed"; return DBEEL_ERR_NOMEM; }
    dbeel_out out{od.p, dc, 0, oi.p, ic, 0, bc ? ob.p : nullptr, bc, 0, 0};
    // lsm_tree.rs:1002-1076 -- the merge core, on the GPU
    rc = dbeel_compact(t->engine, runs.data(), n, &opts, &out);
    if (rc) { t->err = dbeel_last_error(t->engine); return rc; }

    return commit_compaction(t, indices_to_compact, n, output_index, od.p, out.data_len, oi.p, out.index_len, ob.p, out.bloom_len,
                             out.items_written);
}

int dbeel_tree_compact_many(dbeel_tree *t, const uint64_t *members, const uint32_t *group_start, uint32_t n_groups,
                            const uint64_t *output_index, const int32_t *keep_tombstones, const uint8_t *bloom_seeds) {
    if (!t || (n_groups && (!members || !group_start || !output_index || !keep_tombstones))) return DBEEL_ERR_INVALID_ARG;
    t->err.clear();
    const uint32_t total = n_groups ? group_start[n_groups] : 0;
    std::vector<PinnedBuf> data(total), index(total);
    std::vector<dbeel_run> runs(total);
    for (uint32_t i = 0; i < total; i++) { // lsm_tree.rs:956-993 for every group
        std::string dp = file_path(t->dir, members[i], kData), ip = file_path(t->dir, members[i], kIndex);
        if (!exists(dp) || !exists(ip)) { t->err = "no such sstable: " + dp; return DBEEL_ERR_NO_SSTABLE; }
        int rc = read_file(t, dp, &data[i]);
        if (!rc) rc = read_file(t, ip, &index[i]);
        if (rc) return rc;
        runs[i] = dbeel_run{data[i].p, data[i].len, index[i].p, index[i].len};
    }
    std::vector<dbeel_job> jobs(n_groups);
    for (uint32_t g = 0; g < n_groups; g++)
        jobs[g] = dbeel_job{runs.data() + group_start[g], group_start[g + 1] - group_start[g], keep_tombstones[g],
                            bloom_seeds ? bloom_seeds + 32 * g : nullptr};
    uint64_t dc, ic, bc;
    int rc = dbeel_compact_many_bound(jobs.data(), n_groups, t->bloom_min_size, DBEEL_DEFAULT_BLOOM_FP, &dc, &ic, &bc);
    if (rc) return rc;
    PinnedBuf od(dc), oi(ic), ob(bc);
    if (!od.p || !oi.p || !ob.p) { t->err = "dbeel_host_alloc failed"; return DBEEL_ERR_NOMEM; }
    dbeel_out out{od.p, dc, 0, oi.p, ic, 0, bc ? ob.p : nullptr, bc, 0, 0};
    std::vector<dbeel_job_result> res(n_groups);
    rc = dbeel_compact_many(t->engine, jobs.data(), n_groups, t->bloom_min_size, DBEEL_DEFAULT_BLOOM_FP, &out, res.data());
    if (rc) { t->err = dbeel_last_error(t->engine); return rc; }
    for (uint32_t g = 0; g < n_groups; g++) { // the commit protocol, group by group, in the picker's order
        const dbeel_job_result &r = res[g];
        rc = commit_compaction(t, members + group_start[g], group_start[g + 1] - group_start[g], output_index[g], od.p + r.data_off,
                               r.data_len, oi.p + r.index_off, r.index_len, ob.p + r.bloom_off, r.bloom_len, r.items_written);
        if (rc) return rc;
    }
    return DBEEL_OK;
}

int dbeel_tree_flush(dbeel_tree *t, const dbeel_run *batch, uint64_t *written_index, uint64_t *items_written) {
    if (!t || !batch) return DBEEL_ERR_INVALID_ARG;
    t->err.clear();
    if (batch->index_len < DBEEL_INDEX_ENTRY_SIZE) return DBEEL_OK; // flush of an empty memtable is a no-op (lsm_tree.rs:850-852)
    PinnedBuf od(batch->data_len), oi(batch->index_len);
    if (!od.p || !oi.p) { t->err = "dbeel_host_alloc failed"; return DBEEL_ERR_NOMEM; }
    dbeel_out out{od.p, batch->data_len, 0, oi.p, batch->index_len / 16 * 16, 0, nullptr, 0, 0, 0};
    int rc = dbeel_flush(t->engine, batch, &out);
    if (rc) { t->err = dbeel_last_error(t->engine); return rc; }
    const uint64_t idx = t->write_sstable_index; // lsm_tree.rs:875-880
    rc = write_file(t, file_path(t->dir, idx, kData), od.p, out.data_len);
    if (!rc) rc = write_file(t, file_path(t->dir, idx, kIndex), oi.p, out.index_len);
    if (!rc && t->page_sink) dbeel_out_pages(od.p, out.data_len, oi.p, out.index_len, idx, t->page_sink, t->page_ctx);
    if (rc) return rc;
    t->sstables.push_back({idx, out.items_written}); // lsm_tree.rs:903-915 (bloom: None)
    t->write_sstable_index = idx + 2;
    if (written_index) *written_index = idx;
    if (items_written) *items_written = out.items_written;
    return DBEEL_OK;
}

int dbeel_tree_get_many(dbeel_tree *t, const void *keys, const uint64_t *key_offsets, uint64_t n_keys, uint32_t mode,
                        dbeel_lookup_result *results) {
    if (!t || (n_keys && (!key_offsets || !results))) return DBEEL_ERR_INVALID_ARG;
    t->err.clear();
    // get_entry walks `self.sstables` (ascending index) newest first (lsm_tree.rs:686-688); every table brings its
    // .bloom if one exists on disk (SSTable::new_with_bloom_read, :94-101)
    const size_t n = t->sstables.size();
    std::vector<PinnedBuf> data(n), index(n), bloom(n);
    std::vector<dbeel_table> tables(n);
    for (size_t i = 0; i < n; i++) {
        const uint64_t idx = t->sstables[i].index;
        int rc = read_file(t, file_path(t->dir, idx, kData), &data[i]);
        if (!rc) rc = read_file(t, file_path(t->dir, idx, kIndex), &index[i]);
        const std::string bp = file_path(t->dir, idx, kBloom);
        if (!rc && exists(bp)) rc = read_file(t, bp, &bloom[i]);
        if (rc) return rc;
        tables[i] = dbeel_table{data[i].p, data[i].len, index[i].p, index[i].len, bloom[i].len ? bloom[i].p : nullptr, bloom[i].len};
    }
    int rc = dbeel_get_many(t->engine, tables.data(), (uint32_t)n, keys, key_offsets, n_keys, mode, results);
    if (rc) t->err = dbeel_last_error(t->engine);
    return rc;
}

int dbeel_tree_scan_ranges(dbeel_tree *t, const dbeel_run *memtables, uint32_t n_memtables, const dbeel_hash_range *ranges,
                           uint32_t n_ranges, uint32_t mode, dbeel_out *out, dbeel_flush_table *per_range, dbeel_scan_stop *stop) {
    if (!t || (n_memtables && !memtables) || !stop) return DBEEL_ERR_INVALID_ARG;
    t->err.clear();
    // AsyncIter walks `self.sstables` (ascending index) and then the memtables (lsm_tree.rs:155-173, 213-282); an empty
    // memtable yields nothing and is left out (an empty table in front of the engine stops the scan)
    const size_t n = t->sstables.size();
    std::vector<PinnedBuf> data(n), index(n);
    std::vector<dbeel_run> tables;
    std::vector<int32_t> position; // tables[k] is the caller's table position[k]: SSTables, then memtables
    for (size_t i = 0; i < n; i++) {
        const uint64_t idx = t->sstables[i].index;
        int rc = read_file(t, file_path(t->dir, idx, kData), &data[i]);
        if (!rc) rc = read_file(t, file_path(t->dir, idx, kIndex), &index[i]);
        if (rc) return rc;
        tables.push_back(dbeel_run{data[i].p, data[i].len, index[i].p, index[i].len});
        position.push_back((int32_t)i);
    }
    for (uint32_t m = 0; m < n_memtables; m++) {
        if (memtables[m].index_len < DBEEL_INDEX_ENTRY_SIZE) continue;
        tables.push_back(memtables[m]);
        position.push_back((int32_t)(n + m));
    }
    int rc = dbeel_scan_ranges(t->engine, tables.data(), (uint32_t)tables.size(), ranges, n_ranges, mode, out, per_range, stop);
    if (stop->table >= 0 && (size_t)stop->table < position.size()) stop->table = position[stop->table];
    if (rc) t->err = dbeel_last_error(t->engine);
    return rc;
}

// The file edge of a streamed scan (dbeel_scan_ranges_stream): the tables' descriptors (or the caller's memtables) on the
// way in, two files per range on the way out, written like StreamFiles' outputs (mapped when the volume has room, else pwrite).
namespace {
struct ScanFiles {
    std::vector<int> data_fd, index_fd;   // -1: a memtable, read from `mem`
    std::vector<const dbeel_run *> mem;
    std::vector<std::string> out_path;    // [2 r] = <r>.data, [2 r + 1] = <r>.index
    std::vector<int> out_fd;
    std::vector<uint8_t *> out_map;
    std::vector<uint64_t> out_cap;
    std::atomic<int> saved_errno{0};
    void unmap() {
        for (size_t k = 0; k < out_map.size(); k++)
            if (out_map[k]) { munmap(out_map[k], out_cap[k]); out_map[k] = nullptr; }
    }
    ~ScanFiles() {
        unmap();
        for (int fd : data_fd) if (fd >= 0) close(fd);
        for (int fd : index_fd) if (fd >= 0) close(fd);
        for (int fd : out_fd) if (fd >= 0) close(fd);
    }
};

int scan_read(void *ctx, uint32_t table, uint32_t kind, uint64_t off, uint64_t len, void *dst) {
    auto *f = static_cast<ScanFiles *>(ctx);
    if (table >= f->mem.size()) return DBEEL_ERR_INVALID_ARG;
    if (const dbeel_run *m = f->mem[table]) {
        const uint64_t n = kind == DBEEL_STREAM_DATA ? m->data_len : m->index_len;
        if (off > n || len > n - off) return DBEEL_ERR_INVALID_ARG;
        memcpy(dst, static_cast<const uint8_t *>(kind == DBEEL_STREAM_DATA ? m->data : m->index) + off, len);
        return 0;
    }
    const int fd = kind == DBEEL_STREAM_DATA ? f->data_fd[table] : f->index_fd[table];
    uint8_t *p = static_cast<uint8_t *>(dst);
    while (len) {
        const ssize_t r = pread(fd, p, len, (off_t)off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) { f->saved_errno.store(r < 0 ? errno : EIO); return DBEEL_ERR_IO; }
        p += r; off += (uint64_t)r; len -= (uint64_t)r;
    }
    return 0;
}

int scan_write(void *ctx, uint32_t range, uint32_t kind, uint64_t off, const void *src, uint64_t len) {
    auto *f = static_cast<ScanFiles *>(ctx);
    if (kind != DBEEL_STREAM_DATA && kind != DBEEL_STREAM_INDEX) return DBEEL_ERR_INVALID_ARG;
    const size_t k = 2ull * range + (kind == DBEEL_STREAM_INDEX ? 1 : 0);
    if (k >= f->out_fd.size()) return DBEEL_ERR_INVALID_ARG;
    if (f->out_map[k]) {
        if (off > f->out_cap[k] || len > f->out_cap[k] - off) return DBEEL_ERR_CAPACITY;
        memcpy(f->out_map[k] + off, src, len);
        return 0;
    }
    const uint8_t *p = static_cast<const uint8_t *>(src);
    while (len) {
        const ssize_t r = pwrite(f->out_fd[k], p, len, (off_t)off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) { f->saved_errno.store(r < 0 ? errno : EIO); return DBEEL_ERR_IO; }
        p += r; off += (uint64_t)r; len -= (uint64_t)r;
    }
    return 0;
}
} // namespace

int dbeel_tree_scan_ranges_to_dir(dbeel_tree *t, const dbeel_run *memtables, uint32_t n_memtables, const dbeel_hash_range *ranges,
                                  uint32_t n_ranges, uint32_t mode, const char *out_dir, dbeel_flush_table *per_range,
                                  dbeel_scan_stop *stop) {
    if (!t || (n_memtables && !memtables) || !stop || !out_dir || (n_ranges && !ranges)) return DBEEL_ERR_INVALID_ARG;
    if (n_ranges > DBEEL_MAX_SCAN_RANGES) return DBEEL_ERR_INVALID_ARG;
    t->err.clear();
    // the same tables as dbeel_tree_scan_ranges: SSTables (ascending index), then the non-empty memtables
    ScanFiles f;
    std::vector<dbeel_run> tables;
    std::vector<int32_t> position;
    uint64_t in_data = 0, in_records = 0;
    for (size_t i = 0; i < t->sstables.size(); i++) {
        const std::string dp = file_path(t->dir, t->sstables[i].index, kData), ip = file_path(t->dir, t->sstables[i].index, kIndex);
        const int dfd = open(dp.c_str(), O_RDONLY), ifd = open(ip.c_str(), O_RDONLY);
        f.data_fd.push_back(dfd);
        f.index_fd.push_back(ifd);
        f.mem.push_back(nullptr);
        struct stat sd, si;
        if (dfd < 0 || ifd < 0 || fstat(dfd, &sd) != 0 || fstat(ifd, &si) != 0) return io_fail(t, "open " + dp);
        tables.push_back(dbeel_run{nullptr, (uint64_t)sd.st_size, nullptr, (uint64_t)si.st_size});
        position.push_back((int32_t)i);
    }
    for (uint32_t m = 0; m < n_memtables; m++) {
        if (memtables[m].index_len < DBEEL_INDEX_ENTRY_SIZE) continue;
        f.data_fd.push_back(-1);
        f.index_fd.push_back(-1);
        f.mem.push_back(&memtables[m]);
        tables.push_back(memtables[m]);
        position.push_back((int32_t)(t->sstables.size() + m));
    }
    for (const dbeel_run &r : tables) {
        in_data += r.data_len;
        in_records += r.index_len / DBEEL_INDEX_ENTRY_SIZE;
    }
    std::error_code ec;
    fs::create_directories(out_dir, ec);
    auto drop_outputs = [&]() { for (const std::string &p : f.out_path) unlink(p.c_str()); };
    for (uint32_t r = 0; r < n_ranges; r++) {
        for (const char *ext : {kData, kIndex}) {
            const std::string p = (fs::path(out_dir) / (std::to_string(r) + "." + ext)).string();
            const int fd = open(p.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644); // read-write: a shared writable mapping needs it
            if (fd < 0) { const int rc = io_fail(t, "create " + p); drop_outputs(); return rc; }
            f.out_path.push_back(p);
            f.out_fd.push_back(fd);
            f.out_map.push_back(nullptr);
            f.out_cap.push_back(0);
        }
    }
    if (stream_maps() && n_ranges) {
        // Any one range can take every selected byte, so every file is mapped at the whole bound; the ranges are disjoint, so
        // what they write together is the bound once: that is what the volume must have room for (see tree_compact_streamed).
        const uint64_t cap_d = in_data, cap_i = 16 * in_records;
        struct statvfs vfs;
        if (fstatvfs(f.out_fd[0], &vfs) == 0 && (uint64_t)vfs.f_bavail * (uint64_t)vfs.f_frsize >= cap_d + cap_i + (64ull << 20)) {
            for (size_t k = 0; k < f.out_fd.size(); k++) {
                const uint64_t cap = k & 1 ? cap_i : cap_d;
                if (!cap || ftruncate(f.out_fd[k], (off_t)cap) != 0) continue;
                void *m = mmap(nullptr, cap, PROT_READ | PROT_WRITE, MAP_SHARED, f.out_fd[k], 0);
                if (m == MAP_FAILED) { if (ftruncate(f.out_fd[k], 0) != 0) {} continue; }
                f.out_map[k] = static_cast<uint8_t *>(m);
                f.out_cap[k] = cap;
            }
        }
    }
    dbeel_scan_io io{scan_read, scan_write, &f};
    int rc = dbeel_scan_ranges_stream(t->engine, tables.data(), (uint32_t)tables.size(), ranges, n_ranges, mode, &io, 0, per_range, stop);
    if (stop->table >= 0 && (size_t)stop->table < position.size()) stop->table = position[stop->table];
    if (rc) {
        if (rc == DBEEL_ERR_IO) { errno = f.saved_errno.load(); io_fail(t, "streamed scan"); }
        else t->err = dbeel_last_error(t->engine);
        drop_outputs();
        return rc;
    }
    f.unmap();
    for (uint32_t r = 0; r < n_ranges; r++) {
        for (int k = 0; k < 2; k++) { // cut to the final length (mapped files were sized to the bound)
            const size_t j = 2ull * r + k;
            const bool cut = ftruncate(f.out_fd[j], (off_t)(k ? per_range[r].index_len : per_range[r].data_len)) == 0;
            const bool closed = close(f.out_fd[j]) == 0;
            f.out_fd[j] = -1;
            if (!cut || !closed) { rc = io_fail(t, "close " + f.out_path[j]); drop_outputs(); return rc; }
        }
    }
    return DBEEL_OK;
}

int dbeel_tree_recover_wal(dbeel_tree *t, uint32_t tree_capacity, uint64_t *wal_file_index, uint64_t *items_written) {
    if (!t) return DBEEL_ERR_INVALID_ARG;
    t->err.clear();
    if (items_written) *items_written = 0;
    std::error_code ec;
    std::vector<uint64_t> wal;
    uint64_t idx;
    for (auto &de : fs::directory_iterator(t->dir, ec))
        if (parse_name(de.path().filename().string(), kMemtable, &idx)) wal.push_back(idx);
    std::sort(wal.begin(), wal.end()); // lsm_tree.rs:467-476
    uint64_t current = 0;
    if (wal.size() == 1) {
        current = wal[0];
    } else if (wal.size() == 2) { // "A flush did not finish for some reason, do it now." (:481-511)
        current = wal[1];
        const std::string old_path = file_path(t->dir, wal[0], kMemtable);
        PinnedBuf log;
        int rc = read_file(t, old_path, &log);
        if (rc) return rc;
        const uint64_t pages = (log.len + 4095) / 4096;
        PinnedBuf od(log.len), oi(pages * 16);
        if (!od.p || !oi.p) { t->err = "dbeel_host_alloc failed"; return DBEEL_ERR_NOMEM; }
        dbeel_out out{od.p, log.len, 0, oi.p, pages * 16, 0, nullptr, 0, 0, 0};
        rc = dbeel_wal_flush(t->engine, log.p, log.len, tree_capacity, &out); // read_memtable_from_wal_file + flush_memtable_to_disk
        if (rc) { t->err = dbeel_last_error(t->engine); return rc; }
        // The reference writes the recovered table under the NEWER log's index (get_data_file_paths(&dir, wal_file_index),
        // :491-492), not under the index the interrupted flush would have used, and does not add it to `sstables` for
        // this open (the list was built before, :440-459): the next open discovers it.  Mirrored as is.
        rc = write_file(t, file_path(t->dir, current, kData), od.p, out.data_len);
        if (!rc) rc = write_file(t, file_path(t->dir, current, kIndex), oi.p, out.index_len);
        if (!rc && t->page_sink) dbeel_out_pages(od.p, out.data_len, oi.p, out.index_len, current, t->page_sink, t->page_ctx);
        if (rc) return rc;
        if (unlink(old_path.c_str()) != 0) return io_fail(t, "remove " + old_path); // :510
        if (items_written) *items_written = out.items_written;
    } else if (wal.size() > 2) {
        t->err = "Cannot have more than 2 WAL files"; // the reference panics (:513)
        return DBEEL_ERR_INVALID_ARG;
    }
    if (wal_file_index) *wal_file_index = current;
    return DBEEL_OK;
}

// ---- shard ring (src/shards.rs:95-109,213-214,586-598,657-670): host arithmetic, same code text as the routing kernel

uint32_t dbeel_murmur3_32(const void *bytes, uint64_t len, uint32_t seed) {
    const uint8_t *p = static_cast<const uint8_t *>(bytes);
    return dbeel::murmur3_32(len, seed, [p, len](uint64_t q) {
        uint64_t w = 0;
        const uint64_t left = len - 8 * q;
        memcpy(&w, p + 8 * q, left < 8 ? left : 8);
        return w;
    });
}

uint32_t dbeel_ring_owner(const uint32_t *ring_hashes, uint32_t n_shards, uint32_t key_hash) {
    if (!ring_hashes || !n_shards) return 0;
    return dbeel::ring_owner(n_shards, key_hash, [ring_hashes](uint32_t s) { return ring_hashes[s]; });
}

int dbeel_shard_ring(const char *node_name, uint32_t n_shards, uint32_t *ring_hashes, uint32_t *ring_ids) {
    if (!ring_hashes || !ring_ids || !n_shards || n_shards > 65536) return DBEEL_ERR_INVALID_ARG;
    std::vector<std::pair<uint32_t, uint32_t>> ring;
    for (uint32_t id = 0; id < n_shards; id++) {
        const std::string name = std::string(node_name ? node_name : "dbeel") + "-" + std::to_string(id); // shards.rs:213
        ring.emplace_back(dbeel_murmur3_32(name.data(), name.size(), 0), id);
    }
    std::sort(ring.begin(), ring.end());
    for (uint32_t p = 0; p < n_shards; p++) {
        if (p && ring[p].first == ring[p - 1].first) return DBEEL_ERR_INVALID_ARG;
        ring_hashes[p] = ring[p].first;
        ring_ids[p] = ring[p].second;
    }
    return DBEEL_OK;
}

uint64_t dbeel_memtable_cut(const dbeel_run *batch, uint64_t first_record, uint32_t capacity) {
    if (!batch || !capacity) return 0;
    const uint8_t *ix = static_cast<const uint8_t *>(batch->index), *d = static_cast<const uint8_t *>(batch->data);
    const uint64_t n = batch->index_len / DBEEL_INDEX_ENTRY_SIZE;
    std::unordered_set<std::string_view> keys;
    keys.reserve(capacity * 2);
    uint64_t i = first_record;
    for (; i < n; i++) {
        uint64_t off;
        uint32_t ks;
        memcpy(&off, ix + 16 * i, 8);
        memcpy(&ks, ix + 16 * i + 8, 4);
        if (ks < 8 || off > batch->data_len || ks > batch->data_len - off) break; // undecodable: the batch ends here
        keys.emplace(reinterpret_cast<const char *>(d + off + 8), ks - 8);
        if (keys.size() == capacity) { i++; break; } // active_memtable_full() right after the insert
    }
    return i - first_record;
}

uint32_t dbeel_plan_compactions(const uint64_t *indices, const uint64_t *sizes, uint32_t n, uint32_t compaction_factor,
                                uint64_t *members, uint32_t *group_start, uint64_t *output_index, int32_t *keep_tombstones) {
    if (compaction_factor < 2) return 0; // compaction.rs:105-108
    auto lz = [](uint64_t v) -> uint32_t { return v ? (uint32_t)__builtin_clzll(v) : 64u; };
    // compaction.rs:38-43
    uint64_t next_out = 1;
    for (uint32_t i = 0; i < n; i++)
        if (indices[i] & 1) next_out = std::max(next_out, indices[i] + 2);
    // compaction.rs:45-52: group by leading_zeros(size), smallest tables (most zeros) first
    std::map<uint32_t, std::vector<uint32_t>, std::greater<uint32_t>> groups;
    for (uint32_t i = 0; i < n; i++) groups[lz(sizes[i])].push_back(i);
    // compaction.rs:55-80: promote a tier whose summed size crosses into a larger order
    std::map<uint32_t, std::vector<uint32_t>> optimized; // ascending order = largest tables first
    for (auto &g : groups) {
        std::vector<uint32_t> items = g.second;
        auto it = optimized.find(g.first);
        if (it != optimized.end()) {
            items.insert(items.end(), it->second.begin(), it->second.end());
            optimized.erase(it);
        }
        uint64_t sum = 0;
        for (uint32_t i : items) sum += sizes[i];
        uint32_t est = lz(sum);
        uint32_t order = est < g.first ? est : g.first;
        auto &dst = optimized[order];
        dst.insert(dst.end(), items.begin(), items.end());
    }
    // compaction.rs:82-101 -- enumerate() counts skipped groups too
    uint32_t n_groups = 0, pos = 0, i = 0;
    group_start[0] = 0;
    for (auto &g : optimized) {
        const bool run = g.second.size() >= 2 && g.second.size() >= compaction_factor;
        if (run) {
            for (uint32_t m : g.second) members[pos++] = indices[m];
            output_index[n_groups] = next_out;
            keep_tombstones[n_groups] = i > 0 ? 1 : 0;
            next_out += 2;
            n_groups++;
            group_start[n_groups] = pos;
        }
        i++;
    }
    return n_groups;
}

} // extern "C"
