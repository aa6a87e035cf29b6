// Whole-file driver (csq_run_files).  The B200 analogue of cutadapt's reader / worker / ordered-writer runner behind
// runner.run(pipeline, Progress(), outfiles) in reference run.py:436-473 / 753-794 (`-t N`): batches are contiguous
// record ranges, any GPU takes the next one, the outputs are reassembled in input order.
//
//   sequencer   (one thread) decides what every batch is, in order, WITHOUT touching the payload more than it must:
//                 plain files   counts line ends in the page cache (mmap, a few threads) -> byte ranges
//                 BGZF files    walks the member headers; line ends per member come from the GPUs (index jobs:
//                               csq_bgzf_count_lines), batches are runs of whole members + "skip k lines"
//                 other input   (single-member gzip, pipes, .bz2/.xz through the transcoder) the serial text reader
//   loaders     (pool) pread the byte range of a job - text or compressed members - into its pinned buffer
//   GPU workers (one thread per GPU, two batches in flight each) csq_submit_text / csq_submit_bgzf + csq_wait
//   writer      outputs are sized in batch order (a file offset per batch and stream), the bytes are then written
//               by the pool with pwrite, in any order; .gz outputs arrive as gzip members from the device
//               (CSQ_PLAN_GZIP_OUT) when every output is a .gz, else host zlib members are made by the pool
// Nothing in the data path is one thread per run: the sequencer only produces descriptors.
#include <cuda_runtime.h>
#include <errno.h>
#include <fcntl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "host_io.h"

void csq_set_error(const char* msg);
struct csq_text_reader;
int csq_text_reader_next_into(csq_text_reader* r, csqio::PinnedBuf* bufs, uint32_t max_reads, csq_batch_text* in);
extern "C" int csq_text_reader_open_flags(const char* path1, const char* path2, uint32_t plan_flags, csq_text_reader** out);
extern "C" void csq_text_reader_close(csq_text_reader* r);

namespace {

using Clock = std::chrono::steady_clock;
double seconds_since(Clock::time_point t0) { return std::chrono::duration<double>(Clock::now() - t0).count(); }

template <typename T>
class Queue {
   public:
    void push(T v) {
        {
            std::lock_guard<std::mutex> g(m_);
            q_.push_back(std::move(v));
        }
        cv_.notify_one();
    }
    // returns false when the queue is closed and empty
    bool pop(T& out) {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [&] { return !q_.empty() || closed_; });
        if (q_.empty()) return false;
        out = std::move(q_.front());
        q_.pop_front();
        return true;
    }
    // 1: got one, 0: nothing there right now, -1: closed and empty
    int try_pop(T& out) {
        std::lock_guard<std::mutex> g(m_);
        if (q_.empty()) return closed_ ? -1 : 0;
        out = std::move(q_.front());
        q_.pop_front();
        return 1;
    }
    void close() {
        {
            std::lock_guard<std::mutex> g(m_);
            closed_ = true;
        }
        cv_.notify_all();
    }

   private:
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<T> q_;
    bool closed_ = false;
};

class Pool {  // worker threads for loads, host deflate and writes
   public:
    explicit Pool(int n) {
        for (int i = 0; i < n; i++)
            threads_.emplace_back([this] {
                std::function<void()> f;
                while (q_.pop(f)) f();
            });
    }
    ~Pool() {
        q_.close();
        for (auto& t : threads_) t.join();
    }
    void run(std::function<void()> f) { q_.push(std::move(f)); }

   private:
    Queue<std::function<void()>> q_;
    std::vector<std::thread> threads_;
};

enum JobKind { J_TEXT = 0, J_BGZF = 1, J_INDEX = 2 };

struct Job {
    long index = -1;
    int kind = J_TEXT;
    // what to load from the input files (plain text ranges or runs of BGZF members); len == 0: nothing to load
    uint64_t load_off[2] = {0, 0}, load_len[2] = {0, 0};
    bool append_nl[2] = {false, false};
    csqio::PinnedBuf in_buf[2];            // FASTQ text or compressed members
    std::vector<uint32_t> moff[2], ooff[2];  // BGZF: member / text offsets of the run
    uint32_t skip[2] = {0, 0};
    int index_mate = 0;                    // J_INDEX: which input file
    size_t index_first = 0;                // ... first member of the range
    csq_batch_text tin;
    csq_batch_bgzf bin;
    csqio::PinnedBuf outbuf[CSQ_N_DEST][2];
    csq_batch_out out;
    int slot = 0;
    float total_ms = 0, kernel_ms = 0;
    std::atomic<int> parts{0};             // outstanding load / deflate / write pieces
    struct Piece {
        int d, m;
        const uint8_t* src;
        size_t n;
        std::vector<uint8_t> z;  // host deflate
        uint64_t file_off = 0;
    };
    std::vector<Piece> pieces;             // writer side
};

struct Shared {
    std::mutex err_m;
    int err_code = 0;
    std::string err_msg;
    std::atomic<bool> stop{false};
    Queue<Job*>*free_q = nullptr, *ready_q = nullptr;
    std::condition_variable* wake = nullptr;
    void fail(int code, const char* msg) {
        {
            std::lock_guard<std::mutex> g(err_m);
            if (!err_code) {
                err_code = code;
                err_msg = msg ? msg : "";
            }
            stop = true;
        }
        // unblock everybody
        if (free_q) free_q->close();
        if (ready_q) ready_q->close();
        if (wake) wake->notify_all();
    }
};

struct OutStream {
    int fd = -1;
    std::string path;
    bool gzip = false;
    int level = 1;
    uint64_t pos = 0;  // next free file offset
    bool seekable = true;  // false: a pipe (the .bz2 / .xz transcoders, process substitution) - written in order with write()
};

bool ends_with_gz(const char* p) {
    const size_t n = strlen(p);
    return n > 3 && !strcmp(p + n - 3, ".gz");
}

bool full_pwrite(int fd, const uint8_t* p, size_t n, uint64_t off) {
    while (n) {
        const ssize_t w = pwrite(fd, p, n, (off_t)off);
        if (w < 0) {
            if (errno == EINTR) continue;
            return false;
        }
        p += w;
        n -= (size_t)w;
        off += (uint64_t)w;
    }
    return true;
}

bool full_write(int fd, const uint8_t* p, size_t n) {
    while (n) {
        const ssize_t w = write(fd, p, n);
        if (w < 0) {
            if (errno == EINTR) continue;
            return false;
        }
        p += w;
        n -= (size_t)w;
    }
    return true;
}

bool full_pread(int fd, uint8_t* p, size_t n, uint64_t off) {
    while (n) {
        const ssize_t r = pread(fd, p, n, (off_t)off);
        if (r < 0) {
            if (errno == EINTR) continue;
            return false;
        }
        if (r == 0) return false;
        p += r;
        n -= (size_t)r;
        off += (uint64_t)r;
    }
    return true;
}

// ---- what kind of input is this ------------------------------------------------------------------------------------
struct InFile {
    int fd = -1;
    uint64_t size = 0;
    const uint8_t* map = nullptr;
    bool regular = false, gz = false, bgzf = false;
    // BGZF: file offset of every member (+ the end), uncompressed size of every member
    std::vector<uint64_t> moff;
    std::vector<uint32_t> isize;
    ~InFile() {
        if (map) munmap((void*)map, (size_t)size);
        if (fd >= 0) close(fd);
    }
};

size_t bgzf_member_size_at(const uint8_t* p, size_t n) {
    if (n < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return 0;
    const size_t xlen = p[10] | ((size_t)p[11] << 8);
    if (12 + xlen > n) return 0;
    for (size_t q = 12; q + 4 <= 12 + xlen;) {
        const size_t slen = p[q + 2] | ((size_t)p[q + 3] << 8);
        if (p[q] == 'B' && p[q + 1] == 'C' && slen == 2 && q + 6 <= 12 + xlen) {
            const size_t total = (size_t)(p[q + 4] | ((size_t)p[q + 5] << 8)) + 1;
            return total >= 12 + xlen + 8 && total <= n ? total : 0;
        }
        q += 4 + slen;
    }
    return 0;
}

int open_infile(const char* path, InFile& f, bool want_bgzf_index) {
    f.fd = open(path, O_RDONLY);
    if (f.fd < 0) return csqio::io_fail(CSQ_ERR_IO, "cannot open %s: %s", path, strerror(errno));
    struct stat sb;
    if (fstat(f.fd, &sb) != 0) return csqio::io_fail(CSQ_ERR_IO, "cannot stat %s: %s", path, strerror(errno));
    f.regular = S_ISREG(sb.st_mode);
    f.size = f.regular ? (uint64_t)sb.st_size : 0;
    if (!f.regular || f.size == 0) return 0;
    void* m = mmap(nullptr, (size_t)f.size, PROT_READ, MAP_SHARED, f.fd, 0);
    if (m == MAP_FAILED) {
        f.regular = false;  // falls back to the serial reader
        return 0;
    }
    f.map = (const uint8_t*)m;
    f.gz = f.size >= 2 && f.map[0] == 0x1f && f.map[1] == 0x8b;
    if (f.gz && want_bgzf_index && bgzf_member_size_at(f.map, (size_t)f.size)) {
        uint64_t off = 0;
        while (off < f.size) {
            const size_t total = bgzf_member_size_at(f.map + off, (size_t)(f.size - off));
            if (!total) {  // not BGZF all the way: the serial reader takes the file
                f.moff.clear();
                f.isize.clear();
                return 0;
            }
            const uint8_t* t = f.map + off + total - 4;
            f.moff.push_back(off);
            f.isize.push_back((uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16) | ((uint32_t)t[3] << 24));
            off += total;
        }
        f.moff.push_back(off);
        f.bgzf = true;
    }
    return 0;
}

// Plain file: where does the batch of `max_reads` records that starts at byte `off` end?  Counts line ends in the
// mapped file with a few threads; nothing is copied.
struct PlainCutter {
    const InFile* f = nullptr;
    uint64_t off = 0;
    size_t hint = 0;
    uint64_t records_done = 0;
    int threads = 2;
    std::string name;
    csqio::RecordCut rc;
    // -> 0 ok (len == 0 and n == 0 at the end of the file), else error code
    int next(uint32_t max_reads, uint64_t* start, uint64_t* len, uint32_t* n, bool* append_nl) {
        *start = off;
        *len = 0;
        *n = 0;
        *append_nl = false;
        if (off >= f->size) return 0;
        const uint64_t target = rc.target(max_reads);
        const uint8_t* base = f->map + off;
        const uint64_t left = f->size - off;
        uint64_t pos = 0, lines = 0;
        size_t want = hint ? hint + hint / 32 + (64u << 10) : (size_t)max_reads * 384 + (64u << 10);
        for (;;) {
            uint64_t round = want > pos ? want - pos : 0;
            if (round > left - pos) round = left - pos;
            if (round == 0) break;
            int nt = threads;
            if ((uint64_t)nt > round / (4u << 20) + 1) nt = (int)(round / (4u << 20) + 1);
            std::vector<uint64_t> cnt((size_t)nt, 0);
            const uint64_t per = (round + (uint64_t)nt - 1) / (uint64_t)nt;
            auto work = [&](int t) {
                const uint64_t b = pos + (uint64_t)t * per, e = std::min(pos + round, b + per);
                cnt[(size_t)t] = e > b ? rc.count(base + b, (size_t)(e - b), b ? base[b - 1] : (uint8_t)'\n') : 0;
            };
            std::vector<std::thread> helpers;
            for (int t = 1; t < nt; t++) helpers.emplace_back(work, t);
            work(0);
            for (auto& th : helpers) th.join();
            for (int t = 0; t < nt; t++) {
                const uint64_t b = pos + (uint64_t)t * per, e = std::min(pos + round, b + per);
                if (lines + cnt[(size_t)t] >= target) {
                    const uint64_t rel = rc.cut(base + b, (size_t)(e - b), target - lines, b ? base[b - 1] : (uint8_t)'\n');
                    const uint64_t cut = b + rel;
                    *len = cut;
                    *n = max_reads;
                    off += cut;
                    hint = (size_t)cut;
                    records_done += max_reads;
                    return 0;
                }
                lines += cnt[(size_t)t];
            }
            pos += round;
            want = (size_t)(pos + pos / 8 + (256u << 10));
        }
        // the rest of the file holds fewer than max_reads records: dnaio accepts a missing final line end and blank
        // lines behind the last record
        uint64_t end = left;
        if (rc.fasta) {  // every record start left is a record of the batch; text without one must be blank
            if (lines == 0) {
                for (uint64_t i = 0; i < end; i++)
                    if (base[i] != ' ' && (base[i] < 9 || base[i] > 13))
                        return csqio::io_fail(CSQ_ERR_FORMAT, "%s: FASTA input does not start with a '>' header (line %llu)", name.c_str(),
                                              (unsigned long long)(csqio::count_newlines(base, (size_t)i) + 1));
                end = 0;
            }
            *append_nl = end && base[end - 1] != '\n';
            *len = end;
            *n = (uint32_t)lines;
            records_done += lines;
            off = f->size;
            return 0;
        }
        if (end && base[end - 1] != '\n') {
            *append_nl = true;
            lines++;
        }
        while (lines % 4 != 0 && end >= 2 && !*append_nl) {
            uint64_t q = end - 1;  // base[q] == '\n'
            if (q >= 1 && base[q - 1] == '\r') q--;
            if (q >= 1 && base[q - 1] == '\n') {
                end = q;
                lines--;
            } else {
                break;
            }
        }
        if (lines == 1 && end <= 2 && !*append_nl) {  // a file of just "\n"
            end = 0;
            lines = 0;
        }
        if (lines % 4 != 0)
            return csqio::io_fail(CSQ_ERR_FORMAT, "%s: FASTQ file ended prematurely (line %llu)", name.c_str(),
                                  (unsigned long long)(4 * records_done + lines + 1));
        *len = end;
        *n = (uint32_t)(lines / 4);
        records_done += lines / 4;
        off = f->size;
        return 0;
    }
};

}  // namespace

extern "C" int csq_run_files(const csq_op* ops_r1, int n1, const csq_op* ops_r2, int n2, const csq_filters* filters,
                             uint32_t plan_flags, const csq_files* files, csq_counters* counters, csq_timing* timing) {
    if (!files || !files->in[0] || !filters) {
        csq_set_error("null argument");
        return CSQ_ERR_INVALID;
    }
    const auto t_start = Clock::now();
    const bool trace = getenv("CSQ_TRACE") != nullptr;  // phase timestamps on stderr
    auto stamp = [&](const char* what) {
        if (trace) fprintf(stderr, "[csq_run_files] %8.3f s  %s\n", seconds_since(t_start), what);
    };
    const int n_mates = files->in[1] ? 2 : 1;
    if ((n_mates == 2) != (n2 > 0)) {
        csq_set_error("number of input files does not match the program (paired vs single-end)");
        return CSQ_ERR_INVALID;
    }
    const int n_dev = files->n_devices > 0 ? files->n_devices : 1;
    const int n_threads = files->n_threads > 0 ? files->n_threads : 4;

    // ---- outputs: device gzip when every output is a .gz ----
    bool any_out = false, all_gz = true;
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < n_mates; m++)
            if (files->out[d][m]) {
                any_out = true;
                all_gz = all_gz && ends_with_gz(files->out[d][m]);
            }
    const bool device_gzip = any_out && all_gz && !getenv("CSQ_HOST_DEFLATE");
    if (device_gzip) plan_flags |= CSQ_PLAN_GZIP_OUT;

    // ---- inputs ----
    InFile inf[2];
    const bool want_bgzf = !getenv("CSQ_HOST_INFLATE");
    for (int m = 0; m < n_mates; m++) {
        int rc = open_infile(files->in[m], inf[m], want_bgzf);
        if (rc) {
            csq_set_error(csqio::io_error());
            return rc;
        }
    }
    bool all_plain = true, all_bgzf = true;
    for (int m = 0; m < n_mates; m++) {
        all_plain = all_plain && inf[m].regular && inf[m].map && !inf[m].gz;
        all_bgzf = all_bgzf && inf[m].bgzf;
    }
    for (int m = 0; m < n_mates; m++)
        if (inf[m].regular && inf[m].size == 0) all_plain = all_bgzf = false;  // empty files: the serial reader knows what to do
    // FASTA never takes mode 1: the line ends per member do not tell where FASTA records start
    const bool fasta = (plan_flags & CSQ_PLAN_FASTA) != 0;
    if (fasta) all_bgzf = false;
    const int mode = all_plain ? 0 : all_bgzf ? 1 : 2;  // 0 plain ranges, 1 BGZF member runs, 2 serial text reader
    const csqio::RecordCut record_cut{fasta};
    // records in a sample of text (a FASTA record has any number of lines)
    auto sample_records = [&](const uint8_t* t, size_t n) -> double {
        return fasta ? (double)csqio::count_fasta_records(t, n, '\n') : (double)csqio::count_newlines(t, n) / 4.0;
    };
    const uint32_t batch_reads = files->batch_reads ? files->batch_reads : (mode == 2 ? (1u << 16) : (1u << 18));

    // plans: one thread per GPU creates its context and plan (0.3 - 0.5 s each when done one after the other)
    std::vector<csq_plan*> plans((size_t)n_dev, nullptr);
    auto destroy_plans = [&] {
        std::vector<std::thread> ts;
        for (csq_plan* p : plans)
            if (p) ts.emplace_back([p] { csq_plan_destroy(p); });
        for (auto& t : ts) t.join();
    };
    {
        std::vector<int> rcs((size_t)n_dev, 0);
        std::vector<std::string> msgs((size_t)n_dev);
        std::vector<std::thread> ts;
        for (int d = 0; d < n_dev; d++)
            ts.emplace_back([&, d] {
                const int dev = files->devices ? files->devices[d] : d;
                rcs[(size_t)d] = csq_plan_create(ops_r1, n1, ops_r2, n2, filters, dev, plan_flags, &plans[(size_t)d]);
                if (rcs[(size_t)d]) msgs[(size_t)d] = csq_last_error();
            });
        for (auto& t : ts) t.join();
        for (int d = 0; d < n_dev; d++)
            if (rcs[(size_t)d]) {
                csq_set_error(msgs[(size_t)d].c_str());
                destroy_plans();
                return rcs[(size_t)d];
            }
    }
    stamp("plans created");

    csq_text_reader* reader = nullptr;
    if (mode == 2) {
        int rc = csq_text_reader_open_flags(files->in[0], files->in[1], plan_flags, &reader);
        if (rc) {
            destroy_plans();
            return rc;
        }
    }
    OutStream outs[CSQ_N_DEST][2];
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < n_mates; m++)
            if (files->out[d][m]) {
                OutStream& o = outs[d][m];
                o.path = files->out[d][m];
                o.gzip = ends_with_gz(files->out[d][m]);
                o.level = files->gzip_level > 0 ? files->gzip_level : 1;  // cutadapt / xopen default
                o.fd = open(files->out[d][m], O_WRONLY | O_CREAT | O_TRUNC, 0666);
                if (o.fd < 0) {
                    char msg[512];
                    snprintf(msg, sizeof(msg), "cannot create %s: %s", files->out[d][m], strerror(errno));
                    csq_set_error(msg);
                    for (int dd = 0; dd < CSQ_N_DEST; dd++)
                        for (int mm = 0; mm < 2; mm++)
                            if (outs[dd][mm].fd >= 0) close(outs[dd][mm].fd);
                    if (reader) csq_text_reader_close(reader);
                    destroy_plans();
                    return CSQ_ERR_IO;
                }
                o.seekable = lseek(o.fd, 0, SEEK_CUR) != (off_t)-1;
            }

    Shared sh;
    const int n_jobs = 3 * n_dev + 3;
    std::vector<std::unique_ptr<Job>> jobs;
    Queue<Job*> free_q, ready_q;
    sh.free_q = &free_q;
    sh.ready_q = &ready_q;
    for (int i = 0; i < n_jobs; i++) jobs.emplace_back(new Job());
    std::unique_ptr<Pool> pool_owner(new Pool(std::max(2, n_threads)));
    Pool& pool = *pool_owner;

    // ---- host buffers of the jobs: sized from a sample of the input and pinned side by side, by a few threads of their
    // own, while the first batches are already on their way (pinning is the fixed cost of a run: ~2 GB/s when the
    // batches allocate one after the other as they come; a job joins the circulation when its buffers are there) ----
    std::unique_ptr<Pool> warm_owner(new Pool(std::max(2, std::min(8, n_threads / 2))));
    Pool& warm = *warm_owner;
    std::atomic<bool> warm_stop{false};  // the run is over: buffers nobody will use are not pinned any more
    auto output_sizes = [&](const uint64_t text[2], uint32_t n, uint64_t want[CSQ_N_DEST][2]) {
        for (int m = 0; m < 2; m++) {
            uint64_t full = 64;
            if (m < n_mates) {
                // renaming can only shorten a record, bar "_" + UMI; a FASTA record comes out with at most one line end
                // more than it had (">a\n" in front of the next header: ">a\n\n")
                full = text[m] + 64ull * n + 4096;
                if (device_gzip) full = full / 2;   // the packed size is reported when this guess is too small
            }
            for (int d = 0; d < CSQ_N_DEST; d++) want[d][m] = m >= n_mates ? 64 : d == CSQ_DEST_TRIMMED ? full : full / 8 + 4096;
        }
    };
    int jobs_in_use = n_jobs;
    // With several GPUs the jobs are released together, when the last one is pinned: a registration holds the driver's
    // lock across every context of the process, and the first submits of N GPUs (device allocations, module loads) would
    // queue behind each of them (measured at N = 4: first batch out after 0.97 s instead of 0.3 s).
    std::atomic<int> warm_left{0};
    std::vector<Job*> warm_held;
    std::mutex warm_m;
    {
        uint64_t est_text[2] = {0, 0}, est_load[2] = {0, 0};
        double n_batches_est = 0, all_text = 0;
        bool have_est = true;
        for (int m = 0; m < n_mates && have_est; m++) {
            double bpr = 0, ratio = 1.0;  // text bytes per record, compressed / text bytes
            uint64_t total_text = 0;
            if (mode == 2) {
                // the serial reader's inputs: a sample of a regular file's text tells the batch size (the reader's own
                // buffers would grow by doubling, every step a pinned allocation); pipes cannot be sampled
                if (!inf[m].regular || !inf[m].map || inf[m].size == 0) {
                    have_est = false;
                    break;
                }
                std::vector<uint8_t> text((size_t)1 << 20);
                long got = 0;
                if (inf[m].gz) {
                    csqio::Inflater inflater;
                    inflater.reset(inf[m].map, (size_t)std::min<uint64_t>(inf[m].size, 1u << 20));
                    got = inflater.read(text.data(), text.size() / 2);  // (a truncated view: stop well inside what it holds)
                    total_text = inf[m].size * 4;                       // a guess; only bounds the number of jobs
                } else {
                    got = (long)std::min<uint64_t>(inf[m].size, text.size());
                    memcpy(text.data(), inf[m].map, (size_t)got);
                    total_text = inf[m].size;
                }
                const double recs = got > 0 ? sample_records(text.data(), (size_t)got) : 0;
                if (recs >= 1) bpr = (double)got / recs;
            } else if (mode == 0) {
                const size_t sample = (size_t)std::min<uint64_t>(inf[m].size, 4u << 20);
                const double recs = sample_records(inf[m].map, sample);
                if (recs >= 1) bpr = (double)sample / recs;
                total_text = inf[m].size;
            } else {
                for (size_t i = 0; i < inf[m].isize.size() && bpr == 0; i++) {
                    if (!inf[m].isize[i]) continue;
                    std::vector<uint8_t> text(inf[m].isize[i] + 64);
                    csqio::Inflater inflater;
                    inflater.reset(inf[m].map + inf[m].moff[i], (size_t)(inf[m].moff[i + 1] - inf[m].moff[i]));
                    const long got = inflater.read(text.data(), inf[m].isize[i]);
                    const uint64_t lines = got > 0 ? csqio::count_newlines(text.data(), (size_t)got) : 0;
                    if (lines >= 4) bpr = (double)got / ((double)lines / 4.0);
                    break;
                }
                for (uint32_t v : inf[m].isize) total_text += v;
                if (total_text) ratio = (double)inf[m].size / (double)total_text;
            }
            if (bpr <= 0) {
                have_est = false;
                break;
            }
            const double batch_text = std::min((double)batch_reads * bpr * 1.02 + 65536.0, (double)total_text + 65536.0);
            est_text[m] = (uint64_t)batch_text;
            est_load[m] = (uint64_t)(batch_text * ratio * (mode == 1 ? 1.06 : 1.0)) + 65536;
            if (mode == 2) est_load[m] += 5u << 20;  // the reader asks for a piece (<= 4 MiB) more than the batch holds
            if (mode == 1) est_load[m] = std::max<uint64_t>(est_load[m], std::min<uint64_t>(inf[m].size, (48ull << 20) + 65536));
            n_batches_est = std::max(n_batches_est, (double)total_text / std::max(1.0, (double)batch_reads * bpr));
            all_text += (double)total_text;
        }
        uint64_t want[CSQ_N_DEST][2];
        output_sizes(est_text, batch_reads, want);
        // How many jobs does this input deserve?  Pinning runs at a few GB/s and holds the driver's lock (a submit that
        // meets it waits: measured, 15 jobs warming beside the first batches of a 4-GPU run delayed them by 2.4 s), so
        // the jobs in circulation are bounded by ~15 % of the input's text: a 20 M-pair file gets 5 jobs on any number
        // of GPUs (it cannot keep more than two or three busy), a 200 M-pair file all 3 N + 3.
        int n_use = n_jobs;
        if (have_est) {
            double job_bytes = 0;
            for (int m = 0; m < n_mates; m++) job_bytes += 1.125 * (double)est_load[m];
            for (int d = 0; d < CSQ_N_DEST; d++)
                for (int m = 0; m < n_mates; m++) job_bytes += 1.125 * (double)want[d][m];
            const int by_size = (int)(0.15 * all_text / std::max(1.0, job_bytes));
            const int by_batches = (int)(n_batches_est + 1.0 + (mode == 1 ? 2.0 : 0.0));
            n_use = std::max(std::min(n_jobs, 4), std::min(n_jobs, std::min(by_size, by_batches)));
            if (by_batches < n_use) n_use = std::max(1, by_batches);
        }
        if (trace) fprintf(stderr, "[csq_run_files] %8.3f s  %d of %d jobs in circulation\n", seconds_since(t_start), n_use, n_jobs);
        jobs_in_use = n_use;
        const int n_warm = have_est ? n_use : 0;
        warm_left = n_warm;
        for (int i = 0; i < n_use; i++) {
            Job* j = jobs[(size_t)i].get();
            if (i >= n_warm) {
                free_q.push(j);
                continue;
            }
            j->parts = n_mates + CSQ_N_DEST * 2;
            auto done_one = [&free_q, &warm_left, &warm_held, &warm_m, n_dev, j, i, trace, t_start] {
                if (--j->parts == 0) {
                    if (trace) fprintf(stderr, "[csq_run_files] %8.3f s  job %d warmed\n", seconds_since(t_start), i);
                    if (n_dev == 1) {
                        free_q.push(j);
                        return;
                    }
                    std::lock_guard<std::mutex> g(warm_m);
                    warm_held.push_back(j);
                    if (--warm_left == 0) {
                        for (Job* h : warm_held) free_q.push(h);
                        warm_held.clear();
                    }
                }
            };
            for (int m = 0; m < n_mates; m++) {
                const size_t need = (size_t)est_load[m] + 64;
                warm.run([j, m, need, done_one, &warm_stop, &sh] {
                    if (!warm_stop && !sh.stop) j->in_buf[m].reserve(need + need / 8, 0, 2);  // a failure shows when the batch reserves for real
                    done_one();
                });
            }
            for (int d = 0; d < CSQ_N_DEST; d++)
                for (int m = 0; m < 2; m++) {
                    const size_t need = (size_t)want[d][m];
                    warm.run([j, d, m, need, done_one, &warm_stop, &sh] {
                        if (!warm_stop && !sh.stop) j->outbuf[d][m].reserve(need + need / 8, 0, 2);
                        done_one();
                    });
                }
        }
    }
    std::atomic<double> t_read{0}, t_write{0};
    auto add_time = [](std::atomic<double>& a, double v) {
        double cur = a.load();
        while (!a.compare_exchange_weak(cur, cur + v)) {
        }
    };

    // ---- writer state ----
    std::mutex w_m;
    std::condition_variable w_cv;
    sh.wake = &w_cv;
    std::map<long, Job*> sized_wait;  // finished batches that wait for their predecessors to be sized
    long next_to_size = 0, written = 0, n_batches = -1;

    auto recycle = [&](Job* j) {
        {
            std::lock_guard<std::mutex> g(w_m);
            written++;
        }
        w_cv.notify_all();
        free_q.push(j);
    };
    // every stream of the batch gets its place in its file; the pool then writes the pieces in any order
    auto size_and_write = [&](Job* j) {  // w_m held
        int n_parts = 0;
        for (Job::Piece& pc : j->pieces) {
            OutStream& o = outs[pc.d][pc.m];
            const size_t n = o.gzip && !device_gzip ? pc.z.size() : pc.n;
            pc.file_off = o.pos;
            o.pos += n;
            if (n && !o.seekable) {  // batches are sized in order, so this is the stream order
                const auto t0 = Clock::now();
                if (!sh.stop && !full_write(o.fd, o.gzip && !device_gzip ? pc.z.data() : pc.src, n)) {
                    char msg[512];
                    snprintf(msg, sizeof(msg), "write to %s failed: %s", o.path.c_str(), strerror(errno));
                    sh.fail(CSQ_ERR_IO, msg);
                }
                add_time(t_write, seconds_since(t0));
            } else if (n) {
                n_parts++;
            }
        }
        if (n_parts == 0) {  // nothing to write (w_m is held)
            written++;
            w_cv.notify_all();
            free_q.push(j);
            return;
        }
        j->parts = n_parts;
        for (Job::Piece& pc : j->pieces) {
            OutStream& o = outs[pc.d][pc.m];
            const bool host_z = o.gzip && !device_gzip;
            const size_t n = host_z ? pc.z.size() : pc.n;
            if (!n || !o.seekable) continue;
            Job::Piece* p = &pc;
            pool.run([&, j, p, host_z, n] {
                if (!sh.stop) {
                    const auto t0 = Clock::now();
                    OutStream& os = outs[p->d][p->m];
                    if (!full_pwrite(os.fd, host_z ? p->z.data() : p->src, n, p->file_off)) {
                        char msg[512];
                        snprintf(msg, sizeof(msg), "write to %s failed: %s", os.path.c_str(), strerror(errno));
                        sh.fail(CSQ_ERR_IO, msg);
                    }
                    add_time(t_write, seconds_since(t0));
                }
                if (--j->parts == 0) recycle(j);
            });
        }
    };
    auto batch_sized = [&](Job* j) {
        std::lock_guard<std::mutex> g(w_m);
        sized_wait[j->index] = j;
        while (!sized_wait.empty() && sized_wait.begin()->first == next_to_size) {
            Job* w = sized_wait.begin()->second;
            sized_wait.erase(sized_wait.begin());
            next_to_size++;
            if (sh.stop) {
                written++;
                free_q.push(w);
                continue;
            }
            size_and_write(w);
        }
        w_cv.notify_all();
    };
    // a batch has come back from its GPU: cut its streams into pieces (and deflate them on the host if need be)
    const size_t PIECE = 8u << 20;
    auto batch_done = [&](Job* j) {
        j->pieces.clear();
        bool host_deflate = false;
        for (int d = 0; d < CSQ_N_DEST; d++)
            for (int m = 0; m < n_mates; m++) {
                // paired --auto-rc on '-' strand: R1 goes to the R2 file and vice versa (trimmed only)
                const int fm = (d == CSQ_DEST_TRIMMED && files->swap_sink && n_mates == 2) ? 1 - m : m;
                if (outs[d][fm].fd < 0) continue;
                const csq_text_out& t = j->out.text[d][m];
                const bool hz = outs[d][fm].gzip && !device_gzip;
                host_deflate = host_deflate || (hz && t.bytes);
                const size_t step = hz ? (4u << 20) : PIECE;
                for (size_t off = 0; off < t.bytes; off += step) {
                    Job::Piece pc;
                    pc.d = d;
                    pc.m = fm;
                    pc.src = t.data + off;
                    pc.n = (size_t)std::min<uint64_t>(step, t.bytes - off);
                    j->pieces.push_back(std::move(pc));
                }
            }
        if (!host_deflate) {
            batch_sized(j);
            return;
        }
        int nz = 0;
        for (Job::Piece& pc : j->pieces) nz += outs[pc.d][pc.m].gzip ? 1 : 0;
        j->parts = nz;
        for (Job::Piece& pc : j->pieces) {
            if (!outs[pc.d][pc.m].gzip) continue;
            Job::Piece* p = &pc;
            pool.run([&, j, p] {
                if (!sh.stop) {
                    const auto t0 = Clock::now();
                    if (csqio::gzip_member(p->src, p->n, outs[p->d][p->m].level, p->z)) sh.fail(CSQ_ERR_IO, csqio::io_error());
                    add_time(t_write, seconds_since(t0));
                }
                if (--j->parts == 0) batch_sized(j);
            });
        }
    };

    // ---- loaders: the byte ranges of a job, in pieces, then the job is ready for a GPU ----
    std::mutex ld_m;
    std::condition_variable ld_cv;
    int loading = 0;  // jobs whose pieces are still being read (the ready queue is closed only behind the last of them)
    auto load_and_ready = [&](Job* j) {
        int n_parts = 0;
        for (int m = 0; m < n_mates; m++) n_parts += (int)((j->load_len[m] + PIECE - 1) / PIECE);
        if (n_parts == 0) {
            ready_q.push(j);
            return;
        }
        {
            std::lock_guard<std::mutex> g(ld_m);
            loading++;
        }
        j->parts = n_parts;
        for (int m = 0; m < n_mates; m++)
            for (uint64_t o = 0; o < j->load_len[m]; o += PIECE) {
                const uint64_t n = std::min<uint64_t>(PIECE, j->load_len[m] - o);
                pool.run([&, j, m, o, n] {
                    if (!sh.stop) {
                        const auto t0 = Clock::now();
                        if (!full_pread(inf[m].fd, j->in_buf[m].p + o, (size_t)n, j->load_off[m] + o)) {
                            char msg[512];
                            snprintf(msg, sizeof(msg), "read error in %s: %s", files->in[m], errno ? strerror(errno) : "file changed while it was read");
                            sh.fail(CSQ_ERR_IO, msg);
                        }
                        add_time(t_read, seconds_since(t0));
                    }
                    if (--j->parts == 0) {
                        if (j->kind == J_TEXT)
                            for (int mm = 0; mm < n_mates; mm++)
                                if (j->append_nl[mm]) j->in_buf[mm].p[j->load_len[mm]] = '\n';
                        if (trace && j->index >= 0) fprintf(stderr, "[csq_run_files] %8.3f s  batch %ld loaded\n", seconds_since(t_start), j->index);
                        ready_q.push(j);
                        {
                            std::lock_guard<std::mutex> g(ld_m);
                            loading--;
                        }
                        ld_cv.notify_all();
                    }
                });
            }
    };

    // ---- BGZF index shared between the sequencer and the GPU workers ----
    std::mutex ix_m;
    std::condition_variable ix_cv;
    std::vector<uint32_t> mlines[2];     // line ends per member (bit 31: the member's text does not end in '\n')
    std::vector<uint8_t> mdone[2];
    int index_jobs_out = 0;              // index jobs on their way (under ix_m)
    for (int m = 0; m < n_mates && mode == 1; m++) {
        mlines[m].assign(inf[m].isize.size(), 0);
        mdone[m].assign(inf[m].isize.size(), 0);
    }

    // ---- the sequencer ----
    std::thread sequencer([&] {
        long index = 0;
        uint64_t first_record = 0;
        auto finish = [&] {
            {
                std::lock_guard<std::mutex> g(w_m);
                n_batches = index;
            }
            w_cv.notify_all();
            {  // the last jobs may still be loading
                std::unique_lock<std::mutex> g(ld_m);
                while (loading != 0 && !sh.stop.load()) ld_cv.wait_for(g, std::chrono::milliseconds(50));
            }
            ready_q.close();
            stamp("sequencer done");
        };
        Job* j = nullptr;
        if (mode == 2) {
            while (!sh.stop && free_q.pop(j)) {
                const auto t0 = Clock::now();
                j->kind = J_TEXT;
                j->load_len[0] = j->load_len[1] = 0;
                int r = csq_text_reader_next_into(reader, j->in_buf, batch_reads, &j->tin);
                add_time(t_read, seconds_since(t0));
                if (r) {
                    sh.fail(r, csq_last_error());
                    break;
                }
                if (j->tin.n_reads == 0) {
                    free_q.push(j);
                    break;
                }
                j->index = index++;
                ready_q.push(j);
            }
            finish();
            return;
        }
        if (mode == 0) {
            PlainCutter cut[2];
            for (int m = 0; m < n_mates; m++) {
                cut[m].f = &inf[m];
                cut[m].name = files->in[m];
                cut[m].threads = std::max(1, std::min(6, n_threads / (2 * n_mates)));
                cut[m].rc = record_cut;
            }
            while (!sh.stop && free_q.pop(j)) {
                uint32_t n[2] = {0, 0};
                int rcs[2] = {0, 0};
                std::string msgs[2];
                auto work = [&](int m) {
                    rcs[m] = cut[m].next(batch_reads, &j->load_off[m], &j->load_len[m], &n[m], &j->append_nl[m]);
                    if (rcs[m]) msgs[m] = csqio::io_error();
                };
                if (n_mates == 2) {
                    std::thread t(work, 1);
                    work(0);
                    t.join();
                } else {
                    work(0);
                }
                int bad = rcs[0] ? 0 : rcs[1] ? 1 : -1;
                if (bad >= 0) {
                    sh.fail(rcs[bad], msgs[bad].c_str());
                    break;
                }
                if (n_mates == 2 && n[0] != n[1]) {
                    sh.fail(CSQ_ERR_FORMAT, "paired input files have different numbers of records");
                    break;
                }
                if (n[0] == 0) {
                    free_q.push(j);
                    break;
                }
                j->kind = J_TEXT;
                memset(&j->tin, 0, sizeof(j->tin));
                j->tin.n_reads = n[0];
                j->tin.n_mates = (uint32_t)n_mates;
                j->tin.first_record = first_record;
                bool ok = true;
                for (int m = 0; m < n_mates; m++) {
                    const size_t need = (size_t)j->load_len[m] + 64;
                    if (j->in_buf[m].cap < need && !j->in_buf[m].reserve(need + need / 8, 0)) ok = false;
                    j->tin.mate[m].text = j->in_buf[m].p;
                    j->tin.mate[m].bytes = j->load_len[m] + (j->append_nl[m] ? 1 : 0);
                }
                if (!ok) {
                    sh.fail(CSQ_ERR_NOMEM, "out of host memory for a batch");
                    break;
                }
                first_record += n[0];
                j->index = index++;
                if (trace) fprintf(stderr, "[csq_run_files] %8.3f s  batch %ld cut\n", seconds_since(t_start), j->index);
                load_and_ready(j);
            }
            finish();
            return;
        }
        // mode 1: BGZF.  Index jobs run ahead (line ends per member, counted on the GPUs); a batch is cut as soon as
        // the index covers it in every input file.
        const uint64_t INDEX_BYTES = 48ull << 20;
        size_t next_index_member[2] = {0, 0};   // first member without an index job
        size_t indexed[2] = {0, 0};             // members [0, indexed) have their line counts
        std::vector<uint64_t> cum[2];           // cum[m][i] = line ends in members [0, i)
        for (int m = 0; m < n_mates; m++) cum[m].assign(1, 0);
        bool eof_fix[2] = {false, false};
        uint64_t total_records = UINT64_MAX;
        auto absorb = [&] {  // ix_m held: extend the indexed prefixes
            for (int m = 0; m < n_mates; m++)
                while (indexed[m] < mdone[m].size() && mdone[m][indexed[m]]) {
                    cum[m].push_back(cum[m].back() + (mlines[m][indexed[m]] & 0x7FFFFFFFu));
                    indexed[m]++;
                }
        };
        for (;;) {
            if (sh.stop) break;
            int jobs_out;
            {
                std::lock_guard<std::mutex> g(ix_m);
                absorb();
                jobs_out = index_jobs_out;
            }
            // everything indexed: the number of records is known
            if (total_records == UINT64_MAX) {
                bool all = true;
                for (int m = 0; m < n_mates; m++) all = all && indexed[m] == inf[m].isize.size();
                if (all) {
                    uint64_t recs[2] = {0, 0};
                    bool bad = false;
                    for (int m = 0; m < n_mates; m++) {
                        uint64_t lines = cum[m].back();
                        // the last member with text decides whether the file ends in a line end
                        for (size_t i = inf[m].isize.size(); i-- > 0;)
                            if (inf[m].isize[i]) {
                                if (mlines[m][i] & 0x80000000u) {
                                    eof_fix[m] = true;
                                    lines++;
                                }
                                break;
                            }
                        if (lines % 4 != 0) {
                            char msg[512];
                            snprintf(msg, sizeof(msg), "%s: FASTQ file ended prematurely (%llu lines)", files->in[m], (unsigned long long)lines);
                            sh.fail(CSQ_ERR_FORMAT, msg);
                            bad = true;
                            break;
                        }
                        recs[m] = lines / 4;
                    }
                    if (bad) break;
                    if (n_mates == 2 && recs[0] != recs[1]) {
                        sh.fail(CSQ_ERR_FORMAT, "paired input files have different numbers of records");
                        break;
                    }
                    total_records = recs[0];
                }
            }
            if (total_records != UINT64_MAX && first_record >= total_records) break;
            // can the next batch be cut?
            const uint64_t want_n = total_records != UINT64_MAX ? std::min<uint64_t>(batch_reads, total_records - first_record) : batch_reads;
            const uint64_t s_line = 4 * first_record, e_line = 4 * (first_record + want_n);
            bool covered = true;
            for (int m = 0; m < n_mates; m++) {
                const bool fix = total_records != UINT64_MAX && eof_fix[m] && first_record + want_n == total_records;
                covered = covered && (cum[m].back() + (fix ? 1 : 0) >= e_line);
            }
            if (covered) {
                if (!free_q.pop(j)) break;
                j->kind = J_BGZF;
                memset(&j->bin, 0, sizeof(j->bin));
                j->bin.n_reads = (uint32_t)want_n;
                j->bin.n_mates = (uint32_t)n_mates;
                j->bin.first_record = first_record;
                bool ok = true;
                for (int m = 0; m < n_mates; m++) {
                    const std::vector<uint64_t>& c = cum[m];
                    // first member: the one that holds line end number s_line - 1 (the record starts behind it)
                    size_t f = 0;
                    if (s_line > 0) f = (size_t)(std::lower_bound(c.begin(), c.end(), s_line) - c.begin()) - 1;  // c[f] < s_line <= c[f+1]
                    const bool fix = eof_fix[m] && first_record + want_n == total_records;
                    size_t l;  // last member: the one that holds line end number e_line - 1
                    if (fix && c.back() < e_line)
                        l = inf[m].isize.size() - 1;
                    else
                        l = (size_t)(std::lower_bound(c.begin(), c.end(), e_line) - c.begin()) - 1;
                    if (l < f) l = f;
                    j->skip[m] = (uint32_t)(s_line - c[f]);
                    j->load_off[m] = inf[m].moff[f];
                    j->load_len[m] = inf[m].moff[l + 1] - inf[m].moff[f];
                    j->moff[m].resize(l - f + 2);
                    j->ooff[m].resize(l - f + 2);
                    uint64_t t = 0;
                    for (size_t i = f; i <= l + 1; i++) {
                        j->moff[m][i - f] = (uint32_t)(inf[m].moff[i] - inf[m].moff[f]);
                        j->ooff[m][i - f] = (uint32_t)t;
                        if (i <= l) t += inf[m].isize[i];
                    }
                    if (t >= (1ull << 32) - (1u << 20) || j->load_len[m] >= (1ull << 32)) {
                        sh.fail(CSQ_ERR_LIMIT, "a batch of BGZF members exceeds 4 GiB: use a smaller batch_reads");
                        ok = false;
                        break;
                    }
                    const size_t need = (size_t)j->load_len[m] + 64;
                    if (j->in_buf[m].cap < need && !j->in_buf[m].reserve(need + need / 8, 0)) {
                        sh.fail(CSQ_ERR_NOMEM, "out of host memory for a batch");
                        ok = false;
                        break;
                    }
                    csq_bgzf_in& bi = j->bin.mate[m];
                    bi.data = j->in_buf[m].p;
                    bi.bytes = j->load_len[m];
                    bi.member_off = j->moff[m].data();
                    bi.text_off = j->ooff[m].data();
                    bi.n_members = (uint32_t)(l - f + 1);
                    bi.skip_lines = j->skip[m];
                    bi.append_newline = fix ? 1u : 0u;
                }
                if (!ok) break;
                first_record += want_n;
                j->index = index++;
                load_and_ready(j);
                continue;
            }
            // not covered: send the next index job (for the input file whose index is further behind), or wait for results
            int m_next = -1;
            double behind = 2.0;
            for (int m = 0; m < n_mates; m++)
                if (next_index_member[m] < inf[m].isize.size()) {
                    const double frac = (double)inf[m].moff[next_index_member[m]] / (double)inf[m].size;
                    if (frac < behind) {
                        behind = frac;
                        m_next = m;
                    }
                }
            if (m_next >= 0 && jobs_out < std::max(1, std::min(2 * n_dev + 1, jobs_in_use / 2))) {
                if (!free_q.pop(j)) break;
                const int m = m_next;
                size_t f = next_index_member[m], l = f;
                while (l < inf[m].isize.size() && inf[m].moff[l + 1] - inf[m].moff[f] <= INDEX_BYTES) l++;
                if (l == f) l = f + 1;
                j->kind = J_INDEX;
                j->index = -1;
                j->index_mate = m;
                j->index_first = f;
                j->load_off[0] = j->load_off[1] = 0;
                j->load_len[0] = j->load_len[1] = 0;
                j->load_off[m] = inf[m].moff[f];
                j->load_len[m] = inf[m].moff[l] - inf[m].moff[f];
                j->moff[m].resize(l - f + 1);
                j->ooff[m].resize(l - f + 1);
                uint64_t t = 0;
                for (size_t i = f; i <= l; i++) {
                    j->moff[m][i - f] = (uint32_t)(inf[m].moff[i] - inf[m].moff[f]);
                    j->ooff[m][i - f] = (uint32_t)t;
                    if (i < l) t += inf[m].isize[i];
                }
                const size_t need = (size_t)j->load_len[m] + 64;
                if (j->in_buf[m].cap < need && !j->in_buf[m].reserve(need + need / 8, 0)) {
                    sh.fail(CSQ_ERR_NOMEM, "out of host memory for an index range");
                    break;
                }
                next_index_member[m] = l;
                {
                    std::lock_guard<std::mutex> g(ix_m);
                    index_jobs_out++;
                }
                load_and_ready(j);
                continue;
            }
            if (m_next < 0 && jobs_out == 0) {
                bool all = true;
                for (int m = 0; m < n_mates; m++) all = all && indexed[m] == inf[m].isize.size();
                if (all && total_records != UINT64_MAX) {  // fully indexed and still not covered: cannot happen with consistent counts
                    sh.fail(CSQ_ERR_FORMAT, "BGZF index does not cover the records it announced");
                    break;
                }
                if (all) continue;  // the totals are computed at the top of the loop
            }
            {  // wait for an index job to come back
                std::unique_lock<std::mutex> g(ix_m);
                const size_t b0 = indexed[0], b1 = indexed[1];
                absorb();
                if (indexed[0] == b0 && indexed[1] == b1) ix_cv.wait_for(g, std::chrono::milliseconds(20));
            }
        }
        finish();
    });

    // ---- GPU workers ----
    std::vector<std::thread> workers;
    std::vector<double> gpu_total((size_t)n_dev, 0.0), gpu_kernel((size_t)n_dev, 0.0);
    auto size_job_outputs = [&](Job& j, bool first_try) -> bool {
        uint64_t text[2] = {0, 0}, first[CSQ_N_DEST][2];
        for (int m = 0; m < n_mates; m++) text[m] = j.kind == J_BGZF ? (j.ooff[m].empty() ? 0 : j.ooff[m].back()) : j.tin.mate[m].bytes;
        output_sizes(text, j.kind == J_BGZF ? j.bin.n_reads : j.tin.n_reads, first);
        for (int m = 0; m < 2; m++)
            for (int d = 0; d < CSQ_N_DEST; d++) {
                const uint64_t want = first_try || m >= n_mates ? first[d][m] : j.out.text[d][m].bytes + 4096;
                if (want > j.outbuf[d][m].cap && !j.outbuf[d][m].reserve(want + want / 8, 0)) return false;
                j.out.text[d][m].data = j.outbuf[d][m].p;
                j.out.text[d][m].capacity = j.outbuf[d][m].cap;
            }
        return true;
    };
    for (int d = 0; d < n_dev; d++) {
        workers.emplace_back([&, d] {
            csq_plan* plan = plans[(size_t)d];
            std::deque<Job*> inflight;
            int next_slot = 0;
            auto finish_one = [&]() -> bool {
                Job* j = inflight.front();
                inflight.pop_front();
                int r = csq_wait(plan, j->slot);
                if (r == CSQ_ERR_CAPACITY) {  // grow to the reported sizes and fetch again
                    if (!size_job_outputs(*j, false)) {
                        sh.fail(CSQ_ERR_NOMEM, "out of host memory for output buffers");
                        return false;
                    }
                    r = csq_wait(plan, j->slot);
                }
                if (r) {
                    sh.fail(r, csq_last_error());
                    return false;
                }
                csq_slot_times(plan, j->slot, &j->total_ms, &j->kernel_ms);
                if (trace) fprintf(stderr, "[csq_run_files] %8.3f s  batch %ld back from GPU %d (%.1f ms)\n", seconds_since(t_start), j->index, d, j->total_ms);
                gpu_total[(size_t)d] += j->total_ms * 1e-3;
                gpu_kernel[(size_t)d] += j->kernel_ms * 1e-3;
                batch_done(j);
                return true;
            };
            for (;;) {
                if (sh.stop) break;
                // never sit on a finished batch: with one in flight and nothing ready, complete it first
                Job* j = nullptr;
                const int got = ready_q.try_pop(j);
                if (got < 0) break;
                if (got == 0) {
                    if (!inflight.empty()) {
                        if (!finish_one()) break;
                        continue;
                    }
                    if (!ready_q.pop(j)) break;
                }
                if (j->kind == J_INDEX) {
                    const int m = j->index_mate;
                    csq_bgzf_in bi;
                    memset(&bi, 0, sizeof(bi));
                    bi.data = j->in_buf[m].p;
                    bi.bytes = j->load_len[m];
                    bi.member_off = j->moff[m].data();
                    bi.text_off = j->ooff[m].data();
                    bi.n_members = (uint32_t)(j->moff[m].size() - 1);
                    std::vector<uint32_t> lines(bi.n_members);
                    int r = csq_bgzf_count_lines(plan, 2 + (next_slot & 1), &bi, lines.data());
                    if (r) {
                        sh.fail(r, csq_last_error());
                        break;
                    }
                    {
                        std::lock_guard<std::mutex> g(ix_m);
                        for (uint32_t i = 0; i < bi.n_members; i++) {
                            mlines[m][j->index_first + i] = lines[i];
                            mdone[m][j->index_first + i] = 1;
                        }
                    }
                    {
                        std::lock_guard<std::mutex> g(ix_m);
                        index_jobs_out--;
                    }
                    free_q.push(j);
                    ix_cv.notify_all();
                    continue;
                }
                if (!size_job_outputs(*j, true)) {
                    sh.fail(CSQ_ERR_NOMEM, "out of host memory for output buffers");
                    break;
                }
                j->slot = next_slot;
                next_slot ^= 1;
                int r = j->kind == J_BGZF ? csq_submit_bgzf(plan, j->slot, &j->bin, &j->out) : csq_submit_text(plan, j->slot, &j->tin, &j->out);
                if (r) {
                    sh.fail(r, csq_last_error());
                    break;
                }
                if (trace) fprintf(stderr, "[csq_run_files] %8.3f s  batch %ld submitted on GPU %d\n", seconds_since(t_start), j->index, d);
                inflight.push_back(j);
                if (inflight.size() == 2 && !finish_one()) break;
            }
            while (!sh.stop && !inflight.empty())
                if (!finish_one()) break;
        });
    }

    sequencer.join();
    for (auto& w : workers) w.join();
    stamp("workers done");
    {  // every batch written?
        std::unique_lock<std::mutex> g(w_m);
        w_cv.wait(g, [&] { return sh.stop || (n_batches >= 0 && written >= n_batches); });
    }
    stamp("writer done");
    warm_stop = true;
    free_q.close();

    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < 2; m++) {
            OutStream& o = outs[d][m];
            if (o.fd < 0) continue;
            if (o.gzip && o.pos == 0 && !sh.err_code) {  // an empty gzip file is still a valid (empty) member, like xopen writes
                std::vector<uint8_t> z;
                if (csqio::gzip_member((const uint8_t*)"", 0, o.level, z) || !full_write(o.fd, z.data(), z.size()))
                    sh.fail(CSQ_ERR_IO, "cannot write the empty gzip member");
            }
            if (close(o.fd) != 0 && !sh.err_code) sh.fail(CSQ_ERR_IO, "closing an output file failed");
            o.fd = -1;
            if (sh.err_code) unlink(o.path.c_str());  // no partial outputs behind a failed run
        }
    if (counters) {
        memset(counters, 0, sizeof(*counters));
        for (csq_plan* p : plans) {
            csq_counters c;
            if (csq_stats(p, &c) == 0) {
                uint64_t* dst = (uint64_t*)counters;
                const uint64_t* src = (const uint64_t*)&c;
                for (size_t w = 0; w < sizeof(csq_counters) / sizeof(uint64_t); w++) dst[w] += src[w];
            }
        }
    }
    if (timing) {
        memset(timing, 0, sizeof(*timing));
        timing->read_inflate = t_read.load();  // busy seconds of the loaders (or of the serial reader)
        timing->parse = 0;
        for (int d = 0; d < n_dev; d++) {
            timing->h2d_kernels_d2h += gpu_total[(size_t)d];
            timing->kernels += gpu_kernel[(size_t)d];
        }
        timing->write_deflate = t_write.load();
        timing->total = seconds_since(t_start);
    }
    stamp("outputs closed");
    // tear down side by side: un-pinning the jobs' host buffers and freeing the plans' device buffers are slow driver calls
    warm_owner.reset();  // (a run that ended early: the remaining buffers are still pinned and released right away)
    pool_owner.reset();  // joins the pool: no task refers to a job any more
    stamp("pools joined");
    {
        std::vector<std::thread> unpin;
        for (auto& j : jobs) unpin.emplace_back([&j] { j.reset(); });
        if (reader) csq_text_reader_close(reader);
        destroy_plans();
        stamp("plans destroyed");
        for (auto& t : unpin) t.join();
    }
    stamp("teardown done");
    if (sh.err_code) {
        csq_set_error(sh.err_msg.c_str());
        return sh.err_code;
    }
    return 0;
}
