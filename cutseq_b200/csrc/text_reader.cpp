// Host side of text batches: the reader only moves bytes.  It inflates (or reads) the input
// straight into pinned memory, counts line ends to cut the stream at a record boundary
// (4 lines per record, the same number of records for both mates; FASTA: record starts, '>' at the
// start of a line) and hands the bytes to
// csq_submit_text; FASTQ parsing and validation happen on the device (parse.cu).
// Stands where xopen + dnaio's chunked reader (read_paired_chunks) sit behind cutadapt's
// InputPaths in the reference (run.py:434-436, 751-753).
#include <errno.h>
#include <fcntl.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <atomic>
#include <thread>

#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include "host_io.h"

void csq_set_error(const char* msg);

namespace csqio {

uint64_t count_newlines(const uint8_t* p, size_t n) {
    uint64_t c = 0;
    size_t i = 0;
#if defined(__SSE2__)
    const __m128i nl = _mm_set1_epi8('\n');
    for (; i + 64 <= n; i += 64) {
        const unsigned m0 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(p + i)), nl));
        const unsigned m1 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(p + i + 16)), nl));
        const unsigned m2 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(p + i + 32)), nl));
        const unsigned m3 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(p + i + 48)), nl));
        c += (unsigned)__builtin_popcountll((uint64_t)m0 | ((uint64_t)m1 << 16) | ((uint64_t)m2 << 32) | ((uint64_t)m3 << 48));
    }
#endif
    for (; i < n; i++) c += p[i] == '\n';
    return c;
}

uint64_t after_kth_newline(const uint8_t* p, size_t n, uint64_t k) {
    if (k == 0) return 0;
    // skip whole 4 KiB blocks by count, then walk the block that holds the k-th line end
    size_t i = 0;
    while (i < n) {
        const size_t len = n - i < 4096 ? n - i : 4096;
        const uint64_t c = count_newlines(p + i, len);
        if (c >= k) break;
        k -= c;
        i += len;
    }
    while (i < n) {
        const uint8_t* q = (const uint8_t*)memchr(p + i, '\n', n - i);
        if (!q) return UINT64_MAX;
        i = (size_t)(q - p) + 1;
        if (--k == 0) return i;
    }
    return UINT64_MAX;
}

#if defined(__SSE2__)
// bit i set <=> p[i] == c, for the 64 bytes at p
static inline uint64_t eq_mask64(const uint8_t* p, __m128i c) {
    const uint64_t m0 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)p), c));
    const uint64_t m1 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(p + 16)), c));
    const uint64_t m2 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(p + 32)), c));
    const uint64_t m3 = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(_mm_loadu_si128((const __m128i*)(p + 48)), c));
    return m0 | (m1 << 16) | (m2 << 32) | (m3 << 48);
}
#endif

uint64_t count_fasta_records(const uint8_t* p, size_t n, uint8_t prev) {
    uint64_t c = 0, line_start = prev == '\n' ? 1 : 0;
    size_t i = 0;
#if defined(__SSE2__)
    const __m128i gt = _mm_set1_epi8('>'), nl = _mm_set1_epi8('\n');
    for (; i + 64 <= n; i += 64) {
        const uint64_t g = eq_mask64(p + i, gt), l = eq_mask64(p + i, nl);
        c += (uint64_t)__builtin_popcountll(g & ((l << 1) | line_start));
        line_start = l >> 63;
    }
#endif
    for (; i < n; i++) {
        c += p[i] == '>' && line_start;
        line_start = p[i] == '\n';
    }
    return c;
}

uint64_t kth_fasta_record(const uint8_t* p, size_t n, uint64_t k, uint8_t prev) {
    if (k == 0) return UINT64_MAX;
    // skip whole 4 KiB blocks by count, then walk the block that holds the k-th record start
    size_t i = 0;
    while (i < n) {
        const size_t len = n - i < 4096 ? n - i : 4096;
        const uint64_t c = count_fasta_records(p + i, len, i ? p[i - 1] : prev);
        if (c >= k) break;
        k -= c;
        i += len;
    }
    uint8_t before = i ? p[i - 1] : prev;
    for (; i < n; i++) {
        if (p[i] == '>' && before == '\n' && --k == 0) return i;
        before = p[i];
    }
    return UINT64_MAX;
}

// ---- decompressed byte stream of one input file --------------------------------------------
RawSource::~RawSource() { close(); }

void RawSource::close() {
    delete fast;
    fast = nullptr;
    delete par;
    par = nullptr;
    if (map) munmap((void*)map, map_len);
    map = nullptr;
    map_len = 0;
    if (zs) {
        inflateEnd((z_stream*)zs);
        delete (z_stream*)zs;
        zs = nullptr;
    }
    if (fd >= 0) ::close(fd);
    fd = -1;
}

long RawSource::fill() {
    in_pos = 0;
    in_len = 0;
    for (;;) {
        ssize_t got = ::read(fd, inbuf.data(), inbuf.size());
        if (got < 0) {
            if (errno == EINTR) continue;
            io_fail(CSQ_ERR_IO, "read error in %s: %s", name.c_str(), strerror(errno));
            return -1;
        }
        in_len = (size_t)got;
        return (long)got;
    }
}

static std::atomic<int> g_streams_side_by_side(2);

int RawSource::open(const char* path) {
    close();
    name = path;
    fd = ::open(path, O_RDONLY);
    if (fd < 0) return io_fail(CSQ_ERR_IO, "cannot open %s: %s", path, strerror(errno));
#ifdef POSIX_FADV_SEQUENTIAL
    posix_fadvise(fd, 0, 0, POSIX_FADV_SEQUENTIAL);
#endif
    inbuf.resize(1u << 20);
    file_eof = stream_end = false;
    if (fill() < 0) return CSQ_ERR_IO;
    gz = in_len >= 2 && inbuf[0] == 0x1f && inbuf[1] == 0x8b;
    const char* use_zlib = getenv("CSQ_ZLIB_INFLATE");
    struct stat sb;
    // the built-in decoder sees the whole compressed file at once (mmap); a pipe (stdin, process substitution) streams
    // through zlib instead
    const bool mappable = fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size > 0;
    if (gz && mappable && !(use_zlib && use_zlib[0] == '1')) {
        void* m = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m == MAP_FAILED) return io_fail(CSQ_ERR_IO, "cannot map %s: %s", path, strerror(errno));
        madvise(m, (size_t)sb.st_size, MADV_SEQUENTIAL);
        map = (const uint8_t*)m;
        map_len = (size_t)sb.st_size;
        // large files: several threads decode the one stream (pinflate.cpp); CSQ_INFLATE_THREADS=1 keeps the serial decoder
        const char* pt = getenv("CSQ_INFLATE_THREADS");
        const unsigned hw = std::thread::hardware_concurrency();
        // the host's cores are shared by the mates that are read side by side (csq_text_reader_open says how many)
        const unsigned share = (unsigned)std::max(1, g_streams_side_by_side.load());
        int threads = pt ? atoi(pt) : (int)std::min(16u, std::max(2u, hw / share));
        const char* pm = getenv("CSQ_PINFLATE_MIN");  // smallest file that is worth the threads (tests lower it)
        const size_t min_len = pm ? (size_t)atol(pm) : (size_t)(16u << 20);
        if (map_len >= min_len && threads > 1) {
            par = new ParallelInflater(map, map_len, threads);
            return 0;
        }
        fast = new Inflater();
        fast->reset(map, map_len);
        return 0;
    }
    if (gz) {
        z_stream* z = new z_stream();
        memset(z, 0, sizeof(*z));
        if (inflateInit2(z, 15 + 16) != Z_OK) {
            delete z;
            return io_fail(CSQ_ERR_IO, "inflateInit2 failed for %s", path);
        }
        zs = z;
    }
    return 0;
}

// Up to n decompressed bytes into dst; 0 at the end of the input, -1 on error.
long RawSource::read(uint8_t* dst, size_t n) {
    size_t done = 0;
    if (!gz) {
        if (in_pos < in_len) {  // what open() read while looking at the magic bytes
            const size_t c = in_len - in_pos < n ? in_len - in_pos : n;
            memcpy(dst, inbuf.data() + in_pos, c);
            in_pos += c;
            done = c;
        }
        while (done < n && !file_eof) {
            ssize_t got = ::read(fd, dst + done, n - done);
            if (got < 0) {
                if (errno == EINTR) continue;
                io_fail(CSQ_ERR_IO, "read error in %s: %s", name.c_str(), strerror(errno));
                return -1;
            }
            if (got == 0) file_eof = true;
            done += (size_t)got;
        }
        return (long)done;
    }
    if (par) {
        const long got = par->read(dst, n);
        if (got < 0) {
            io_fail(CSQ_ERR_IO, "%s: %s", name.c_str(), par->error());
            return -1;
        }
        return got;
    }
    if (fast) {
        const long got = fast->read(dst, n);
        if (got < 0) {
            io_fail(CSQ_ERR_IO, "%s: %s", name.c_str(), fast->error());
            return -1;
        }
        return got;
    }
    z_stream* z = (z_stream*)zs;
    while (done < n) {
        if (in_pos == in_len && !file_eof) {
            const long got = fill();
            if (got < 0) return -1;
            if (got == 0) file_eof = true;
        }
        if (stream_end) {
            // another gzip member may follow (concatenated members are one valid gzip file); zero padding is ignored
            while (in_pos < in_len && inbuf[in_pos] == 0) in_pos++;
            if (in_pos == in_len) {
                if (file_eof) break;
                continue;
            }
            if (inflateReset(z) != Z_OK) {
                io_fail(CSQ_ERR_IO, "inflateReset failed for %s", name.c_str());
                return -1;
            }
            stream_end = false;
        }
        if (in_pos == in_len && file_eof) {
            io_fail(CSQ_ERR_IO, "%s: compressed file ended before the end-of-stream marker was reached", name.c_str());
            return -1;
        }
        z->next_in = inbuf.data() + in_pos;
        z->avail_in = (uInt)(in_len - in_pos);
        z->next_out = dst + done;
        const size_t room = n - done < (1u << 30) ? n - done : (1u << 30);
        z->avail_out = (uInt)room;
        const int rc = inflate(z, Z_NO_FLUSH);
        in_pos = in_len - z->avail_in;
        done += room - z->avail_out;
        if (rc == Z_STREAM_END) {
            stream_end = true;
        } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
            io_fail(CSQ_ERR_IO, "%s: inflate failed (%d: %s)", name.c_str(), rc, z->msg ? z->msg : "?");
            return -1;
        }
    }
    return (long)done;
}

static size_t bgzf_member_size(const uint8_t* p, size_t n);

int MateTextReader::open(const char* path) {
    carry.clear();
    carry_pos = 0;
    eof = false;
    records_done = 0;
    plain_file = false;
    file_off = file_size = 0;
    const int rc = src.open(path);
    if (rc) return rc;
    struct stat sb;
    bgzf = false;
    gz_off = 0;
    if (src.gz && src.map && bgzf_member_size(src.map, src.map_len)) {
        bgzf = true;
        const char* env = getenv("CSQ_READ_THREADS");
        read_threads = env ? atoi(env) : (int)(std::thread::hardware_concurrency() / 3);
        if (!env && read_threads > 8) read_threads = 8;
        if (read_threads < 1) read_threads = 1;
        if (read_threads > 16) read_threads = 16;
    }
    if (!src.gz && fstat(src.fd, &sb) == 0 && S_ISREG(sb.st_mode)) {
        plain_file = true;
        file_size = (uint64_t)sb.st_size;
        const char* env = getenv("CSQ_READ_THREADS");
        const unsigned hw = std::thread::hardware_concurrency();
        read_threads = env ? atoi(env) : (int)(hw / 3);  // two mates read side by side; a third of the cores each, at most 8
        if (!env && read_threads > 8) read_threads = 8;
        if (read_threads < 1) read_threads = 1;
        if (read_threads > 16) read_threads = 16;
    }
    return 0;
}

// Length of the BGZF member at p (n bytes left in the file), 0 if it is not one: gzip header with FEXTRA holding
// the subfield 'B' 'C' of two bytes = total member size - 1 (SAM/BAM specification, section 4.1).
static size_t bgzf_member_size(const uint8_t* p, size_t n) {
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

int MateTextReader::next_bgzf(uint32_t max_reads, PinnedBuf& buf, uint64_t* bytes, uint32_t* n_reads) {
    const uint64_t target = rc.target(max_reads);
    *bytes = 0;
    *n_reads = 0;
    size_t pos = 0;      // bytes in buf
    uint64_t lines = 0;  // line ends among them
    const size_t avail = carry.size() - carry_pos;
    if (avail) {  // what the previous batch left behind its cut
        const uint8_t* c = carry.data() + carry_pos;
        const uint64_t k = rc.count(c, avail, '\n');
        if (k >= target) {
            const uint64_t cut = rc.cut(c, avail, target, '\n');
            if (!buf.reserve((size_t)cut + 64, 0)) return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
            memcpy(buf.p, c, (size_t)cut);
            carry_pos += (size_t)cut;
            *bytes = cut;
            *n_reads = max_reads;
            records_done += max_reads;
            return 0;
        }
        if (!buf.reserve(avail + 64, 0)) return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
        memcpy(buf.p, c, avail);
        pos = avail;
        lines = k;
    }
    carry.clear();
    carry_pos = 0;
    struct Member {
        const uint8_t* p;
        size_t clen, isize, out_off;
        uint64_t lines;
        const char* err;
    };
    std::vector<Member> mems;
    size_t want = hint_bytes ? hint_bytes + hint_bytes / 32 + (128u << 10) : (size_t)max_reads * 384 + (128u << 10);
    while (gz_off < src.map_len) {
        // the members that hold the next `round` bytes
        const size_t round = want > pos ? want - pos : (size_t)(64u << 10);
        mems.clear();
        size_t acc = 0;
        while (acc < round && gz_off < src.map_len) {
            const uint8_t* p = src.map + gz_off;
            const size_t left = src.map_len - (size_t)gz_off;
            const size_t total = bgzf_member_size(p, left);
            if (!total) return io_fail(CSQ_ERR_IO, "%s: not a BGZF member at offset %llu (the file started as BGZF)", src.name.c_str(), (unsigned long long)gz_off);
            const size_t isize = p[total - 4] | ((size_t)p[total - 3] << 8) | ((size_t)p[total - 2] << 16) | ((size_t)p[total - 1] << 24);
            mems.push_back(Member{p, total, isize, pos + acc, 0, nullptr});
            acc += isize;
            gz_off += total;
        }
        if (!buf.reserve(pos + acc + 64, pos)) return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
        std::atomic<size_t> cursor{0};
        auto work = [&] {
            Inflater inf;
            for (;;) {
                const size_t i = cursor++;
                if (i >= mems.size()) return;
                Member& mb = mems[i];
                inf.reset(mb.p, mb.clen);
                size_t done = 0;
                while (done < mb.isize) {
                    const long got = inf.read(buf.p + mb.out_off + done, mb.isize - done);
                    if (got <= 0) break;
                    done += (size_t)got;
                }
                uint8_t probe;
                if (done != mb.isize || inf.read(&probe, 1) != 0) {
                    mb.err = inf.error()[0] ? "corrupt BGZF member" : "BGZF member size does not match its trailer";
                    continue;
                }
                mb.lines = rc.count(buf.p + mb.out_off, mb.isize, 0);  // + the record start at its edge, below
            }
        };
        int nt = read_threads;
        if ((size_t)nt > mems.size()) nt = (int)mems.size();
        std::vector<std::thread> helpers;
        for (int t = 1; t < nt; t++) helpers.emplace_back(work);
        work();
        for (auto& th : helpers) th.join();
        for (Member& mb : mems) {
            if (mb.err) return io_fail(CSQ_ERR_IO, "%s: %s", src.name.c_str(), mb.err);
            mb.lines += rc.edge(buf.p + mb.out_off, mb.isize, mb.out_off ? buf.p[mb.out_off - 1] : '\n');
        }
        for (const Member& mb : mems) {
            if (lines + mb.lines >= target) {
                const uint64_t rel = rc.cut(buf.p + mb.out_off, mb.isize, target - lines, mb.out_off ? buf.p[mb.out_off - 1] : '\n');
                const size_t cut = mb.out_off + (size_t)rel;
                carry.assign(buf.p + cut, buf.p + pos + acc);
                hint_bytes = cut;
                *bytes = cut;
                *n_reads = max_reads;
                records_done += max_reads;
                return 0;
            }
            lines += mb.lines;
        }
        pos += acc;
        want = pos + pos / 8 + (256u << 10);
    }
    eof = true;
    return finish_at_eof(buf, pos, lines, bytes, n_reads);
}

// End of the input: a missing final line end is accepted, and so are blank lines behind the last record (dnaio).
int MateTextReader::finish_at_eof(PinnedBuf& buf, size_t pos, uint64_t lines, uint64_t* bytes, uint32_t* n_reads) {
    if (rc.fasta) return finish_fasta_at_eof(buf, pos, bytes, n_reads);
    if (pos && buf.p[pos - 1] != '\n') {
        if (!buf.reserve(pos + 64, pos)) return io_fail(CSQ_ERR_NOMEM, "out of host memory");
        buf.p[pos++] = '\n';
        lines++;
    }
    while (lines % 4 != 0 && pos >= 2) {
        size_t q = pos - 1;  // buf[q] == '\n'
        if (q >= 1 && buf.p[q - 1] == '\r') q--;
        if (q >= 1 && buf.p[q - 1] == '\n') {  // the last line is blank: drop it
            pos = q;
            lines--;
        } else {
            break;
        }
    }
    if (lines == 1 && pos <= 2) {  // a file of just "\n"
        pos = 0;
        lines = 0;
    }
    if (lines % 4 != 0)
        return io_fail(CSQ_ERR_FORMAT, "%s: FASTQ file ended prematurely (line %llu)", src.name.c_str(),
                       (unsigned long long)(4 * records_done + lines + 1));
    *bytes = pos;
    *n_reads = (uint32_t)(lines / 4);
    records_done += lines / 4;
    return 0;
}

// FASTA: every record start left is a record of the batch; a missing final line end is added.  Text without a record
// (only possible in front of the first one) must be blank.
int MateTextReader::finish_fasta_at_eof(PinnedBuf& buf, size_t pos, uint64_t* bytes, uint32_t* n_reads) {
    const uint64_t n = count_fasta_records(buf.p, pos, '\n');
    if (n == 0) {
        for (size_t i = 0; i < pos; i++)
            if (buf.p[i] != ' ' && (buf.p[i] < 9 || buf.p[i] > 13))
                return io_fail(CSQ_ERR_FORMAT, "%s: FASTA input does not start with a '>' header (line %llu)", src.name.c_str(),
                               (unsigned long long)(count_newlines(buf.p, i) + 1));
        pos = 0;
    } else if (buf.p[pos - 1] != '\n') {
        if (!buf.reserve(pos + 64, pos)) return io_fail(CSQ_ERR_NOMEM, "out of host memory");
        buf.p[pos++] = '\n';
    }
    *bytes = pos;
    *n_reads = (uint32_t)n;
    records_done += n;
    return 0;
}

// Plain regular file: the next batch is [file_off, file_off + cut).  Its size is known to within a few per cent
// from the previous batch, so `read_threads` threads pread() disjoint pieces of that range at once and count
// their line ends; nothing is carried over between batches (what lies behind the cut is read again next time,
// from the page cache).
int MateTextReader::next_plain(uint32_t max_reads, PinnedBuf& buf, uint64_t* bytes, uint32_t* n_reads) {
    const uint64_t target = rc.target(max_reads);
    *bytes = 0;
    *n_reads = 0;
    if (file_off >= file_size) {
        eof = true;
        return 0;
    }
    size_t pos = 0;        // bytes of the file, from file_off on, that are in buf
    uint64_t lines = 0;    // line ends among them
    size_t want = hint_bytes ? hint_bytes + hint_bytes / 32 + (64u << 10) : (size_t)max_reads * 384 + (64u << 10);
    struct Piece {
        size_t begin, len;
        uint64_t lines;
        long got;
        int err;
    };
    std::vector<Piece> pieces;  // of the most recent round, in file order
    for (;;) {
        const uint64_t left = file_size - (file_off + pos);
        size_t round = want > pos ? want - pos : (size_t)0;
        if (round > left) round = (size_t)left;
        if (round == 0) break;  // the whole rest of the file is here
        if (!buf.reserve(pos + round + 64, pos)) return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
        int nt = read_threads;
        if ((size_t)nt > round / (1u << 20) + 1) nt = (int)(round / (1u << 20) + 1);  // at least 1 MiB per thread
        pieces.assign((size_t)nt, Piece{0, 0, 0, 0, 0});
        const size_t per = (round + (size_t)nt - 1) / (size_t)nt;
        for (int t = 0; t < nt; t++) {
            pieces[(size_t)t].begin = pos + (size_t)t * per;
            const size_t end = pos + ((size_t)(t + 1) * per < round ? (size_t)(t + 1) * per : round);
            pieces[(size_t)t].len = end > pieces[(size_t)t].begin ? end - pieces[(size_t)t].begin : 0;
        }
        auto work = [&](int t) {
            Piece& pc = pieces[(size_t)t];
            size_t done = 0;
            while (done < pc.len) {
                const ssize_t got = pread(src.fd, buf.p + pc.begin + done, pc.len - done, (off_t)(file_off + pc.begin + done));
                if (got < 0) {
                    if (errno == EINTR) continue;
                    pc.err = errno;
                    break;
                }
                if (got == 0) break;  // the file shrank under us
                done += (size_t)got;
            }
            pc.got = (long)done;
            pc.lines = rc.count(buf.p + pc.begin, done, 0);  // + the record start at its edge, below
        };
        std::vector<std::thread> helpers;
        for (int t = 1; t < nt; t++) helpers.emplace_back(work, t);
        work(0);
        for (auto& th : helpers) th.join();
        bool short_read = false;
        for (int t = 0; t < nt; t++) {
            const Piece& pc = pieces[(size_t)t];
            if (pc.err) return io_fail(CSQ_ERR_IO, "read error in %s: %s", src.name.c_str(), strerror(pc.err));
            if ((size_t)pc.got != pc.len) short_read = true;
        }
        if (short_read) return io_fail(CSQ_ERR_IO, "%s: file changed while it was read", src.name.c_str());
        // is the last line end (FASTA: the first record start behind the batch) inside this round?
        for (int t = 0; t < nt; t++) {
            Piece& pc = pieces[(size_t)t];
            const uint8_t prev = pc.begin ? buf.p[pc.begin - 1] : (uint8_t)'\n';
            pc.lines += rc.edge(buf.p + pc.begin, pc.len, prev);
            if (lines + pc.lines >= target) {
                const uint64_t rel = rc.cut(buf.p + pc.begin, pc.len, target - lines, prev);
                const size_t cut = pc.begin + (size_t)rel;
                file_off += cut;
                hint_bytes = cut;
                *bytes = cut;
                *n_reads = max_reads;
                records_done += max_reads;
                return 0;
            }
            lines += pc.lines;
        }
        pos += round;
        want = pos + pos / 8 + (256u << 10);  // not enough line ends yet: longer records than the previous batch had
    }
    // the rest of the file holds fewer than max_reads records
    eof = true;
    file_off = file_size;
    return finish_at_eof(buf, pos, lines, bytes, n_reads);
}

// The next max_reads records (fewer at the end of the input) as raw text into buf.
int MateTextReader::next(uint32_t max_reads, PinnedBuf& buf, uint64_t* bytes, uint32_t* n_reads) {
    if (plain_file) return next_plain(max_reads, buf, bytes, n_reads);
    if (bgzf) return next_bgzf(max_reads, buf, bytes, n_reads);
    const uint64_t target = rc.target(max_reads);
    size_t piece = (size_t)max_reads * 512;
    piece = piece < (64u << 10) ? (64u << 10) : piece > (4u << 20) ? (4u << 20) : piece;
    size_t pos = 0;
    uint64_t lines = 0;
    *bytes = 0;
    *n_reads = 0;
    const size_t avail = carry.size() - carry_pos;
    // pinned memory is expensive to grow: reserve what the previous batch needed (first batch: a guess)
    // (what a batch needs is its own size plus one piece; when that is not there, allocate it with 1/8 to spare, so
    // that batches a few bytes longer than the previous one do not trigger another - doubling - allocation)
    const size_t need = (hint_bytes ? hint_bytes : (size_t)max_reads * 96) + piece + 64;
    if (buf.cap < need && !buf.reserve(need + need / 8, 0))
        return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
    if (avail) {
        const uint8_t* c = carry.data() + carry_pos;
        const uint64_t k = rc.count(c, avail, '\n');
        if (k >= target) {  // the batch is already here
            const uint64_t cut = rc.cut(c, avail, target, '\n');
            if (!buf.reserve((size_t)cut + 64, 0)) return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
            memcpy(buf.p, c, (size_t)cut);
            carry_pos += (size_t)cut;
            *bytes = cut;
            *n_reads = max_reads;
            records_done += max_reads;
            return 0;
        }
        if (!buf.reserve(avail + piece + 64, 0)) return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
        memcpy(buf.p, c, avail);
        pos = avail;
        lines = k;
    }
    carry.clear();
    carry_pos = 0;
    size_t last_start = pos;      // start of the most recent piece, line ends before it
    uint64_t lines_before = lines;
    while (lines < target && !eof) {
        if (!buf.reserve(pos + piece + 64, pos)) return io_fail(CSQ_ERR_NOMEM, "out of host memory for a batch of %u reads", max_reads);
        const long got = src.read(buf.p + pos, piece);
        if (got < 0) return CSQ_ERR_IO;
        if (got == 0) {
            eof = true;
            break;
        }
        last_start = pos;
        lines_before = lines;
        lines += rc.count(buf.p + pos, (size_t)got, pos ? buf.p[pos - 1] : (uint8_t)'\n');
        pos += (size_t)got;
    }
    if (lines >= target) {
        const uint64_t rel = rc.cut(buf.p + last_start, pos - last_start, target - lines_before, last_start ? buf.p[last_start - 1] : (uint8_t)'\n');
        const size_t cut = last_start + (size_t)rel;
        carry.assign(buf.p + cut, buf.p + pos);
        hint_bytes = cut;
        *bytes = cut;
        *n_reads = max_reads;
        records_done += max_reads;
        return 0;
    }
    return finish_at_eof(buf, pos, lines, bytes, n_reads);
}

}  // namespace csqio

using namespace csqio;

struct csq_text_reader {
    MateTextReader mate[2];
    int n_mates = 1;
    uint64_t first_record = 0;
    PinnedBuf own[CSQ_N_SLOTS][2];
};

static int report(int rc) {
    if (rc) csq_set_error(io_error());
    return rc;
}

int csq_text_reader_next_into(csq_text_reader* r, csqio::PinnedBuf* bufs /*[2]*/, uint32_t max_reads, csq_batch_text* in) {
    int rcs[2] = {0, 0};
    char errs[2][512] = {"", ""};
    uint64_t bytes[2] = {0, 0};
    uint32_t n[2] = {0, 0};
    auto work = [&](int m) {
        rcs[m] = r->mate[m].next(max_reads, bufs[m], &bytes[m], &n[m]);
        if (rcs[m]) snprintf(errs[m], sizeof(errs[m]), "%s", io_error());
    };
    if (r->n_mates == 2) {
        std::thread t(work, 1);
        work(0);
        t.join();
    } else {
        work(0);
    }
    for (int m = 0; m < r->n_mates; m++)
        if (rcs[m]) {
            csq_set_error(errs[m]);
            return rcs[m];
        }
    if (r->n_mates == 2 && n[0] != n[1]) {
        csq_set_error("paired input files have different numbers of records");
        return CSQ_ERR_FORMAT;
    }
    memset(in, 0, sizeof(*in));
    in->n_reads = n[0];
    in->n_mates = (uint32_t)r->n_mates;
    in->first_record = r->first_record;
    r->first_record += n[0];
    for (int m = 0; m < r->n_mates; m++) {
        in->mate[m].text = bufs[m].p;
        in->mate[m].bytes = bytes[m];
    }
    return 0;
}

extern "C" {

int csq_text_reader_open(const char* path1, const char* path2, csq_text_reader** out) {
    return csq_text_reader_open_flags(path1, path2, 0, out);
}

int csq_text_reader_open_flags(const char* path1, const char* path2, uint32_t plan_flags, csq_text_reader** out) {
    if (!path1 || !out) {
        csq_set_error("null argument");
        return CSQ_ERR_INVALID;
    }
    csq_text_reader* r = new csq_text_reader();
    r->n_mates = path2 ? 2 : 1;
    for (int m = 0; m < 2; m++) r->mate[m].rc.fasta = (plan_flags & CSQ_PLAN_FASTA) != 0;
    g_streams_side_by_side = r->n_mates;
    int rc = r->mate[0].open(path1);
    if (!rc && path2) rc = r->mate[1].open(path2);
    if (rc) {
        delete r;
        return report(rc);
    }
    *out = r;
    return 0;
}

int csq_text_reader_next(csq_text_reader* r, int buffer, uint32_t max_reads, csq_batch_text* in) {
    if (!r || !in || buffer < 0 || buffer >= CSQ_N_SLOTS || max_reads == 0) {
        csq_set_error("bad argument");
        return CSQ_ERR_INVALID;
    }
    return csq_text_reader_next_into(r, r->own[buffer], max_reads, in);
}

void csq_text_reader_close(csq_text_reader* r) { delete r; }

// gzip data in memory -> dst, produced in pieces of `piece` bytes (exercises the decoder's resumption points)
int csq_gunzip_mem(const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t piece, uint64_t* out_n) {
    if (!src || !dst || !out_n || piece == 0) {
        csq_set_error("bad argument");
        return CSQ_ERR_INVALID;
    }
    Inflater inf;
    inf.reset(src, (size_t)n);
    uint64_t total = 0;
    for (;;) {
        const uint64_t want = cap - total < piece ? cap - total : piece;
        if (want == 0) {  // is there more?
            uint8_t probe;
            const long g = inf.read(&probe, 1);
            if (g < 0) break;
            *out_n = total;
            if (g == 0) return 0;
            csq_set_error("output buffer too small");
            return CSQ_ERR_CAPACITY;
        }
        const long got = inf.read(dst + total, (size_t)want);
        if (got < 0) break;
        total += (uint64_t)got;
        if ((uint64_t)got < want) {
            *out_n = total;
            return 0;
        }
    }
    csq_set_error(inf.error());
    return CSQ_ERR_IO;
}

uint64_t csq_count_newlines(const uint8_t* text, uint64_t n_bytes) { return text ? count_newlines(text, (size_t)n_bytes) : 0; }

uint64_t csq_after_kth_newline(const uint8_t* text, uint64_t n_bytes, uint64_t k) {
    return text ? after_kth_newline(text, (size_t)n_bytes, k) : UINT64_MAX;
}

uint64_t csq_after_kth_fasta_record(const uint8_t* text, uint64_t n_bytes, uint64_t k) {
    return text ? kth_fasta_record(text, (size_t)n_bytes, k + 1, '\n') : UINT64_MAX;
}

int csq_format_fastq(const csq_mate_in* mate, uint32_t n_reads, uint8_t* out, uint64_t capacity, uint64_t* bytes) {
    if (!mate || !bytes || (n_reads && !out)) {
        csq_set_error("null argument");
        return CSQ_ERR_INVALID;
    }
    uint64_t need = 0;
    for (uint32_t i = 0; i < n_reads; i++) need += (uint64_t)(mate->name_off[i + 1] - mate->name_off[i]) + 2ull * mate->seq_len[i] + 6;
    *bytes = need;
    if (need > capacity) {
        csq_set_error("caller buffer too small");
        return CSQ_ERR_CAPACITY;
    }
    uint8_t* p = out;
    for (uint32_t i = 0; i < n_reads; i++) {
        const uint32_t nl = mate->name_off[i + 1] - mate->name_off[i], sl = mate->seq_len[i];
        *p++ = '@';
        memcpy(p, mate->name + mate->name_off[i], nl);
        p += nl;
        *p++ = '\n';
        memcpy(p, mate->seq + mate->seq_off[i], sl);
        p += sl;
        *p++ = '\n';
        *p++ = '+';
        *p++ = '\n';
        memcpy(p, mate->qual + mate->seq_off[i], sl);
        p += sl;
        *p++ = '\n';
    }
    return 0;
}

}  // extern "C"
