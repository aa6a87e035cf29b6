// Host-side I/O helpers shared by fastq_io.cpp and pipeline.cpp (not part of the public ABI).
#pragma once

#include <stdint.h>
#include <stdio.h>

#include <string>
#include <vector>

#include "../../include/cutseq_b200.h"

namespace csqio {

int io_fail(int code, const char* fmt, ...);
const char* io_error();

struct PinnedBuf {  // growable host buffer, pinned when a CUDA context is available
    uint8_t* p = nullptr;
    size_t cap = 0;
    bool pinned = false;
    int kind = 0;        // 0 malloc, 1 cudaHostAlloc, 2 mmap + cudaHostRegister
    size_t map_len = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf&) = delete;
    PinnedBuf& operator=(const PinnedBuf&) = delete;
    ~PinnedBuf();
    bool reserve(size_t bytes, size_t keep, int touch_threads = 4);
    void release();
};

struct MateSoA {  // csq_mate_in backing store
    PinnedBuf seq, qual, seq_off, seq_len, name, name_off;
    uint32_t n = 0;
    uint64_t seq_bytes = 0, name_bytes = 0, total_bases = 0;
    void clear();
    bool presize(uint32_t reads, uint32_t read_len, uint32_t name_len);
    void view(csq_mate_in* mi) const;
};

struct ByteSource {
    void* gz = nullptr;
    std::string name;
    ~ByteSource();
    int open(const char* path);
    long read(uint8_t* dst, size_t n);
    void close();
};

struct MateParser {
    ByteSource src;
    std::vector<uint8_t> carry;
    size_t carry_pos = 0;
    bool eof = false;
    uint64_t line_no = 0;
    uint32_t hint_read_len = 0, hint_name_len = 0;  // pool sizing hints learnt from the first records
    int open(const char* path);
    int next(uint32_t max_reads, MateSoA& out);
};

// ---- text batches (text_reader.cpp) ----
uint64_t count_newlines(const uint8_t* p, size_t n);
uint64_t after_kth_newline(const uint8_t* p, size_t n, uint64_t k);  // offset one past the k-th '\n', UINT64_MAX if fewer
// FASTA record starts ('>' as the first byte of a line); `prev` is the byte in front of p ('\n' at a line start)
uint64_t count_fasta_records(const uint8_t* p, size_t n, uint8_t prev);
uint64_t kth_fasta_record(const uint8_t* p, size_t n, uint64_t k, uint8_t prev);  // offset of the k-th (k >= 1), UINT64_MAX if fewer

// How a byte stream is cut into batches of whole records: FASTQ after 4 k line ends, FASTA in front of the (k + 1)-th
// record start.  Counts and cuts work on pieces of the stream; `prev` is the byte in front of a piece.
struct RecordCut {
    bool fasta = false;
    uint64_t target(uint32_t max_reads) const { return fasta ? (uint64_t)max_reads + 1 : 4ull * max_reads; }
    uint64_t count(const uint8_t* p, size_t n, uint8_t prev) const {
        return fasta ? count_fasta_records(p, n, prev) : count_newlines(p, n);
    }
    uint64_t cut(const uint8_t* p, size_t n, uint64_t k, uint8_t prev) const {
        return fasta ? kth_fasta_record(p, n, k, prev) : after_kth_newline(p, n, k);
    }
    // a piece counted without its `prev` (pieces counted side by side): the record start it may hold at offset 0
    uint64_t edge(const uint8_t* p, size_t n, uint8_t prev) const { return fasta && n && p[0] == '>' && prev == '\n' ? 1 : 0; }
};

// gzip / DEFLATE decoder (inflate.cpp): whole compressed input in memory, output into the caller's buffer in
// pieces of any size.
class Inflater {
   public:
    Inflater();
    ~Inflater();
    Inflater(const Inflater&) = delete;
    Inflater& operator=(const Inflater&) = delete;
    void reset(const uint8_t* data, size_t n);
    long read(uint8_t* dst, size_t n);  // bytes produced (< n only at the end of the input), -1 on error
    const char* error() const { return err_ ? err_ : ""; }

   private:
    struct Tables;
    enum State { S_HEADER, S_BLOCK, S_STORED, S_HUFFMAN, S_TRAILER, S_DONE, S_ERROR };
    bool need(int n);
    uint32_t take(int n);
    void align_to_byte();
    bool fail(const char* msg);
    bool parse_header();
    bool parse_block_header();
    uint8_t hist_byte(const uint8_t* base, const uint8_t* out, uint32_t dist) const;
    uint8_t* run_huffman(uint8_t* base, uint8_t* out, uint8_t* out_end);
    Tables* t_;
    const uint8_t *in_ = nullptr, *in_end_ = nullptr;
    uint64_t bitbuf_ = 0;
    int bits_ = 0;
    State state_ = S_HEADER;
    bool last_block_ = false;
    uint32_t stored_left_ = 0, pend_len_ = 0, pend_dist_ = 0;
    uint8_t win_[32768];
    size_t win_len_ = 0;
    uint32_t crc_ = 0, isize_ = 0;
    uint64_t members_ = 0;
    const char* err_ = nullptr;
};

uint32_t crc32_fast(uint32_t crc, const uint8_t* p, size_t n);  // zlib's crc32() semantics, PCLMULQDQ folding where there is one

// Ordinary (single-stream) gzip files decoded by several threads at once (pinflate.cpp): same interface as Inflater.
class ParallelInflater {
   public:
    ParallelInflater(const uint8_t* data, size_t n, int threads);
    ~ParallelInflater();
    ParallelInflater(const ParallelInflater&) = delete;
    ParallelInflater& operator=(const ParallelInflater&) = delete;
    long read(uint8_t* dst, size_t n);  // bytes produced (< n only at the end of the input), -1 on error
    const char* error() const;
    struct Impl;

   private:
    Impl* p_;
};

// Ordinary gzip files decoded on a GPU (gz_stream.cu, csq_gz_stream_inflate), or by its host twin (device < 0): same
// interface as Inflater.  (The file driver keeps ParallelInflater: on one B200 box this decoder was measured slower on
// the files.gzip workload, DESIGN.md section 4.6.)
// Span and round sizes in compressed bytes, 0: the default (CSQ_GZ_STREAM_SPAN / CSQ_GZ_STREAM_ROUND, else 128 KiB and
// 64 MiB).  chain_log, when given, receives every span of the decode chain in file order.
struct ChainEntry {
    uint64_t start_bit, end_bit;
    uint32_t n_sym;
};
class GzStreamInflater {
   public:
    GzStreamInflater(const uint8_t* data, size_t n, int device, uint64_t span_bytes = 0, uint64_t round_bytes = 0,
                     std::vector<ChainEntry>* chain_log = nullptr);
    ~GzStreamInflater();
    GzStreamInflater(const GzStreamInflater&) = delete;
    GzStreamInflater& operator=(const GzStreamInflater&) = delete;
    long read(uint8_t* dst, size_t n);  // bytes produced (< n only at the end of the input), -1 on error
    const char* error() const;
    struct Impl;

   private:
    Impl* p_;
};

struct RawSource {  // decompressed byte stream of a plain or gzip (multi-member) file, read into caller memory
    int fd = -1;
    bool gz = false, file_eof = false, stream_end = false;
    void* zs = nullptr;            // zlib stream (CSQ_ZLIB_INFLATE=1: A/B runs against the built-in decoder)
    Inflater* fast = nullptr;      // built-in decoder over the mmap-ed file
    ParallelInflater* par = nullptr;  // ... by several threads (files of 16 MB and more)
    const uint8_t* map = nullptr;
    size_t map_len = 0;
    std::vector<uint8_t> inbuf;
    size_t in_pos = 0, in_len = 0;
    std::string name;
    ~RawSource();
    int open(const char* path);
    long read(uint8_t* dst, size_t n);
    long fill();
    void close();
};

struct MateTextReader {  // cuts the byte stream of one mate into batches of whole records
    RawSource src;
    RecordCut rc;
    std::vector<uint8_t> carry;  // bytes behind the last cut
    size_t carry_pos = 0;
    bool eof = false;
    uint64_t records_done = 0;
    size_t hint_bytes = 0;       // size of the previous batch: the next buffer is reserved in one go
    // plain regular files: several threads pread() disjoint pieces of the next batch straight into the pinned buffer
    // and count their line ends (the page-cache copy of one thread, ~1.5 GB/s in a VM, is what bounded whole-file runs)
    bool plain_file = false;
    uint64_t file_off = 0, file_size = 0;
    int read_threads = 1;
    int open(const char* path);
    int next(uint32_t max_reads, PinnedBuf& buf, uint64_t* bytes, uint32_t* n_reads);
    int next_plain(uint32_t max_reads, PinnedBuf& buf, uint64_t* bytes, uint32_t* n_reads);
    // BGZF (bgzip) files: every member carries its compressed size in a 'BC' extra field and its uncompressed size
    // in the trailer, so the members of the next batch are inflated side by side straight into the pinned buffer
    bool bgzf = false;
    uint64_t gz_off = 0;         // file offset of the next member
    int next_bgzf(uint32_t max_reads, PinnedBuf& buf, uint64_t* bytes, uint32_t* n_reads);
    int finish_at_eof(PinnedBuf& buf, size_t pos, uint64_t lines, uint64_t* bytes, uint32_t* n_reads);
    int finish_fasta_at_eof(PinnedBuf& buf, size_t pos, uint64_t* bytes, uint32_t* n_reads);
};

int parse_records(const uint8_t* text, size_t n_bytes, bool at_eof, uint32_t max_reads, MateSoA& out, size_t* consumed,
                  uint64_t* line_no, const char* fname);

struct OutFile {
    FILE* f = nullptr;
    std::string path;
    bool gzip = false, wrote_any = false;
    int gz_level = 1;
    int open(const char* p, int level);
    int write_raw(const uint8_t* data, size_t n);
    int close();
};

int gzip_member(const uint8_t* src, size_t n, int level, std::vector<uint8_t>& dst);

}  // namespace csqio
