// Native FASTA / FASTQ ingest (host only): file -> one contiguous byte-per-base buffer + record table.
//
// Stands in for what the reference takes from pyfastx (perfect_repeat_finder.py:117-137: iterate the records,
// `.name` = first whitespace-delimited token of the header, `.seq` = the record's lines joined, case preserved).
// Plain or gzip (multi-member / bgzip too).  The buffer is laid out exactly as crf_seq_load_ascii wants it
// (records back to back + n+1 offsets), so a whole file goes to the GPU with one call and no Python-side copy.
//
// Included at the end of crf_api.cu (shares set_err()).
#pragma once
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include "crf_codes.h"
#include "crf_inflate.h"

#include <atomic>
#include <exception>
#include <chrono>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>

enum HostKind { HOST_NONE, HOST_PINNED, HOST_HEAP, HOST_MAPPED };

// Gives a HostBuf's block back (a static function, so the destructor stays a one-line inline call and the library exports
// nothing new).
static void host_release(uint8_t *p, size_t size, HostKind kind) {
    if (kind == HOST_PINNED) cudaFreeHost(p);
    else if (kind == HOST_HEAP) free(p);
    else munmap(p, size);
}

// One block of host memory, given back the way it was obtained: page-locked (cudaHostAlloc), heap (malloc) or a mapping
// (munmap).  It uses nothing else from the CUDA runtime, so the reader builds without it (tests/fuzz_*.cpp stub these).
struct HostBuf {
    uint8_t *p = nullptr;
    size_t size = 0;
    HostKind kind = HOST_NONE;

    HostBuf() = default;
    HostBuf(const HostBuf &) = delete;
    HostBuf &operator=(const HostBuf &) = delete;
    HostBuf(HostBuf &&o) noexcept { *this = std::move(o); }
    HostBuf &operator=(HostBuf &&o) noexcept {           // (what this held goes with o)
        std::swap(p, o.p);
        std::swap(size, o.size);
        std::swap(kind, o.kind);
        return *this;
    }
    ~HostBuf() { if (p) host_release(p, size, kind); }
    bool pinned() const { return kind == HOST_PINNED; }

    // n >= 1 bytes, page-locked; false (nothing held) when there is no device or no page-locked memory left.
    bool pin(size_t n) {
        void *q = nullptr;
        if (cudaHostAlloc(&q, n, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return false; }
        p = (uint8_t *)q; size = n; kind = HOST_PINNED;
        return true;
    }
    // n >= 1 bytes, page-locked if asked and possible, else plain pages (2 MB ones when large).  false: out of memory.
    bool alloc(size_t n, bool page_locked) {
        if (page_locked && pin(n)) return true;
        if (!(p = (uint8_t *)malloc(n))) return false;
        size = n; kind = HOST_HEAP;
#if defined(__linux__) && defined(MADV_HUGEPAGE)
        if (n >= ((size_t)8 << 20)) {                    // gigabytes touched for the first time by their writer: 2 MB pages
            const uintptr_t lo = ((uintptr_t)p + 4095) & ~(uintptr_t)4095, hi = ((uintptr_t)p + n) & ~(uintptr_t)4095;
            if (hi > lo) madvise((void *)lo, hi - lo, MADV_HUGEPAGE);   // (advice only; the block is never realloc'ed)
        }
#endif
        return true;
    }
    // Takes over the mapping [m, m + n).
    void adopt(void *m, size_t n) { p = (uint8_t *)m; size = n; kind = HOST_MAPPED; }
};

// What crf_fasta_format returns.
enum FastaFormat { FORMAT_FASTA = 0, FORMAT_FASTQ = 1, FORMAT_2BIT = 2, FORMAT_BAM = 3 };

struct crf_fasta {
    std::vector<uint64_t> offsets;      // n_records + 1
    std::vector<uint64_t> name_off;     // into names (NUL-separated, record order: what crf_write_rows takes)
    std::vector<char> names;
    // The text (total bytes) and a FASTQ / BAM file's qualities laid out like it (kept with crf_fasta_open(pinned & 4)).
    // bases and quals are their addresses as plain pointers: always the buffers' own, whatever the buffers are reassigned.
    HostBuf bases_buf, quals_buf;
    uint8_t *&bases = bases_buf.p;
    uint8_t *&quals = quals_buf.p;
    uint64_t total = 0;
    // packed planes (crf_fasta_packed): H, L, NM of plane_words words each, one allocation
    HostBuf planes;
    uint64_t plane_words = 0;
    std::vector<uint64_t> exotic;
    FastaFormat format = FORMAT_FASTA;
    // .2bit and BAM: the bases as codes (crf_codes.h), record r's from byte rec_byte[r]; page-locked with pinned & 3.  The text
    // (bases) is decoded on the first crf_fasta_data.
    //   .2bit: the file's bytes as they are (else mapped); n_runs, mask_runs: its N blocks and mask blocks as sorted
    //   disjoint runs of concatenated positions.
    //   BAM: the reads' 4-bit codes with reverse complements applied (else an anonymous mapping); nib_exotic: codes other
    //   than A, C, G, T, N as (position in the offsets' space << 8 | letter), ascending.
    HostBuf codes;
    std::vector<uint64_t> rec_byte, n_runs, mask_runs, nib_exotic;
    std::mutex decode_mu;
    int pinned = 0;                                      // the pinned argument of crf_fasta_open
    uint32_t n_threads = 1;
};

namespace fasta_detail {

// The file's bytes: mapped when possible (pages are then faulted in by the worker threads, in parallel), else read.
struct FileBytes {
    const uint8_t *data = nullptr;
    size_t size = 0;
    void *map = nullptr;
    std::vector<uint8_t> owned;
    ~FileBytes() {
        if (map) munmap(map, size);
    }
};

static bool read_file(const char *path, std::vector<uint8_t> &out);

static bool open_bytes(const char *path, FileBytes &fb) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return false;
    struct stat st;
    if (fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
        void *m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m != MAP_FAILED) {
            madvise(m, (size_t)st.st_size, MADV_SEQUENTIAL);
            fb.map = m;
            fb.data = (const uint8_t *)m;
            fb.size = (size_t)st.st_size;
            close(fd);
            return true;
        }
    }
    close(fd);
    if (!read_file(path, fb.owned)) return false;
    fb.data = fb.owned.data();
    fb.size = fb.owned.size();
    return true;
}

static bool read_file(const char *path, std::vector<uint8_t> &out) {
    FILE *f = fopen(path, "rb");
    if (!f) return false;
    bool ok = true;
    if (fseeko(f, 0, SEEK_END) == 0) {
        const off_t n = ftello(f);
        rewind(f);
        if (n > 0) {
            out.resize((size_t)n);
            ok = fread(out.data(), 1, (size_t)n, f) == (size_t)n;
        }
    } else {                                            // not seekable (a pipe)
        uint8_t buf[1 << 16];
        size_t got;
        while ((got = fread(buf, 1, sizeof buf, f)) > 0) out.insert(out.end(), buf, buf + got);
        ok = !ferror(f);
    }
    fclose(f);
    return ok;
}

// gzip -> text; concatenated members (bgzip) are decoded one after the other
static bool inflate_all(const FileBytes &in, std::vector<uint8_t> &out) {
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, 16 + MAX_WBITS) != Z_OK) return false;
    out.resize(std::max<size_t>(in.size * 4, 1 << 16));
    size_t in_pos = 0, out_pos = 0;
    bool ok = true;
    int rc = Z_OK;
    while (in_pos < in.size) {
        if (out_pos == out.size()) out.resize(out.size() + out.size() / 2);
        const size_t in_chunk = std::min<size_t>(in.size - in_pos, 1u << 30);
        const size_t out_chunk = std::min<size_t>(out.size() - out_pos, 1u << 30);
        zs.next_in = const_cast<Bytef *>(in.data + in_pos);
        zs.avail_in = (uInt)in_chunk;
        zs.next_out = out.data() + out_pos;
        zs.avail_out = (uInt)out_chunk;
        rc = inflate(&zs, Z_NO_FLUSH);
        in_pos += in_chunk - zs.avail_in;
        out_pos += out_chunk - zs.avail_out;
        if (rc == Z_STREAM_END) {
            if (in_pos < in.size && inflateReset(&zs) != Z_OK) { ok = false; break; }
        } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
            ok = false;
            break;
        } else if (rc == Z_BUF_ERROR && zs.avail_in == 0 && in_pos == in.size) {
            ok = false;                                 // truncated stream
            break;
        }
    }
    inflateEnd(&zs);
    out.resize(out_pos);
    return ok && rc == Z_STREAM_END;                    // anything else: the last member is truncated
}

struct Piece {                                          // a slice of one record's body text
    uint64_t begin, end;                                // text range
    uint64_t out;                                       // where its bases go
    uint64_t n_eol;                                     // '\n' + '\r' bytes inside
};

static void run_parallel(unsigned n_threads, size_t n_items, const std::function<void(size_t)> &fn) {
    std::atomic<size_t> next{0};
    auto worker = [&]() {
        for (size_t i; (i = next.fetch_add(1)) < n_items;) fn(i);
    };
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < n_threads && t < n_items; ++t) {
        try {
            pool.emplace_back(worker);
        } catch (const std::exception &) {              // no more threads to be had: go on with those we have
            break;
        }
    }
    worker();
    for (auto &th : pool) th.join();
}

// BGZF (bgzip, what `samtools faidx` wants and the reference's Hail pipeline ships: run_hail_batch_pipeline.py:112 takes
// the .gzi next to the FASTA): every gzip member is a self-contained block of <= 64 KiB that says its own compressed size
// in a 'BC' extra field, so the blocks are found by hopping over the headers and inflated on all threads.
// A file that is not BGZF from the first to the last byte is inflated serially instead.
// Each block is decoded by the reader's own DEFLATE decoder (crf_inflate.h, ~2 x zlib on FASTA text) into a scratch buffer --
// its copies may write a few bytes beyond a match, which in the shared output would be the next block's -- and copied to its
// place once length and CRC-32 agree; a block it does not take (or CRF_GUNZIP_ZLIB=1) goes through zlib, which then decides.
// The whole-file output is a mapping of its own (no zero-fill before the blocks arrive, 2 MB pages).
struct BgzfBlock { uint64_t cdata, clen, out; uint32_t isize, crc; };

// The blocks of a BGZF file (false: not BGZF from the first to the last byte); *total = the inflated size.
static bool bgzf_index(const FileBytes &in, std::vector<BgzfBlock> &blocks, uint64_t *total_out) {
    using Block = BgzfBlock;
    const uint8_t *d = in.data;
    const uint64_t n = in.size;
    uint64_t pos = 0, total = 0;
    while (pos < n) {
        if (n - pos < 18 || d[pos] != 0x1f || d[pos + 1] != 0x8b || d[pos + 2] != 8 || !(d[pos + 3] & 4)) return false;
        const uint32_t xlen = d[pos + 10] | (d[pos + 11] << 8);
        if (n - pos < 12ull + xlen + 8) return false;
        uint32_t bsize = 0;
        for (uint32_t x = 0; x + 4 <= xlen;) {           // extra subfields: SI1 SI2 SLEN(2) data
            const uint8_t *f = d + pos + 12 + x;
            const uint32_t slen = f[2] | (f[3] << 8);
            if (f[0] == 'B' && f[1] == 'C' && slen == 2 && x + 6 <= xlen) bsize = (f[4] | (f[5] << 8)) + 1u;
            x += 4 + slen;
        }
        if (bsize < 12 + xlen + 8 || pos + bsize > n) return false;
        if (d[pos + 3] & ~4) return false;                // other header fields (name, comment, crc): not what bgzip writes
        Block b;
        b.cdata = pos + 12 + xlen;
        b.clen = bsize - 12 - xlen - 8;
        const uint8_t *tail = d + pos + bsize - 8;
        b.crc = tail[0] | (tail[1] << 8) | (tail[2] << 16) | ((uint32_t)tail[3] << 24);
        b.isize = tail[4] | (tail[5] << 8) | (tail[6] << 16) | ((uint32_t)tail[7] << 24);
        if (b.isize > 65536) return false;
        b.out = total;
        total += b.isize;
        blocks.push_back(b);
        pos += bsize;
    }
    *total_out = total;
    return true;
}

// Inflates BGZF blocks one after the other on one thread (a worker's state: scratch output, tables, a zlib stream).
struct BgzfInflater {
    const uint8_t *d;                                     // the file's bytes
    bool own_decoder = getenv("CRF_GUNZIP_ZLIB") == nullptr;
    crf_inflate::OutBuf scratch;
    crf_inflate::Tables tables;
    z_stream zs;
    bool zs_ready = false;
    explicit BgzfInflater(const uint8_t *data) : d(data) {}
    ~BgzfInflater() { if (zs_ready) inflateEnd(&zs); }
    // block b -> dst[0, b.isize); false if it is corrupt (length or CRC-32)
    bool run(const BgzfBlock &b, uint8_t *dst) {
        if (b.isize == 0) return true;                    // the empty end-of-file block
        if (own_decoder) {
            crf_inflate::Decoder dec;
            dec.base = dec.in = d + b.cdata;
            dec.in_end = dec.in + b.clen;
            dec.out = &scratch;
            dec.op = 0;
            if (dec.run(tables) == crf_inflate::Decoder::RUN_FINAL && dec.op == b.isize &&
                (uint32_t)crc32(crc32(0L, Z_NULL, 0), scratch.p, b.isize) == b.crc) {
                memcpy(dst, scratch.p, b.isize);
                return true;
            }
        }
        if (!zs_ready) {
            memset(&zs, 0, sizeof zs);
            if (inflateInit2(&zs, -15) != Z_OK) return false;
            zs_ready = true;
        }
        zs.next_in = const_cast<Bytef *>(d + b.cdata);
        zs.avail_in = (uInt)b.clen;
        zs.next_out = dst;
        zs.avail_out = b.isize;
        const int rc = inflate(&zs, Z_FINISH);
        const bool ok = rc == Z_STREAM_END && zs.avail_out == 0 && (uint32_t)crc32(crc32(0L, Z_NULL, 0), dst, b.isize) == b.crc;
        inflateReset(&zs);
        return ok;
    }
};

// Blocks [first, last) on the reader's threads into dst (block i at dst + blocks[i].out - blocks[first].out); false if one
// is corrupt.
static bool inflate_blocks(const uint8_t *d, const std::vector<BgzfBlock> &blocks, size_t first, size_t last,
                           unsigned n_threads, uint8_t *dst, size_t GROUP = 128) {   // GROUP: blocks per work item
    std::atomic<bool> failed{false}, no_memory{false};
    const uint64_t out0 = first < last ? blocks[first].out : 0;
    run_parallel(n_threads, (last - first + GROUP - 1) / GROUP, [&](size_t g) {
      try {
        BgzfInflater inf(d);
        for (size_t i = first + g * GROUP; i < std::min(last, first + (g + 1) * GROUP) && !failed; ++i)
            if (!inf.run(blocks[i], dst + blocks[i].out - out0)) failed = true;
      } catch (const std::bad_alloc &) { no_memory = true; failed = true; }      // (nothing leaves a worker thread)
    });
    if (no_memory) throw std::bad_alloc();
    return !failed;
}

static bool is_space(uint8_t c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n' || c == '\v' || c == '\f'; }

// The record name: the first whitespace-delimited token [*a, returned end) of the header text [*a, h1).
static uint64_t name_token(const uint8_t *t, uint64_t *a, uint64_t h1) {
    while (*a < h1 && is_space(t[*a])) ++*a;
    uint64_t b = *a;
    while (b < h1 && !is_space(t[b])) ++b;
    return b;
}

// The text buffer of total bases: page-locked with pinned & 1 when a device is present, else plain pages.
static bool alloc_bases(crf_fasta *fa, uint64_t total, int pinned) {
    return fa->bases_buf.alloc(std::max<uint64_t>(total, 1), pinned & 1);
}

// src[0, n) into dst, page-locked, copied 64 MiB at a time on the reader's threads; false (dst untouched) when there is no
// page-locked memory to be had.  give_back: each piece's source pages go back to the system once copied (src is an anonymous
// mapping nothing reads again), so the bytes are held twice only a piece at a time.
static bool copy_page_locked(HostBuf &dst, const uint8_t *src, uint64_t n, unsigned n_threads, bool give_back) {
    if (!dst.pin(std::max<uint64_t>(n, 1))) return false;
    const uint64_t PIECE = 64u << 20;
    run_parallel(n_threads, (n + PIECE - 1) / PIECE, [&](size_t i) {
        const uint64_t a = i * PIECE, z = std::min(PIECE, n - a);
        memcpy(dst.p + a, src + a, z);
        if (give_back) madvise(const_cast<uint8_t *>(src) + a, z & ~(uint64_t)4095, MADV_DONTNEED);
    });
    return true;
}

// ---- FASTQ ----
// A record is a header line '@name ...', sequence lines up to a line starting with '+' (the rest of that line is ignored),
// then quality lines until they hold as many bytes as the sequence (which makes quality lines starting with '@' or '+'
// unambiguous).  A line is its bytes up to '\n' or the end of the text, without one trailing '\r'.  Whitespace between
// records is skipped.  Quality bytes are '!'..'~'.
//
// Threaded path: the text is cut into pieces; every piece but the first starts at its first line that begins with '@' and
// whose line after next begins with '+', and parses 4-line records (header, one sequence line not starting with '+', '+'
// line, quality line as long as the sequence) while they start inside the piece.  The result is taken only if every piece
// parsed that way and starts exactly where the previous one's last record ended (the last one ending at the end of the
// text); then it is what the general rules give.  Anything else goes to the serial parser of the general rules, the only
// place that reports errors.

struct Line { uint64_t a, b; };                         // content [a, b)

static inline uint64_t next_line(const uint8_t *t, uint64_t n, uint64_t p, Line &ln) {
    const uint8_t *e = (const uint8_t *)memchr(t + p, '\n', n - p);
    const uint64_t end = e ? (uint64_t)(e - t) : n;
    ln.a = p;
    ln.b = end > p && t[end - 1] == '\r' ? end - 1 : end;
    return e ? end + 1 : n;
}

static inline bool quality_bytes_ok(const uint8_t *q, uint64_t len) {
    uint8_t bad = 0;
    for (uint64_t i = 0; i < len; ++i) bad |= (uint8_t)(q[i] - '!') > ('~' - '!');
    return !bad;
}

// What a parse pass does with the records it finds: count them, or write them into the handle.
struct FastqCount {
    uint64_t records = 0, bases = 0, name_bytes = 0;
    void record(const uint8_t *t, uint64_t a, uint64_t h1) {
        const uint64_t b = name_token(t, &a, h1);
        ++records;
        name_bytes += b - a + 1;
    }
    void seq(const uint8_t *, const Line &ln) { bases += ln.b - ln.a; }
    void qual(const uint8_t *, const Line &) {}
};

struct FastqWrite {
    crf_fasta *fa;
    uint64_t rec, base, name, qbase;                    // cursors: record, base, name byte, quality byte
    void record(const uint8_t *t, uint64_t a, uint64_t h1) {
        const uint64_t e = name_token(t, &a, h1);
        fa->offsets[rec] = base;
        fa->name_off[rec++] = name;
        memcpy(fa->names.data() + name, t + a, e - a);
        name += e - a;
        fa->names[name++] = '\0';
    }
    void seq(const uint8_t *t, const Line &ln) {
        memcpy(fa->bases + base, t + ln.a, ln.b - ln.a);
        base += ln.b - ln.a;
    }
    void qual(const uint8_t *t, const Line &ln) {
        if (fa->quals) memcpy(fa->quals + qbase, t + ln.a, ln.b - ln.a);
        qbase += ln.b - ln.a;
    }
};

// 4-line records from p while they start before stop.  *end = where the last one ends.  false: a record without that shape.
template <class Sink>
static bool fastq_4line(const uint8_t *t, uint64_t n, uint64_t p, uint64_t stop, uint64_t *end, Sink &sink) {
    while (p < stop) {
        Line h, s, plus, q;
        if (t[p] != '@') return false;
        p = next_line(t, n, p, h);
        if (p >= n) return false;
        p = next_line(t, n, p, s);
        if (p >= n || (s.b > s.a && t[s.a] == '+')) return false;
        p = next_line(t, n, p, plus);
        if (p >= n || t[plus.a] != '+') return false;
        p = next_line(t, n, p, q);
        if (q.b - q.a != s.b - s.a || !quality_bytes_ok(t + q.a, q.b - q.a)) return false;
        sink.record(t, h.a + 1, h.b);
        sink.seq(t, s);
        sink.qual(t, q);
    }
    *end = p;
    return true;
}

// The general rules, from p to the end of the text.  Returns 0, or the 1-based number of the record at fault with *why set.
template <class Sink>
static uint64_t fastq_serial(const uint8_t *t, uint64_t n, uint64_t p, Sink &sink, const char **why) {
    for (uint64_t rec = 1;; ++rec) {
        while (p < n && is_space(t[p])) ++p;
        if (p == n) return 0;
        if (t[p] != '@') { *why = "text that is not whitespace before its '@' header"; return rec; }
        Line ln;
        p = next_line(t, n, p, ln);
        sink.record(t, ln.a + 1, ln.b);
        uint64_t len = 0;
        for (;;) {                                      // sequence lines up to the '+' line
            if (p >= n) { *why = "the file ends inside the record"; return rec; }
            p = next_line(t, n, p, ln);
            if (ln.b > ln.a && t[ln.a] == '+') break;
            sink.seq(t, ln);
            len += ln.b - ln.a;
        }
        for (uint64_t got = 0; got < len;) {            // quality lines until they hold len bytes
            if (p >= n) { *why = "the file ends inside the record"; return rec; }
            p = next_line(t, n, p, ln);
            if (got + (ln.b - ln.a) > len) { *why = "its quality is longer than its sequence"; return rec; }
            if (!quality_bytes_ok(t + ln.a, ln.b - ln.a)) { *why = "a quality byte outside '!'..'~'"; return rec; }
            sink.qual(t, ln);
            got += ln.b - ln.a;
        }
    }
}

// The FASTQ text t[lead, n) (t[lead] == '@') into fa.  piece: bytes of text per piece of the threaded path.
// *serial: whether the serial parser made the result.
static int parse_fastq(const char *path, const uint8_t *t, uint64_t n, uint64_t lead, unsigned n_threads, uint64_t piece,
                       int pinned, crf_fasta *fa, bool *serial) {
    fa->format = FORMAT_FASTQ;
    const uint64_t n_pieces = (n - lead + piece - 1) / piece;
    struct Part { uint64_t begin, end; FastqCount count; bool ok; };
    std::vector<Part> parts(n_pieces);
    run_parallel(n_threads, n_pieces, [&](size_t i) {
        Part &pt = parts[i];
        const uint64_t lo = lead + i * piece, hi = std::min(n, lo + piece);
        pt.ok = false;
        pt.begin = pt.end = hi;                         // (no record starts in the piece)
        uint64_t p = lo;
        if (i > 0) {                                    // the first line start at or after lo that looks like a header
            if (t[p - 1] != '\n') {
                const uint8_t *e = (const uint8_t *)memchr(t + p, '\n', n - p);
                p = e ? (uint64_t)(e - t) + 1 : n;
            }
            for (; p < hi; ) {
                Line l1, l2;
                const uint64_t p1 = next_line(t, n, p, l1);
                if (t[p] == '@' && p1 < n) {
                    const uint64_t p2 = next_line(t, n, p1, l2);
                    if (p2 < n && t[p2] == '+') break;
                }
                p = p1;
            }
            if (p >= hi) { pt.ok = true; return; }
        }
        pt.begin = p;
        pt.ok = fastq_4line(t, n, p, hi, &pt.end, pt.count);
    });
    uint64_t at = lead;
    bool chained = true;
    for (const Part &pt : parts) {
        if (!pt.ok) { chained = false; break; }
        if (pt.count.records == 0) continue;            // no record starts in it (text skipped here breaks the chain later)
        if (pt.begin != at) { chained = false; break; }
        at = pt.end;
    }
    chained = chained && at == n;
    *serial = !chained;

    FastqCount total;
    if (chained) {
        for (const Part &pt : parts) {
            total.records += pt.count.records;
            total.bases += pt.count.bases;
            total.name_bytes += pt.count.name_bytes;
        }
    } else {
        const char *why = nullptr;
        if (const uint64_t bad = fastq_serial(t, n, lead, total, &why)) {
            set_err("crf_fasta_open: %s: FASTQ record %llu: %s", path, (unsigned long long)bad, why);
            return CRF_ERR_ARG;
        }
    }
    fa->offsets.assign(total.records + 1, 0);
    fa->name_off.assign(total.records, 0);
    fa->names.assign(total.name_bytes, 0);
    fa->offsets[total.records] = fa->total = total.bases;
    if (!alloc_bases(fa, total.bases, pinned) || ((pinned & 4) && !fa->quals_buf.alloc(std::max<uint64_t>(total.bases, 1), false))) {
        set_err("crf_fasta_open: out of host memory (%llu bases)", (unsigned long long)total.bases);
        return CRF_ERR_NOMEM;
    }
    if (chained) {
        std::vector<FastqWrite> sinks(n_pieces, FastqWrite{fa, 0, 0, 0, 0});
        FastqWrite cur{fa, 0, 0, 0, 0};
        for (uint64_t i = 0; i < n_pieces; ++i) {
            sinks[i] = cur;
            sinks[i].qbase = cur.base;
            cur.rec += parts[i].count.records;
            cur.base += parts[i].count.bases;
            cur.name += parts[i].count.name_bytes;
        }
        run_parallel(n_threads, n_pieces, [&](size_t i) {
            const Part &pt = parts[i];
            uint64_t end;
            if (pt.count.records) (void)fastq_4line(t, n, pt.begin, std::min(n, lead + (i + 1) * piece), &end, sinks[i]);
        });
    } else {
        FastqWrite sink{fa, 0, 0, 0, 0};
        const char *why = nullptr;
        fastq_serial(t, n, lead, sink, &why);
    }
    return CRF_OK;
}

// ---- .2bit (UCSC) ----
// Header: signature 0x1A412743, version (0: 32-bit index offsets, 1: 64-bit ones, faToTwoBit -long), record count,
// reserved; a file with the signature in the other byte order has every integer swapped.  Index: per record a name size
// byte, the name and the offset of the record.  A record: dnaSize, N block count, starts, sizes, mask block count, starts,
// sizes, a reserved word, then (dnaSize + 3) / 4 bytes of packed bases, T=0 C=1 A=2 G=3, the first base in the top two
// bits of its byte.  The bases stay packed in the file's bytes; the text is decoded only when a caller asks for it.
static const uint32_t TWOBIT_SIG = 0x1A412743u;

static bool is_twobit(const uint8_t *t, uint64_t n) {
    if (n < 4) return false;
    uint32_t v;
    memcpy(&v, t, 4);
    return v == TWOBIT_SIG || __builtin_bswap32(v) == TWOBIT_SIG;
}

// One record's blocks [start, start + size) as sorted, merged runs shifted by base (empty blocks dropped).
static void merge_blocks(std::vector<std::pair<uint64_t, uint64_t>> &blk, uint64_t base, std::vector<uint64_t> &out) {
    std::sort(blk.begin(), blk.end());
    bool open = false;
    uint64_t a = 0, b = 0;
    for (const auto &x : blk) {
        if (x.first == x.second) continue;
        if (open && x.first <= b) { b = std::max(b, x.second); continue; }
        if (open) { out.push_back(base + a); out.push_back(base + b); }
        a = x.first; b = x.second; open = true;
    }
    if (open) { out.push_back(base + a); out.push_back(base + b); }
}

// Index, record headers and blocks of the .2bit file t[0, n) into fa, every count, offset and block checked against the
// file size and dnaSize.  The bases are not touched.
static int parse_twobit(const char *path, const uint8_t *t, uint64_t n, crf_fasta *fa) {
    fa->format = FORMAT_2BIT;
    uint32_t sig;
    memcpy(&sig, t, 4);
    const bool swap = sig != TWOBIT_SIG;
    auto u32 = [&](uint64_t p) { uint32_t v; memcpy(&v, t + p, 4); return swap ? __builtin_bswap32(v) : v; };
    auto u64 = [&](uint64_t p) { uint64_t v; memcpy(&v, t + p, 8); return swap ? __builtin_bswap64(v) : v; };
    auto fail = [&](uint64_t rec, const char *why) {
        set_err("crf_fasta_open: %s: .2bit record %llu: %s", path, (unsigned long long)rec, why);
        return CRF_ERR_ARG;
    };
    if (n < 16) { set_err("crf_fasta_open: %s: the .2bit header is truncated", path); return CRF_ERR_ARG; }
    const uint32_t version = u32(4), count = u32(8);
    if (version > 1) { set_err("crf_fasta_open: %s: .2bit version %u (0 or 1 expected)", path, version); return CRF_ERR_ARG; }
    const uint64_t off_bytes = version ? 8 : 4;
    std::vector<uint64_t> rec_off;
    rec_off.reserve(std::min<uint64_t>(count, n / 5));
    uint64_t p = 16;
    for (uint64_t r = 0; r < count; ++r) {
        if (p >= n || n - p - 1 < t[p] + off_bytes) return fail(r + 1, "the index is truncated");
        const uint32_t ns = t[p++];
        fa->name_off.push_back(fa->names.size());
        fa->names.insert(fa->names.end(), t + p, t + p + ns);
        fa->names.push_back('\0');
        p += ns;
        rec_off.push_back(version ? u64(p) : u32(p));
        p += off_bytes;
    }
    fa->offsets.assign((size_t)count + 1, 0);
    fa->rec_byte.assign(count, 0);
    std::vector<std::pair<uint64_t, uint64_t>> blk;
    uint64_t total = 0;
    for (uint64_t r = 0; r < count; ++r) {
        const uint64_t off = rec_off[r];
        if (off >= n) return fail(r + 1, "its offset is past the end of the file");
        if (n - off < 8) return fail(r + 1, "its header runs past the end of the file");
        const uint64_t dna_size = u32(off), nb = u32(off + 4);
        uint64_t q = off + 8;
        for (int kind = 0; kind < 2; ++kind) {                    // N blocks, then mask blocks
            uint64_t cnt = nb;
            if (kind) {
                if (n - q < 4) return fail(r + 1, "its header runs past the end of the file");
                cnt = u32(q);
                q += 4;
            }
            if ((n - q) / 8 < cnt) return fail(r + 1, kind ? "its mask blocks run past the end of the file"
                                                           : "its N blocks run past the end of the file");
            blk.clear();
            for (uint64_t i = 0; i < cnt; ++i) {
                const uint64_t s = u32(q + 4 * i), z = u32(q + 4 * (cnt + i));
                if (s + z > dna_size) return fail(r + 1, kind ? "a mask block ends past its dnaSize" : "an N block ends past its dnaSize");
                blk.push_back({s, s + z});
            }
            merge_blocks(blk, total, kind ? fa->mask_runs : fa->n_runs);
            q += 8 * cnt;
        }
        if (n - q < 4) return fail(r + 1, "its header runs past the end of the file");
        q += 4;                                                   // reserved
        if (n - q < (dna_size + 3) / 4) return fail(r + 1, "the file is shorter than its DNA");
        fa->rec_byte[r] = q;
        fa->offsets[r] = total;
        total += dna_size;
    }
    fa->offsets[count] = fa->total = total;
    // the records' bases may not share bytes: a load masks the N blocks by byte position
    std::vector<uint32_t> order;
    for (uint32_t r = 0; r < count; ++r)
        if (fa->offsets[r + 1] > fa->offsets[r]) order.push_back(r);
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return fa->rec_byte[a] < fa->rec_byte[b]; });
    for (size_t i = 1; i < order.size(); ++i) {
        const uint32_t a = order[i - 1], b = order[i];
        if (fa->rec_byte[a] + (fa->offsets[a + 1] - fa->offsets[a] + 3) / 4 > fa->rec_byte[b]) {
            set_err("crf_fasta_open: %s: .2bit record %u: its bases overlap those of record %u", path, std::max(a, b) + 1,
                    std::min(a, b) + 1);
            return CRF_ERR_ARG;
        }
    }
    return CRF_OK;
}

// ---- BAM (unaligned reads) ----
// A BGZF stream that starts with "BAM\1": l_text, the header text, n_ref and the reference list, then the records.  A
// record is block_size and block_size bytes: refID, pos, l_read_name (u8), mapq, bin, n_cigar_op (u16), flag (u16), l_seq,
// next_refID, next_pos, tlen (32 bytes in all), read_name (NUL-terminated), cigar (4 n_cigar_op bytes), seq ((l_seq + 1) / 2
// bytes, 4-bit codes =ACMGRSVTWYHKDBN, high nibble first), qual (l_seq bytes, 0xFF... when absent), tags.
// What is kept is what `samtools fastq -n` writes: records with (flag & 0x900) == 0 in file order, the name up to its NUL,
// the bases reverse-complemented when flag & 0x10 (the complement of a code is its 4-bit bit-reversal), qualities + 33 (or
// '"' when absent), reversed with the bases.  The stream is inflated a window of blocks at a time; the bases stay codes.
static const uint64_t BAM_WINDOW = 32u << 20;             // inflated bytes per window (CRF_BAM_WINDOW overrides it)

static bool is_bam_magic(const uint8_t *t, uint64_t n) { return n >= 4 && memcmp(t, "BAM\1", 4) == 0; }

// A growable anonymous mapping: it grows with mremap (the pages are not copied) and nothing is zero-filled by hand.
struct GrowBuf {
    uint8_t *p = nullptr;
    size_t cap = 0;
    ~GrowBuf() { if (p) munmap(p, cap); }
    void reserve(size_t need) {
        if (need <= cap) return;
        size_t nc = std::max<size_t>(std::max<size_t>(need, cap + cap / 2), (size_t)1 << 21);
        nc = (nc + 4095) & ~(size_t)4095;
        void *q = p ? mremap(p, cap, nc, MREMAP_MAYMOVE) : mmap(nullptr, nc, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (q == MAP_FAILED) throw std::bad_alloc();
        p = (uint8_t *)q;
        cap = nc;
    }
    HostBuf release() {                                    // the mapping goes to the caller
        HostBuf b;
        b.adopt(p, cap);
        p = nullptr;
        return b;
    }
};

// The inflated stream, a window of blocks at a time: bytes [pos, end) of buf are inflated and not yet consumed.
struct BamStream {
    const uint8_t *file;
    const std::vector<BgzfBlock> &blocks;
    unsigned n_threads;
    size_t next = 0;                                      // first block not inflated
    uint64_t left;                                        // inflated bytes of the blocks from next on
    uint64_t window;
    GrowBuf buf;
    uint64_t pos = 0, end = 0;
    uint64_t avail() const { return end - pos; }
    // At least one more window, more while fewer than `need` bytes are available and blocks remain.  false: a corrupt block.
    bool fill(uint64_t need) {
        if (pos) { memmove(buf.p, buf.p + pos, end - pos); end -= pos; pos = 0; }
        do {
            if (next == blocks.size()) return true;
            size_t last = next;
            uint64_t bytes = 0;
            while (last < blocks.size() && (last == next || bytes + blocks[last].isize <= window)) bytes += blocks[last++].isize;
            buf.reserve(end + bytes);
            if (!inflate_blocks(file, blocks, next, last, n_threads, buf.p + end, 16)) return false;
            end += bytes;
            left -= bytes;
            next = last;
        } while (end - pos < need);
        return true;
    }
};

static inline uint32_t rd32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static inline uint16_t rd16(const uint8_t *p) { uint16_t v; memcpy(&v, p, 2); return v; }

struct BamRec {                                           // a kept record of the current window
    uint64_t at;                                          // its block_size field, in the stream buffer
    uint64_t base, name;                                  // where its bases and name go
};

// Record number `rec` (1-based) at q (its block_size field) of a buffer holding n >= 4 bytes from q on, complete when
// n >= 4 + block_size.  Returns nullptr if it is well-formed (*kept, *l_seq, *name_len set), else why not.
static const char *bam_check(const uint8_t *q, uint32_t bs, bool *kept, uint64_t *l_seq, uint64_t *name_len) {
    const uint8_t *f = q + 4;
    const uint32_t lrn = f[8], ncig = rd16(f + 12), flag = rd16(f + 14);
    const int32_t ls = (int32_t)rd32(f + 16);
    if (lrn == 0) return "l_read_name is 0";
    if (ls < 0) return "l_seq is negative";
    if (32ull + lrn + 4ull * ncig + ((uint64_t)ls + 1) / 2 + (uint64_t)ls > bs) return "its fields run past its block_size";
    if (f[32 + lrn - 1] != 0) return "its read_name does not end with a NUL";
    *kept = (flag & 0x900) == 0;
    *l_seq = (uint64_t)ls;
    *name_len = strnlen((const char *)f + 32, lrn);
    return nullptr;
}

// A kept record's bases (codes from byte `o` of nib, reverse-complemented when flag & 0x10, a padding nibble 0), its name,
// its qualities (quals may be null) and its exotic codes (appended to ex, positions from `base`).
static void bam_copy(const uint8_t *q, uint8_t *nib, uint64_t o, uint8_t *quals, uint64_t base, char *name_out,
                     std::vector<uint64_t> &ex) {
    static const struct Lut {
        uint8_t comp[16], exotic[16];
        Lut() {
            for (int c = 0; c < 16; ++c) {
                comp[c] = (uint8_t)(((c & 1) << 3) | ((c & 2) << 1) | ((c & 4) >> 1) | ((c & 8) >> 3));
                exotic[c] = !(c == 1 || c == 2 || c == 4 || c == 8 || c == 15);
            }
        }
    } lut;
    const uint8_t *f = q + 4;
    const uint32_t lrn = f[8], ncig = rd16(f + 12), flag = rd16(f + 14);
    const uint64_t n = rd32(f + 16);
    const uint8_t *seq = f + 32 + lrn + 4 * ncig, *qual = seq + (n + 1) / 2;
    const size_t nl = strnlen((const char *)f + 32, lrn);
    memcpy(name_out, f + 32, nl);
    name_out[nl] = '\0';
    uint8_t *d = nib + o;
    const bool rev = flag & 0x10;
    if (!rev) {
        memcpy(d, seq, n / 2);
        if (n & 1) d[n / 2] = seq[n / 2] & 0xF0;
    } else if (n) {                                        // base i = complement of base n - 1 - i, a byte at a time
        const uint64_t last = (n - 1) / 2;
        if (n & 1) {                                       // byte j: high nibble of byte last - j, low of the one before
            for (uint64_t j = 0; j <= last; ++j) {
                const uint64_t k = last - j;
                d[j] = (uint8_t)((lut.comp[seq[k] >> 4] << 4) | (k ? lut.comp[seq[k - 1] & 15] : 0));
            }
        } else {                                           // byte j: byte last - j with its nibbles swapped
            for (uint64_t j = 0; j <= last; ++j) {
                const uint8_t b = seq[last - j];
                d[j] = (uint8_t)((lut.comp[b & 15] << 4) | lut.comp[b >> 4]);
            }
        }
    }
    for (uint64_t i = 0; i < n; i += 2) {                  // exotic codes: rare, found a byte at a time
        const uint8_t b = d[i >> 1];
        if (!lut.exotic[b >> 4] && (i + 1 == n || !lut.exotic[b & 15])) continue;
        for (uint64_t k = i; k < std::min(n, i + 2); ++k) {
            const uint8_t c = k & 1 ? b & 15 : b >> 4;
            if (lut.exotic[c]) ex.push_back(((base + k) << 8) | (uint8_t)PackedCodes<4>::LETTERS[c]);
        }
    }
    if (!quals) return;
    uint8_t *qo = quals + base;
    if (n && qual[0] == 0xFF) memset(qo, '"', n);
    else if (!rev) for (uint64_t i = 0; i < n; ++i) qo[i] = (uint8_t)(qual[i] + 33);
    else for (uint64_t i = 0; i < n; ++i) qo[i] = (uint8_t)(qual[n - 1 - i] + 33);
}

// The BAM stream of the BGZF blocks into fa.  Every count and length is checked against the record and the stream.
static int parse_bam(const char *path, const uint8_t *file, const std::vector<BgzfBlock> &blocks, uint64_t total,
                     unsigned n_threads, int pinned, crf_fasta *fa) {
    fa->format = FORMAT_BAM;
    const char *w = getenv("CRF_BAM_WINDOW");
    BamStream s{file, blocks, n_threads, 0, total, w ? std::max<uint64_t>(strtoull(w, nullptr, 10), 1) : BAM_WINDOW};
    auto corrupt = [&]() { set_err("crf_fasta_open: %s has a corrupt BGZF block", path); return CRF_ERR_ARG; };
    auto header_fail = [&](const char *why) { set_err("crf_fasta_open: %s: BAM header: %s", path, why); return CRF_ERR_ARG; };
    auto rec_fail = [&](uint64_t rec, const char *why) {
        set_err("crf_fasta_open: %s: BAM record %llu: %s", path, (unsigned long long)rec, why);
        return CRF_ERR_ARG;
    };
    // header: the first h bytes of the stream, pulled in as needed (false: shorter than that)
    int bad_block = 0;
    auto have = [&](uint64_t h) {
        if (h <= s.avail()) return true;
        if (h > s.avail() + s.left) return false;
        if (!s.fill(h)) { bad_block = 1; return false; }
        return true;
    };
    if (!have(12)) return bad_block ? corrupt() : header_fail("it is truncated");
    const int32_t l_text = (int32_t)rd32(s.buf.p + s.pos + 4);
    if (l_text < 0) return header_fail("l_text is negative");
    uint64_t h = 8 + (uint64_t)l_text;
    if (!have(h + 4)) return bad_block ? corrupt() : header_fail("the text runs past the end of the data");
    const int32_t n_ref = (int32_t)rd32(s.buf.p + s.pos + h);
    if (n_ref < 0) return header_fail("n_ref is negative");
    h += 4;
    for (int32_t i = 0; i < n_ref; ++i) {
        if (!have(h + 4)) return bad_block ? corrupt() : header_fail("the reference list runs past the end of the data");
        const int32_t l_name = (int32_t)rd32(s.buf.p + s.pos + h);
        if (l_name < 0) return header_fail("a reference's l_name is negative");
        h += 4 + (uint64_t)l_name + 4;
        if (!have(h)) return bad_block ? corrupt() : header_fail("the reference list runs past the end of the data");
    }
    s.pos += h;

    const bool want_quals = pinned & 4;
    GrowBuf nib, quals;
    uint64_t nib_at = 0, base_at = 0, rec = 0;              // output cursors; records seen
    std::vector<BamRec> batch;
    std::vector<std::vector<uint64_t>> ex_parts;
    for (;;) {
        batch.clear();
        uint64_t p = s.pos, name_at = fa->names.size();
        while (s.end - p >= 4) {                            // the complete records of the buffer
            const uint32_t bs = rd32(s.buf.p + p);
            if (bs < 32) return rec_fail(rec + 1, "block_size is less than 32");
            if (s.end - p - 4 < bs) {
                if (bs > s.end - p - 4 + s.left) return rec_fail(rec + 1, "it runs past the end of the data");
                break;
            }
            bool kept;
            uint64_t l_seq, nl;
            if (const char *why = bam_check(s.buf.p + p, bs, &kept, &l_seq, &nl)) return rec_fail(rec + 1, why);
            ++rec;
            if (kept) {
                batch.push_back({p, base_at, name_at});
                fa->offsets.push_back(base_at);
                fa->rec_byte.push_back(nib_at);
                fa->name_off.push_back(name_at);
                base_at += l_seq;
                nib_at += (l_seq + 1) / 2;
                name_at += nl + 1;
            }
            p += 4 + (uint64_t)bs;
        }
        if (!batch.empty()) {                                // copy the window's kept records on the reader's threads
            nib.reserve(nib_at + 16);
            if (want_quals) quals.reserve(base_at + 16);
            fa->names.resize(name_at);
            // (work items of a few records for long reads, thousands for short ones)
            const size_t first = fa->rec_byte.size() - batch.size(), GROUP = (batch.size() + 8 * n_threads - 1) / (8 * n_threads);
            ex_parts.assign((batch.size() + GROUP - 1) / GROUP, {});
            run_parallel(n_threads, ex_parts.size(), [&](size_t g) {
                for (size_t i = g * GROUP; i < std::min(batch.size(), (g + 1) * GROUP); ++i)
                    bam_copy(s.buf.p + batch[i].at, nib.p, fa->rec_byte[first + i], want_quals ? quals.p : nullptr,
                             batch[i].base, fa->names.data() + batch[i].name, ex_parts[g]);
            });
            for (const auto &v : ex_parts) fa->nib_exotic.insert(fa->nib_exotic.end(), v.begin(), v.end());
        }
        s.pos = p;
        if (s.next == blocks.size()) {
            if (s.avail()) return rec_fail(rec + 1, "the data ends inside the record");
            break;
        }
        if (!s.fill(s.avail() >= 4 ? 4 + (uint64_t)rd32(s.buf.p + s.pos) : 4)) return corrupt();
    }
    fa->offsets.push_back(base_at);
    fa->total = base_at;
    nib.reserve(1);
    if (!((pinned & 3) && copy_page_locked(fa->codes, nib.p, nib_at, n_threads, true))) fa->codes = nib.release();
    if (want_quals) {
        quals.reserve(1);
        fa->quals_buf = quals.release();
    }
    return CRF_OK;
}

// Record r's letters from positions [lo, hi) of the concatenated text.
template <int BITS>
static void decode_records(crf_fasta *fa, uint64_t lo, uint64_t hi) {
    const std::vector<uint64_t> &off = fa->offsets;
    uint64_t r = (uint64_t)(std::upper_bound(off.begin(), off.end(), lo) - off.begin()) - 1;
    for (uint64_t pos = lo; pos < hi; ++r) {
        if (off[r + 1] <= pos) continue;
        const uint64_t i1 = std::min(hi, off[r + 1]) - off[r];
        code_letters<BITS>(fa->codes.p + fa->rec_byte[r], pos - off[r], i1, fa->bases + off[r]);
        pos = off[r] + i1;
    }
}

// The text of a .2bit or BAM handle, decoded on first use (nothing to do for the others), on the reader's threads in pieces
// of concatenated positions.  A BAM file's is what samtools fastq writes as bases; a .2bit file's what twoBitToFa writes:
// T/C/A/G, N blocks as 'N', mask blocks lower-cased ('n' inside both).
static int decode_text(crf_fasta *fa) {
    if (fa->format != FORMAT_2BIT && fa->format != FORMAT_BAM) return CRF_OK;
    std::lock_guard<std::mutex> lock(fa->decode_mu);
    if (fa->bases) return CRF_OK;
    try {
        if (!alloc_bases(fa, fa->total, fa->pinned)) {
            set_err("crf_fasta_data: out of host memory (%llu bases)", (unsigned long long)fa->total);
            return CRF_ERR_NOMEM;
        }
        const uint64_t PIECE = 4u << 20, total = fa->total;
        const bool twobit = fa->format == FORMAT_2BIT;
        uint8_t *out = fa->bases;
        run_parallel(fa->n_threads, (total + PIECE - 1) / PIECE, [&](size_t i) {
            const uint64_t lo = i * PIECE, hi = std::min(total, lo + PIECE);
            if (!twobit) { decode_records<4>(fa, lo, hi); return; }
            decode_records<2>(fa, lo, hi);
            for (int kind = 0; kind < 2; ++kind) {                // mask blocks lower-case, then N blocks keep the case
                const std::vector<uint64_t> &runs = kind ? fa->n_runs : fa->mask_runs;
                uint64_t a = 0, b = runs.size() / 2;              // first run that ends after lo
                while (a < b) { const uint64_t m = (a + b) / 2; if (runs[2 * m + 1] <= lo) a = m + 1; else b = m; }
                for (; a < runs.size() / 2 && runs[2 * a] < hi; ++a)
                    for (uint64_t q = std::max(lo, runs[2 * a]), e = std::min(hi, runs[2 * a + 1]); q < e; ++q)
                        out[q] = kind ? (uint8_t)((out[q] & 0x20) | 'N') : (uint8_t)(out[q] | 0x20);
            }
        });
    } catch (const std::bad_alloc &) {
        set_err("crf_fasta_data: out of host memory");
        return CRF_ERR_NOMEM;
    }
    return CRF_OK;
}

// CRF_FASTA_TRACE=1: the stage times of crf_fasta_open on stderr.
struct OpenTrace {
    bool on = getenv("CRF_FASTA_TRACE") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void lap(const char *what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[crf_fasta] %-10s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

// ---- FASTA ----
// A record is a '>' at the start of a line, its header line (the name: its first whitespace-delimited token), then the
// body lines up to the next record, joined without their line ends.
static int parse_fasta(const uint8_t *t, uint64_t n, unsigned n_threads, int pinned, crf_fasta *fa, OpenTrace &trace) {
    const uint64_t PIECE = 8u << 20;
    // headers: a '>' at the start of a line
    std::vector<std::vector<uint64_t>> hdr_in((n + PIECE - 1) / PIECE);
    run_parallel(n_threads, hdr_in.size(), [&](size_t i) {
        const uint64_t hi = std::min<uint64_t>(n, (i + 1) * PIECE);
        for (uint64_t p = i * PIECE; p < hi;) {
            const uint8_t *q = (const uint8_t *)memchr(t + p, '>', hi - p);
            if (!q) break;
            const uint64_t at = q - t;
            if (at == 0 || t[at - 1] == '\n' || t[at - 1] == '\r') hdr_in[i].push_back(at);
            p = at + 1;
        }
    });
    std::vector<uint64_t> hdr;
    for (const auto &v : hdr_in) hdr.insert(hdr.end(), v.begin(), v.end());
    const uint64_t n_rec = hdr.size();
    std::vector<uint64_t> body_lo(n_rec), body_hi(n_rec);
    for (uint64_t r = 0; r < n_rec; ++r) {
        const uint64_t stop = r + 1 < n_rec ? hdr[r + 1] : n;
        const uint8_t *eol = (const uint8_t *)memchr(t + hdr[r], '\n', stop - hdr[r]);
        uint64_t h1 = eol ? (uint64_t)(eol - t) : stop;            // header text = (hdr, h1)
        body_lo[r] = eol ? h1 + 1 : stop;
        body_hi[r] = stop;
        uint64_t a = hdr[r] + 1;
        const uint64_t b = name_token(t, &a, h1);
        fa->name_off.push_back(fa->names.size());
        fa->names.insert(fa->names.end(), t + a, t + b);
        fa->names.push_back('\0');
    }

    trace.lap("headers");
    // bodies in pieces of <= 8 MiB of text: count line ends, prefix-sum, compact
    std::vector<Piece> pieces;
    std::vector<uint64_t> first_piece(n_rec + 1);
    for (uint64_t r = 0; r < n_rec; ++r) {
        first_piece[r] = pieces.size();
        for (uint64_t p = body_lo[r]; p < body_hi[r]; p += PIECE) pieces.push_back({p, std::min(body_hi[r], p + PIECE), 0, 0});
    }
    first_piece[n_rec] = pieces.size();
    run_parallel(n_threads, pieces.size(), [&](size_t i) {
        Piece &pc = pieces[i];
        uint64_t c = 0;
        for (uint64_t p = pc.begin; p < pc.end; ++p) c += (t[p] == '\n') | (t[p] == '\r');
        pc.n_eol = c;
    });
    trace.lap("count");
    fa->offsets.assign(n_rec + 1, 0);
    uint64_t total = 0;
    for (uint64_t r = 0; r < n_rec; ++r) {
        fa->offsets[r] = total;
        for (uint64_t i = first_piece[r]; i < first_piece[r + 1]; ++i) {
            pieces[i].out = total;
            total += pieces[i].end - pieces[i].begin - pieces[i].n_eol;
        }
    }
    fa->offsets[n_rec] = total;
    fa->total = total;

    if (!alloc_bases(fa, total, pinned)) { set_err("crf_fasta_open: out of host memory (%llu bases)", (unsigned long long)total); return CRF_ERR_NOMEM; }

    trace.lap("alloc");
    uint8_t *dst = fa->bases;
    run_parallel(n_threads, pieces.size(), [&](size_t i) {
        const Piece &pc = pieces[i];
        uint8_t *o = dst + pc.out;
        uint64_t p = pc.begin;
        const uint64_t K1 = 0x0101010101010101ull, K80 = 0x8080808080808080ull;
        while (p + 8 <= pc.end) {                       // 8 bytes at a time; a word holding a line end goes byte by byte
            uint64_t w;
            memcpy(&w, t + p, 8);
            const uint64_t a = w ^ (K1 * '\n'), b = w ^ (K1 * '\r');
            if ((((a - K1) & ~a) | ((b - K1) & ~b)) & K80) {
                for (int j = 0; j < 8; ++j) {
                    const uint8_t c = t[p + j];
                    if (c != '\n' && c != '\r') *o++ = c;      // never touch a byte beyond this piece's output
                }
            } else {
                memcpy(o, &w, 8);
                o += 8;
            }
            p += 8;
        }
        for (; p < pc.end; ++p) {
            const uint8_t c = t[p];
            if (c != '\n' && c != '\r') *o++ = c;
        }
    });
    trace.lap("compact");
    return CRF_OK;
}

// Whether a BGZF file is BAM: its first inflated bytes are "BAM\1" (read from as many blocks as they span).
static bool bgzf_is_bam(const uint8_t *file, const std::vector<BgzfBlock> &blocks) {
    std::vector<uint8_t> head;
    BgzfInflater inf(file);
    bool head_ok = true;
    for (size_t b = 0; b < blocks.size() && head.size() < 4 && head_ok; ++b) {
        const size_t at = head.size();
        head.resize(at + blocks[b].isize);
        head_ok = inf.run(blocks[b], head.data() + at);
    }
    return head_ok && is_bam_magic(head.data(), head.size());
}

}  // namespace fasta_detail

static int fasta_open_impl(const char *path, uint32_t n_threads, int pinned, crf_fasta **out);
extern "C" int crf_fasta_close(crf_fasta *fa);

extern "C" int crf_fasta_open(const char *path, uint32_t n_threads, int pinned, crf_fasta **out) {
    if (!path || !out) { set_err("crf_fasta_open: null argument"); return CRF_ERR_ARG; }
    *out = nullptr;
    try {                                               // no exception crosses the C boundary
        return fasta_open_impl(path, n_threads, pinned, out);
    } catch (const std::bad_alloc &) {
        set_err("crf_fasta_open: out of host memory reading %s", path);
        return CRF_ERR_NOMEM;
    } catch (const std::exception &ex) {
        set_err("crf_fasta_open: %s", ex.what());
        return CRF_ERR_ARG;
    }
}

static int fasta_open_impl(const char *path, uint32_t n_threads, int pinned, crf_fasta **out) {
    using namespace fasta_detail;
    OpenTrace trace;
    FileBytes file;
    std::vector<uint8_t> plain;
    crf_inflate::OutBuf inflated;
    if (!open_bytes(path, file)) { set_err("crf_fasta_open: cannot read %s", path); return CRF_ERR_ARG; }
    const uint8_t *t = file.data;
    uint64_t n = file.size;
    if (n_threads == 0) n_threads = std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    std::unique_ptr<crf_fasta, int (*)(crf_fasta *)> fa(new crf_fasta, crf_fasta_close);   // unless handed to the caller
    fa->n_threads = n_threads;
    fa->pinned = pinned;
    const bool gz = n >= 2 && t[0] == 0x1f && t[1] == 0x8b;
    std::vector<BgzfBlock> blocks;
    uint64_t total = 0;
    const bool bgzf = gz && bgzf_index(file, blocks, &total);
    int rc;
    if (is_twobit(t, n)) {                              // (the raw file: a .2bit file is never compressed)
        rc = parse_twobit(path, t, n, fa.get());
        if (rc != CRF_OK) return rc;
        trace.lap("2bit-index");
        if ((pinned & 3) && copy_page_locked(fa->codes, t, n, n_threads, false)) {   // the bytes that get uploaded, page-locked
            trace.lap("2bit-pin");
        } else if (file.map) {                          // the mapping goes to the handle
            fa->codes.adopt(file.map, n);
            file.map = nullptr;
        } else {
            if (!fa->codes.alloc(std::max<uint64_t>(n, 1), false)) throw std::bad_alloc();
            memcpy(fa->codes.p, t, n);
        }
    } else if (bgzf && bgzf_is_bam(t, blocks)) {        // inflated a window at a time by parse_bam
        rc = parse_bam(path, t, blocks, total, n_threads, pinned, fa.get());
        if (rc != CRF_OK) return rc;
        trace.lap("bam");
    } else {
        if (gz) {
            if (bgzf) {
                if (!inflated.reserve(total + 64)) throw std::bad_alloc();
                inflated.size = total;
                if (!inflate_blocks(t, blocks, 0, blocks.size(), n_threads, inflated.p)) {
                    set_err("crf_fasta_open: %s has a corrupt BGZF block", path);
                    return CRF_ERR_ARG;
                }
            }
            // a plain gzip stream: the reader's own decoder (crf_inflate.h); whatever it does not take goes to zlib, which decides
            const bool own = !bgzf && getenv("CRF_GUNZIP_ZLIB") == nullptr && crf_inflate::gunzip(file.data, file.size, inflated, n_threads);
            if (!bgzf && !own && !inflate_all(file, plain)) { set_err("crf_fasta_open: %s is not a valid gzip stream", path); return CRF_ERR_ARG; }
            t = bgzf || own ? inflated.p : plain.data();
            n = bgzf || own ? inflated.size : plain.size();
            if (is_bam_magic(t, n)) {
                set_err("crf_fasta_open: %s is a BAM file compressed as plain gzip, not BGZF: BAM input must be BGZF "
                        "(as samtools writes it)", path);
                return CRF_ERR_ARG;
            }
            trace.lap(bgzf ? "bgzf" : own ? "gunzip" : "gzip/zlib");
        }
        trace.lap("read");
        uint64_t lead = 0;                              // a FASTQ file: '@' is its first byte that is not whitespace
        while (lead < n && is_space(t[lead])) ++lead;
        if (lead < n && t[lead] == '@') {
            bool serial = false;
            rc = parse_fastq(path, t, n, lead, n_threads, 8u << 20, pinned, fa.get(), &serial);
            if (rc != CRF_OK) return rc;
            trace.lap(serial ? "fastq-serial" : "fastq");
        } else {
            rc = parse_fasta(t, n, n_threads, pinned, fa.get(), trace);
            if (rc != CRF_OK) return rc;
        }
    }
    *out = fa.release();
    return CRF_OK;
}

// gzip -> bytes with the reader's decoder (use_zlib == 0: falls back to zlib like the reader does; 2: no fall-back,
// CRF_ERR_UNSUPPORTED instead) or with zlib only (1).
// CRF_ERR_CAPACITY with *out_n = the size needed when `cap` is too small.
extern "C" int crf_gunzip(const uint8_t *gz, uint64_t n, uint8_t *out, uint64_t cap, uint64_t *out_n, int use_zlib) {
    if (!gz || !out_n || (cap && !out)) { set_err("crf_gunzip: null argument"); return CRF_ERR_ARG; }
    try {
        using namespace fasta_detail;
        crf_inflate::OutBuf fast;
        std::vector<uint8_t> slow;
        const uint8_t *p = nullptr;
        uint64_t got = 0;
        if (use_zlib != 1 && crf_inflate::gunzip(gz, (size_t)n, fast, 4)) {
            p = fast.p; got = fast.size;
        } else if (use_zlib == 2) {
            set_err("crf_gunzip: the reader's decoder does not take this stream");
            return CRF_ERR_UNSUPPORTED;
        } else {
            FileBytes in;
            in.data = gz; in.size = (size_t)n;
            if (!inflate_all(in, slow)) { set_err("crf_gunzip: not a valid gzip stream"); return CRF_ERR_ARG; }
            p = slow.data(); got = slow.size();
        }
        *out_n = got;
        if (got > cap) { set_err("crf_gunzip: capacity %llu too small for %llu bytes", (unsigned long long)cap, (unsigned long long)got); return CRF_ERR_CAPACITY; }
        if (got) memcpy(out, p, (size_t)got);
        return CRF_OK;
    } catch (const std::bad_alloc &) {
        set_err("crf_gunzip: out of host memory");
        return CRF_ERR_NOMEM;
    }
}

extern "C" int crf_fasta_info(const crf_fasta *fa, uint64_t *n_records, uint64_t *total_bases, int *pinned) {
    if (!fa) { set_err("null fasta handle"); return CRF_ERR_ARG; }
    if (n_records) *n_records = fa->offsets.size() - 1;
    if (total_bases) *total_bases = fa->total;
    if (pinned) *pinned = fa->bases_buf.pinned() ? 1 : 0;
    return CRF_OK;
}

extern "C" int crf_fasta_data(const crf_fasta *fa, const uint8_t **bases, const uint64_t **offsets, const char **names,
                              uint64_t *names_bytes) {
    if (!fa) { set_err("null fasta handle"); return CRF_ERR_ARG; }
    if (bases) {                                        // a .2bit or BAM file's text: decoded once, under the handle's lock
        const int rc = fasta_detail::decode_text(const_cast<crf_fasta *>(fa));
        if (rc != CRF_OK) return rc;
    }
    if (bases) *bases = fa->bases;
    if (offsets) *offsets = fa->offsets.data();
    if (names) *names = fa->names.data();
    if (names_bytes) *names_bytes = fa->names.size();
    return CRF_OK;
}

extern "C" int crf_fasta_index(const crf_fasta *fa, const uint64_t **offsets, const char **names, uint64_t *names_bytes) {
    if (!fa) { set_err("crf_fasta_index: null fasta handle"); return CRF_ERR_ARG; }
    if (offsets) *offsets = fa->offsets.data();
    if (names) *names = fa->names.data();
    if (names_bytes) *names_bytes = fa->names.size();
    return CRF_OK;
}

extern "C" int crf_fasta_twobit(const crf_fasta *fa, const uint8_t **dna, const uint64_t **rec_byte, const uint64_t **runs,
                                uint64_t *n_runs) {
    if (!fa || !dna || !rec_byte || !runs || !n_runs) { set_err("crf_fasta_twobit: null argument"); return CRF_ERR_ARG; }
    if (fa->format != FORMAT_2BIT) { set_err("crf_fasta_twobit: not a .2bit file"); return CRF_ERR_ARG; }
    *dna = fa->codes.p;
    *rec_byte = fa->rec_byte.data();
    *runs = fa->n_runs.data();
    *n_runs = fa->n_runs.size() / 2;
    return CRF_OK;
}

extern "C" int crf_fasta_nibbles(const crf_fasta *fa, const uint8_t **nib, const uint64_t **rec_byte, const uint64_t **exotic,
                                 uint64_t *n_exotic) {
    if (!fa || !nib || !rec_byte || !exotic || !n_exotic) { set_err("crf_fasta_nibbles: null argument"); return CRF_ERR_ARG; }
    if (fa->format != FORMAT_BAM) { set_err("crf_fasta_nibbles: not a BAM file"); return CRF_ERR_ARG; }
    *nib = fa->codes.p;
    *rec_byte = fa->rec_byte.data();
    *exotic = fa->nib_exotic.data();
    *n_exotic = fa->nib_exotic.size();
    return CRF_OK;
}

extern "C" int crf_fasta_format(const crf_fasta *fa, int *format) {
    if (!fa || !format) { set_err("crf_fasta_format: null argument"); return CRF_ERR_ARG; }
    *format = fa->format;
    return CRF_OK;
}

extern "C" int crf_fasta_quals(const crf_fasta *fa, const uint8_t **quals) {
    if (!fa || !quals) { set_err("crf_fasta_quals: null argument"); return CRF_ERR_ARG; }
    *quals = fa->quals;
    return CRF_OK;
}

extern "C" int crf_fasta_close(crf_fasta *fa) {
    delete fa;
    return CRF_OK;
}
