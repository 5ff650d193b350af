// Sanitizer harness for BAM input: the reader (csrc/crf_fasta.h, fasta_detail::parse_bam and decode_text) and the rows
// writer that reads the motif from the 4-bit codes (csrc/crf_rows.h, crf_write_rows_nibbles), compiled WITHOUT the CUDA
// runtime -- the page-locked allocation is stubbed to "no device" -- under AddressSanitizer + UBSan.
//  * Reader: seeded random BAMs (all flags that matter, every code, absent qualities, names up to 254 characters, CIGAR
//    operations and tags, BGZF blocks of random sizes, with and without the end-of-file block) are read on 1 and 5 threads
//    and windows of one block to the default, and compared with a statement of `samtools fastq -n` written here.
//  * The same streams truncated or with bits flipped (before compression: the parser sees the damage; after: the blocks
//    do): every outcome is CRF_OK (then the text is decoded and the sizes agree) or CRF_ERR_ARG, never a fault.
//  * Writer: crf_write_rows_nibbles against crf_write_rows on the decoded text, BED and TSV, enough rows for several
//    formatting threads and waves.
// Prints "ok <files> files <damaged> damaged <writes> writes" and exits 0 when all match.
//   g++ -std=c++17 -O1 -g -fsanitize=address,undefined -pthread -I csrc -I include fuzz_bam.cpp -lz
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <random>
#include <string>
#include <vector>

#include "crf.h"

typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorNoDevice = 100, cudaHostAllocDefault = 0 };
static cudaError_t cudaHostAlloc(void **, size_t, unsigned) { return cudaErrorNoDevice; }
static cudaError_t cudaFreeHost(void *) { return cudaSuccess; }
static cudaError_t cudaGetLastError() { return cudaSuccess; }
static thread_local char g_err[512];
static void set_err(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

#include "crf_rows.h"
#include "crf_fasta_out.h"
#include "crf_fasta.h"

static const char LET[] = "=ACMGRSVTWYHKDBN";

struct Read {
    std::string name;
    uint16_t flag;
    std::vector<uint8_t> codes;
    std::vector<uint8_t> qual;                        // empty with codes non-empty: absent
    uint16_t n_cigar;
    std::string tags;
};

static std::string slurp(const std::string &path) {
    std::string out;
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) return out;
    char buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) out.append(buf, n);
    fclose(f);
    return out;
}

static void put(std::string &s, uint32_t v, int bytes) { s.append((const char *)&v, bytes); }

static std::string stream_of(const std::vector<Read> &reads) {
    std::string s = "BAM\1";
    const std::string text = "@HD\tVN:1.6\n";
    put(s, (uint32_t)text.size(), 4);
    s += text;
    put(s, 1, 4);
    put(s, 5, 4);
    s += std::string("chr1\0", 5);
    put(s, 1000, 4);
    for (const Read &r : reads) {
        const uint32_t n = (uint32_t)r.codes.size(), lrn = (uint32_t)r.name.size() + 1;
        std::string b;
        put(b, 0xFFFFFFFFu, 4); put(b, 0xFFFFFFFFu, 4);
        put(b, lrn, 1); put(b, 255, 1); put(b, 4680, 2); put(b, r.n_cigar, 2); put(b, r.flag, 2);
        put(b, n, 4); put(b, 0xFFFFFFFFu, 4); put(b, 0xFFFFFFFFu, 4); put(b, 0, 4);
        b += r.name;
        b.push_back('\0');
        b.append(4 * (size_t)r.n_cigar, '\0');
        for (uint32_t i = 0; i < n; i += 2) b.push_back((char)((r.codes[i] << 4) | (i + 1 < n ? r.codes[i + 1] : 0)));
        if (r.qual.empty()) b.append(n, '\xff');
        else b.append((const char *)r.qual.data(), n);
        b += r.tags;
        put(s, (uint32_t)b.size(), 4);
        s += b;
    }
    return s;
}

static std::string bgzf_of(const std::string &raw, std::mt19937_64 &rng, bool eof) {
    std::string out;
    for (size_t i = 0; i < raw.size();) {
        const size_t len = std::min<size_t>(raw.size() - i, 1 + rng() % 65280);
        std::vector<uint8_t> c(compressBound(len) + 64);
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        deflateInit2(&zs, 1 + rng() % 9, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
        zs.next_in = (Bytef *)raw.data() + i;
        zs.avail_in = (uInt)len;
        zs.next_out = c.data();
        zs.avail_out = (uInt)c.size();
        deflate(&zs, Z_FINISH);
        const size_t clen = zs.total_out;
        deflateEnd(&zs);
        std::string h("\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0", 16);
        put(h, (uint32_t)(18 + clen + 8 - 1), 2);
        out += h;
        out.append((const char *)c.data(), clen);
        put(out, (uint32_t)crc32(0, (const Bytef *)raw.data() + i, (uInt)len), 4);
        put(out, (uint32_t)len, 4);
        i += len;
    }
    if (eof) out += std::string("\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0\x1b\0\x03\0\0\0\0\0\0\0\0\0", 28);
    return out;
}

static void write_file(const std::string &path, const std::string &data) {
    FILE *f = fopen(path.c_str(), "wb");
    fwrite(data.data(), 1, data.size(), f);
    fclose(f);
}

// What samtools fastq -n writes, as (names NUL-separated, bases, quals, offsets)
struct Want { std::string names, bases, quals; std::vector<uint64_t> offsets{0}; };
static Want want_of(const std::vector<Read> &reads) {
    Want w;
    for (const Read &r : reads) {
        if (r.flag & 0x900) continue;
        const size_t n = r.codes.size();
        w.names += r.name;
        w.names.push_back('\0');
        for (size_t i = 0; i < n; ++i) {
            const uint8_t c = r.flag & 0x10 ? r.codes[n - 1 - i] : r.codes[i];
            const uint8_t rc = (uint8_t)(((c & 1) << 3) | ((c & 2) << 1) | ((c & 4) >> 1) | ((c & 8) >> 3));
            w.bases.push_back(LET[r.flag & 0x10 ? rc : c]);
            w.quals.push_back(r.qual.empty() ? '"' : (char)(r.qual[r.flag & 0x10 ? n - 1 - i : i] + 33));
        }
        w.offsets.push_back(w.bases.size());
    }
    return w;
}

static bool check_open(const std::string &path, unsigned threads, const Want &w) {
    crf_fasta *fa = nullptr;
    if (crf_fasta_open(path.c_str(), threads, 4, &fa) != CRF_OK) { fprintf(stderr, "open failed: %s\n", g_err); return false; }
    int fmt = -1;
    const uint8_t *bases, *quals;
    const uint64_t *off;
    const char *names;
    uint64_t nb, n_rec, total;
    crf_fasta_format(fa, &fmt);
    crf_fasta_info(fa, &n_rec, &total, nullptr);
    bool ok = fmt == 3 && n_rec + 1 == w.offsets.size() && total == w.bases.size();
    ok = ok && crf_fasta_data(fa, &bases, &off, &names, &nb) == CRF_OK && crf_fasta_quals(fa, &quals) == CRF_OK;
    ok = ok && std::string((const char *)bases, total) == w.bases && std::string((const char *)quals, total) == w.quals;
    ok = ok && std::string(names, nb) == w.names && std::equal(w.offsets.begin(), w.offsets.end(), off);
    crf_fasta_close(fa);
    return ok;
}

int main(int argc, char **argv) {
    const std::string dir = argc > 1 ? argv[1] : "/tmp";
    const std::string path = dir + "/fuzz.bam";
    std::mt19937_64 rng(20260424);
    int files = 0, damaged = 0, writes = 0;
    for (int it = 0; it < 40; ++it) {
        std::vector<Read> reads(rng() % 60);
        const uint16_t flags[] = {0x4, 0x14, 0x0, 0x10, 0x100, 0x800, 0x4d, 0x8d, 0x910, 0x9d};
        for (size_t i = 0; i < reads.size(); ++i) {
            Read &r = reads[i];
            r.name = "r" + std::to_string(i);
            const size_t extra = rng() % 4 == 0 ? 250 : rng() % 20;
            while (r.name.size() < std::min<size_t>(254, 2 + extra)) r.name.push_back((char)('a' + rng() % 26));
            r.flag = flags[rng() % 10];
            r.codes.resize(rng() % 5 == 0 ? 0 : rng() % (rng() % 3 == 0 ? 5000 : 200));
            for (auto &c : r.codes) c = rng() % 8 == 0 ? (uint8_t)(rng() % 16) : (uint8_t)(1u << (rng() % 4));
            if (rng() % 4) { r.qual.resize(r.codes.size()); for (auto &q : r.qual) q = (uint8_t)(rng() % 94); }
            r.n_cigar = rng() % 3 == 0 ? (uint16_t)(rng() % 4) : 0;
            if (rng() % 3 == 0) r.tags = std::string("XZZ") + std::string(rng() % 300, 'k') + std::string("\0", 1);
        }
        const std::string raw = stream_of(reads);
        const Want w = want_of(reads);
        write_file(path, bgzf_of(raw, rng, rng() % 3 != 0));
        for (const char *window : {"1", "70000", ""}) {
            if (*window) setenv("CRF_BAM_WINDOW", window, 1); else unsetenv("CRF_BAM_WINDOW");
            for (unsigned t : {1u, 5u})
                if (!check_open(path, t, w)) { printf("mismatch in file %d (window %s, %u threads)\n", it, window, t); return 1; }
        }
        ++files;
        setenv("CRF_BAM_WINDOW", "1", 1);
        for (int d = 0; d < 40; ++d) {                          // damaged copies: an answer or CRF_ERR_ARG, never a fault
            std::string bad = raw, file;
            const int kind = (int)(rng() % 3);
            if (kind == 0) bad.resize(rng() % (bad.size() + 1));
            else if (kind == 1) for (int k = 0; k < 1 + (int)(rng() % 4); ++k) bad[rng() % bad.size()] ^= (char)(1u << (rng() % 8));
            file = bgzf_of(bad, rng, true);
            if (kind == 2) for (int k = 0; k < 1 + (int)(rng() % 3); ++k) file[rng() % file.size()] ^= (char)(1u << (rng() % 8));
            write_file(path, file);
            crf_fasta *fa = nullptr;
            const int rc = crf_fasta_open(path.c_str(), 1 + (unsigned)(rng() % 5), 4, &fa);
            if (rc == CRF_OK) {
                const uint8_t *bases;
                const uint64_t *off;
                uint64_t n_rec, total;
                crf_fasta_info(fa, &n_rec, &total, nullptr);
                if (crf_fasta_data(fa, &bases, &off, nullptr, nullptr) != CRF_OK || off[n_rec] != total) {
                    printf("inconsistent handle after damage %d of file %d\n", d, it);
                    return 1;
                }
                crf_fasta_close(fa);
            } else if (rc != CRF_ERR_ARG) {
                printf("damage %d of file %d: rc %d (%s)\n", d, it, rc, g_err);
                return 1;
            }
            ++damaged;
        }
        unsetenv("CRF_BAM_WINDOW");
    }
    // the writer: crf_write_rows_nibbles == crf_write_rows on the decoded text
    std::vector<Read> reads(300);
    for (size_t i = 0; i < reads.size(); ++i) {
        reads[i].name = "read" + std::to_string(i);
        reads[i].flag = i % 2 ? 0x14 : 0x4;
        reads[i].codes.resize(100 + rng() % 3000);
        for (auto &c : reads[i].codes) c = rng() % 10 == 0 ? (uint8_t)(rng() % 16) : (uint8_t)(1u << (rng() % 4));
    }
    write_file(path, bgzf_of(stream_of(reads), rng, true));
    crf_fasta *fa = nullptr;
    if (crf_fasta_open(path.c_str(), 3, 0, &fa) != CRF_OK) { printf("writer file: %s\n", g_err); return 1; }
    const uint8_t *bases, *nib;
    const uint64_t *off, *rec_byte, *ex;
    const char *names;
    uint64_t nb, n_ex;
    crf_fasta_data(fa, &bases, &off, &names, &nb);
    crf_fasta_nibbles(fa, &nib, &rec_byte, &ex, &n_ex);
    std::vector<uint32_t> rec, start, end, k;
    for (int i = 0; i < 200000; ++i) rec.push_back((uint32_t)(rng() % reads.size()));
    std::sort(rec.begin(), rec.end());
    for (const uint32_t r : rec) {
        const uint32_t len = (uint32_t)(off[r + 1] - off[r]);
        const uint32_t kk = 1 + (uint32_t)(rng() % 50), s = (uint32_t)(rng() % (len - kk));
        start.push_back(s); end.push_back(std::min(len, s + kk * (1 + (uint32_t)(rng() % 3)))); k.push_back(kk);
    }
    for (int tsv = 0; tsv < 2; ++tsv) {
        uint64_t a = 0, b = 0;
        const std::string pa = dir + "/a.bed", pb = dir + "/b.bed";
        if (crf_write_rows(pa.c_str(), 0, tsv, names, bases, off, rec.data(), start.data(), end.data(), k.data(), rec.size(), &a) ||
            crf_write_rows_nibbles(pb.c_str(), 0, tsv, names, nib, rec_byte, rec.data(), start.data(), end.data(), k.data(),
                                   rec.size(), &b) || a != b || slurp(pa) != slurp(pb)) {
            printf("writer mismatch (tsv %d)\n", tsv);
            return 1;
        }
        ++writes;
    }
    crf_fasta_close(fa);
    printf("ok %d files %d damaged %d writes\n", files, damaged, writes);
    return 0;
}
