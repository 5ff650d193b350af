// Native BED / TSV row writer (host only): result rows -> text, replacing the per-row Python of
// perfect_repeat_finder.py:148-149 (BED: chrom, start, end, motif) and :166-170 (TSV with header).  Rows are formatted on
// several threads, the motif column read back from the host copy of the text (or from a .2bit or BAM file's codes).
//
// Included at the end of crf_api.cu (shares set_err()); tests/fuzz_reader.cpp compiles it without the CUDA runtime.
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <new>
#include <system_error>
#include <thread>
#include <vector>

#include "crf_codes.h"

static inline char *put_u64(char *p, uint64_t v) {
    char tmp[20];
    int n = 0;
    do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) *p++ = tmp[--n];
    return p;
}

// Where the motif column comes from: the text (one byte per base, upper-cased here) ...
struct TextMotif {
    const uint8_t *bases;
    const uint64_t *offsets;
    char *operator()(char *p, uint32_t r, uint32_t start, uint32_t k) const {
        const uint8_t *m = bases + offsets[r] + start;
        for (uint32_t j = 0; j < k; ++j) {
            uint8_t c = m[j];
            if (c >= 'a' && c <= 'z') c -= 32;
            *p++ = (char)c;
        }
        return p;
    }
};

// ... or codes (crf_codes.h): a .2bit file's packed bases (BITS = 2) or a BAM file's 4-bit codes (BITS = 4), record r's
// codes from byte rec_byte[r].  A motif never holds an N, so the codes alone give the letters the text has, upper-cased.
template <int BITS>
struct CodeMotif {
    const uint8_t *codes;
    const uint64_t *rec_byte;
    char *operator()(char *p, uint32_t r, uint32_t start, uint32_t k) const {
        const uint8_t *d = codes + rec_byte[r];
        for (uint64_t i = start, e = (uint64_t)start + k; i < e; ++i) *p++ = (char)code_letter<BITS>(d, i);
        return p;
    }
};

// origin (may be null): per record, added to the printed start and end (the motif is still read at start)
template <class Motif>
static int write_rows_impl(const char *path, int append, int tsv, const char *names, const Motif &motif,
                           const uint64_t *origin, const uint32_t *record, const uint32_t *start,
                           const uint32_t *end, const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes) {
    FILE *f = fopen(path, append ? "ab" : "wb");
    if (!f) { set_err("crf_write_rows: cannot open %s", path); return CRF_ERR_ARG; }
    struct Closer {                                  // the file is closed on every way out (bad_alloc included)
        FILE *f;
        ~Closer() { if (f) fclose(f); }
    } closer{f};
    std::vector<const char *> name_ptr;
    std::vector<size_t> name_len;
    if (!tsv) {
        uint32_t max_rec = 0;
        for (uint64_t i = 0; i < n_rows; ++i) max_rec = std::max(max_rec, record[i]);
        const char *q = names;
        for (uint32_t r = 0; r <= max_rec && n_rows; ++r) {
            name_ptr.push_back(q);
            name_len.push_back(strlen(q));
            q += name_len.back() + 1;
        }
    }
    uint64_t total = 0;
    bool ok = true;
    auto put = [&](const char *p, size_t n) {        // a short write (disk full, I/O error) is an error, not a shorter file
        if (n && ok) {
            const size_t w = fwrite(p, 1, n, f);
            total += w;
            if (w != n) ok = false;
        }
    };
    if (tsv && !append) put("start_0based\tend\tmotif\n", 23);
    // Rows are formatted by a few threads, each a contiguous slice of a "wave" into its own buffer (the motif column is a
    // random read into the text: a cache miss per row), and the buffers of a wave are written in row order.
    auto row_bytes = [&](uint64_t i) -> size_t { return (tsv ? 0 : name_len[record[i]] + 1) + 42 + motif_size[i] + 1; };
    auto format_rows = [&](uint64_t lo, uint64_t hi, std::vector<char> &buf) -> size_t {
        size_t need = 0;
        for (uint64_t i = lo; i < hi; ++i) need += row_bytes(i);
        if (buf.size() < need) buf.resize(need);
        char *p = buf.data();
        for (uint64_t i = lo; i < hi; ++i) {
            const uint32_t r = record[i], k = motif_size[i];
            const uint64_t o = origin ? origin[r] : 0;
            if (!tsv) { memcpy(p, name_ptr[r], name_len[r]); p += name_len[r]; *p++ = '\t'; }
            p = put_u64(p, o + start[i]); *p++ = '\t';
            p = put_u64(p, o + end[i]); *p++ = '\t';
            p = motif(p, r, start[i], k);
            *p++ = '\n';
        }
        return (size_t)(p - buf.data());
    };
    const uint64_t SLICE_ROWS = 1 << 15;
    const uint32_t n_thr = n_rows < 4 * SLICE_ROWS ? 1u : std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    std::vector<std::vector<char>> bufs(n_thr);
    std::vector<size_t> used(n_thr, 0);
    std::vector<std::thread> th(n_thr);
    std::atomic<bool> no_memory{false};             // (set by the formatting threads)
    for (uint64_t wave = 0; wave < n_rows && ok; wave += SLICE_ROWS * n_thr) {
        for (uint32_t t = 0; t < n_thr; ++t) {
            const uint64_t lo = std::min(n_rows, wave + SLICE_ROWS * t), hi = std::min(n_rows, lo + SLICE_ROWS);
            used[t] = 0;
            if (lo == hi) continue;
            auto job = [&, t, lo, hi]() {
                try { used[t] = format_rows(lo, hi, bufs[t]); } catch (const std::bad_alloc &) { no_memory = true; }
            };
            if (n_thr == 1) { job(); continue; }
            try { th[t] = std::thread(job); } catch (const std::system_error &) { job(); }
        }
        for (auto &t : th)
            if (t.joinable()) t.join();
        if (no_memory) throw std::bad_alloc();
        for (uint32_t t = 0; t < n_thr; ++t) put(bufs[t].data(), used[t]);
    }
    if (ferror(f)) ok = false;
    closer.f = nullptr;
    if (fclose(f) != 0) ok = false;
    if (bytes) *bytes = total;
    if (!ok) { set_err("crf_write_rows: write to %s failed (after %llu bytes)", path, (unsigned long long)total); return CRF_ERR_IO; }
    return CRF_OK;
}

// The argument checks and the C boundary of every rows entry point: Motif{src, index} reads the motif column.
template <class Motif>
static int write_rows_checked(const char *path, int append, int tsv, const char *names, const uint8_t *src,
                              const uint64_t *index, const uint64_t *origin, const uint32_t *record, const uint32_t *start,
                              const uint32_t *end, const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes) {
    if (!path || (n_rows && (!src || !index || !record || !start || !end || !motif_size)) || (!tsv && !names)) {
        set_err("crf_write_rows: null argument");
        return CRF_ERR_ARG;
    }
    try {                                            // no exception crosses the C boundary
        return write_rows_impl(path, append, tsv, names, Motif{src, index}, origin, record, start, end, motif_size, n_rows,
                               bytes);
    } catch (const std::bad_alloc &) {
        set_err("crf_write_rows: out of host memory");
        return CRF_ERR_NOMEM;
    }
}

extern "C" int crf_write_rows_at(const char *path, int append, int tsv, const char *names, const uint8_t *bases,
                                 const uint64_t *offsets, const uint64_t *origin, const uint32_t *record, const uint32_t *start,
                                 const uint32_t *end, const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes) {
    return write_rows_checked<TextMotif>(path, append, tsv, names, bases, offsets, origin, record, start, end, motif_size, n_rows,
                                         bytes);
}

extern "C" int crf_write_rows(const char *path, int append, int tsv, const char *names, const uint8_t *bases,
                              const uint64_t *offsets, const uint32_t *record, const uint32_t *start,
                              const uint32_t *end, const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes) {
    return crf_write_rows_at(path, append, tsv, names, bases, offsets, nullptr, record, start, end, motif_size, n_rows, bytes);
}

// The rows of records read from a .2bit file (crf_fasta_twobit: dna, rec_byte), the motif read from the packed bases: the
// same bytes crf_write_rows writes from the file's decoded text, without that text.
extern "C" int crf_write_rows_twobit(const char *path, int append, int tsv, const char *names, const uint8_t *dna,
                                     const uint64_t *rec_byte, const uint32_t *record, const uint32_t *start,
                                     const uint32_t *end, const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes) {
    return write_rows_checked<CodeMotif<2>>(path, append, tsv, names, dna, rec_byte, nullptr, record, start, end, motif_size,
                                            n_rows, bytes);
}

// The rows of reads from a BAM file (crf_fasta_nibbles: nib, rec_byte), the motif read from the codes: the same bytes
// crf_write_rows writes from the file's decoded text, without that text.
extern "C" int crf_write_rows_nibbles(const char *path, int append, int tsv, const char *names, const uint8_t *nib,
                                      const uint64_t *rec_byte, const uint32_t *record, const uint32_t *start,
                                      const uint32_t *end, const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes) {
    return write_rows_checked<CodeMotif<4>>(path, append, tsv, names, nib, rec_byte, nullptr, record, start, end, motif_size,
                                            n_rows, bytes);
}
