// Masked FASTA / FASTQ writer (host only): the records as read, with the bases a mask marks lower-cased (soft) or replaced
// by N (hard) -- what TRF's -m output, dustmasker or a soft-masked reference give.  Formatted on several threads, in waves
// of equal slices of the bases written in order, as crf_rows.h writes rows.
//
// Included at the end of crf_api.cu after crf_rows.h (shares set_err()); tests/fuzz_mask_writer.cpp compiles it without
// the CUDA runtime.
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

// Formats the part of the file that stands for bases [p0, p1) into buf: the header of every record that starts there
// (`last`: also those that start at p1, the empty records at the very end) and the bases with their line breaks.
// quals != NULL: FASTQ, the bases on one line, and the slice that ends a record (or starts it, when it is empty) writes its
// "+" line and qualities.
static size_t fasta_out_slice(const char *const *name_ptr, const size_t *name_len, const uint8_t *bases,
                              const uint8_t *quals, const uint64_t *offsets, uint64_t n_records, const uint32_t *mask,
                              int hard, uint32_t width, uint64_t p0, uint64_t p1, bool last, std::vector<char> &buf) {
    auto ends_here = [&](uint64_t rs, uint64_t re) { return re <= p1 && (re > p0 || (rs == re && rs >= p0)); };
    uint64_t r = (uint64_t)(std::lower_bound(offsets, offsets + n_records, p0) - offsets);
    if (r > 0 && (r == n_records || offsets[r] > p0)) --r;   // the slice starts inside record r - 1
    const uint64_t r_begin = r;
    size_t need = 0;                                         // bytes + one line break per started line + headers
    for (uint64_t q = r_begin; q < n_records && (offsets[q] < p1 || (last && offsets[q] == p1)); ++q) {
        const uint64_t a = std::max(offsets[q], p0), b = std::min(offsets[q + 1], p1);
        if (offsets[q] >= p0) need += name_len[q] + 2;
        if (b > a) need += (b - a) + (b - a) / width + 2;
        if (quals && ends_here(offsets[q], offsets[q + 1])) need += offsets[q + 1] - offsets[q] + 4;
    }
    if (buf.size() < need) buf.resize(need);
    char *out = buf.data();
    for (; r < n_records && (offsets[r] < p1 || (last && offsets[r] == p1)); ++r) {
        const uint64_t rs = offsets[r], re = offsets[r + 1];
        if (rs >= p0) {
            *out++ = quals ? '@' : '>';
            memcpy(out, name_ptr[r], name_len[r]);
            out += name_len[r];
            *out++ = '\n';
        }
        uint64_t p = std::max(rs, p0);
        const uint64_t stop = std::min(re, p1);
        while (p < stop) {                                   // one line, or the part of it inside the slice
            const uint64_t line_end = quals ? re : rs + ((p - rs) / width + 1) * width;
            const uint64_t q = std::min(line_end, stop);
            memcpy(out, bases + p, q - p);
            for (uint64_t w = p >> 5; w <= (q - 1) >> 5; ++w) {
                uint32_t m = mask[w];
                if (w == p >> 5) m &= 0xFFFFFFFFu << (p & 31);
                if (w == (q - 1) >> 5 && (q & 31)) m &= (1u << (q & 31)) - 1u;
                while (m) {
                    const uint64_t i = (w << 5) + (uint64_t)__builtin_ctz(m) - p;
                    m &= m - 1;
                    if (hard) out[i] = 'N';
                    else if (out[i] >= 'A' && out[i] <= 'Z') out[i] = (char)(out[i] + 32);
                }
            }
            out += q - p;
            if (q == line_end || q == re) *out++ = '\n';
            p = q;
        }
        if (quals && ends_here(rs, re)) {
            if (rs == re) *out++ = '\n';
            *out++ = '+';
            *out++ = '\n';
            memcpy(out, quals + rs, re - rs);
            out += re - rs;
            *out++ = '\n';
        }
    }
    return (size_t)(out - buf.data());
}

// fn: the caller's name, for messages
static int write_fasta_masked_impl(const char *fn, const char *path, const char *names, const uint8_t *bases,
                                   const uint8_t *quals, const uint64_t *offsets, uint64_t n_records, const uint32_t *mask,
                                   int hard, uint32_t width, uint64_t *bytes) {
    FILE *f = fopen(path, "wb");
    if (!f) { set_err("%s: cannot open %s", fn, path); return CRF_ERR_ARG; }
    struct Closer {                                  // the file is closed on every way out (bad_alloc included)
        FILE *f;
        ~Closer() { if (f) fclose(f); }
    } closer{f};
    std::vector<const char *> name_ptr(n_records);
    std::vector<size_t> name_len(n_records);
    const char *q = names;
    for (uint64_t r = 0; r < n_records; ++r) {
        name_ptr[r] = q;
        name_len[r] = strlen(q);
        q += name_len[r] + 1;
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
    const uint64_t lo = n_records ? offsets[0] : 0, hi = n_records ? offsets[n_records] : 0;
    const uint64_t SLICE = 1 << 20;                  // bases per thread and wave
    const uint64_t n_slices = n_records ? std::max<uint64_t>(1, (hi - lo + SLICE - 1) / SLICE) : 0;
    const uint32_t n_thr = n_slices < 4 ? 1u : std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    std::vector<std::vector<char>> bufs(n_thr);
    std::vector<size_t> used(n_thr, 0);
    std::vector<std::thread> th(n_thr);
    std::atomic<bool> no_memory{false};             // (set by the formatting threads)
    for (uint64_t wave = 0; wave < n_slices && ok; wave += n_thr) {
        for (uint32_t t = 0; t < n_thr; ++t) {
            const uint64_t j = wave + t, p0 = lo + j * SLICE, p1 = std::min(hi, p0 + SLICE);
            const bool last = j == n_slices - 1;     // (it also writes the empty records that end the file)
            used[t] = 0;
            if (j >= n_slices) continue;
            auto job = [&, t, p0, p1, last]() {
                try {
                    used[t] = fasta_out_slice(name_ptr.data(), name_len.data(), bases, quals, offsets, n_records, mask, hard,
                                              width, p0, p1, last, bufs[t]);
                } catch (const std::bad_alloc &) { no_memory = true; }
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
    if (!ok) {
        set_err("%s: write to %s failed (after %llu bytes)", fn, path, (unsigned long long)total);
        return CRF_ERR_IO;
    }
    return CRF_OK;
}

// The checks and the call both writers share.  quals: NULL for FASTA.
static int write_masked(const char *fn, const char *path, const char *names, const uint8_t *bases, const uint8_t *quals,
                        const uint64_t *offsets, uint64_t n_records, const uint32_t *mask, int hard, uint32_t line_width,
                        uint64_t *bytes) {
    if (!path || (n_records && (!names || !offsets)) || line_width == 0) {
        set_err("%s: null argument or zero line width", fn);
        return CRF_ERR_ARG;
    }
    if (n_records && offsets[n_records] > offsets[0] && (!bases || !mask)) {
        set_err("%s: null bases or mask", fn);
        return CRF_ERR_ARG;
    }
    for (uint64_t r = 0; r < n_records; ++r)
        if (offsets[r + 1] < offsets[r]) { set_err("%s: offsets decrease at record %llu", fn, (unsigned long long)r); return CRF_ERR_ARG; }
    try {                                            // no exception crosses the C boundary
        return write_fasta_masked_impl(fn, path, names, bases, quals, offsets, n_records, mask, hard, line_width, bytes);
    } catch (const std::bad_alloc &) {
        set_err("%s: out of host memory", fn);
        return CRF_ERR_NOMEM;
    }
}

extern "C" int crf_write_fasta_masked(const char *path, const char *names, const uint8_t *bases, const uint64_t *offsets,
                                      uint64_t n_records, const uint32_t *mask, int hard, uint32_t line_width,
                                      uint64_t *bytes) {
    return write_masked("crf_write_fasta_masked", path, names, bases, nullptr, offsets, n_records, mask, hard, line_width,
                        bytes);
}

extern "C" int crf_write_fastq_masked(const char *path, const char *names, const uint8_t *bases, const uint8_t *quals,
                                      const uint64_t *offsets, uint64_t n_records, const uint32_t *mask, int hard,
                                      uint64_t *bytes) {
    if (n_records && !quals) {                       // (an empty read too has a quality line)
        set_err("crf_write_fastq_masked: null qualities");
        return CRF_ERR_ARG;
    }
    return write_masked("crf_write_fastq_masked", path, names, bases, quals, offsets, n_records, mask, hard, UINT32_MAX,
                        bytes);
}
