// Sanitizer harness for .2bit input: the reader (csrc/crf_fasta.h, fasta_detail::parse_twobit and decode_text) and the
// rows writer that reads the motif from the packed bases (csrc/crf_rows.h, crf_write_rows_twobit), compiled WITHOUT the
// CUDA runtime -- the page-locked allocation is stubbed to "no device" -- under AddressSanitizer + UBSan.
//  * Reader: seeded random .2bit files (both byte orders, versions 0 and 1, records of 0 to 300 bases in shuffled data
//    order, N and mask blocks that overlap, come unsorted or are empty) are read on 1 and 5 threads and compared with a
//    statement of twoBitToFa written here one base at a time.
//  * The same files with bytes of the header, index and record headers flipped: every outcome is CRF_OK (then the text is
//    decoded) or CRF_ERR_ARG, never a fault.
//  * Writer: crf_write_rows_twobit against crf_write_rows on the decoded text, BED and TSV, enough rows for several
//    formatting threads and waves.
// Prints "ok <files> files <flips> flips <writes> writes" and exits 0 when all match.
//   g++ -std=c++17 -O1 -g -fsanitize=address,undefined -pthread -I csrc -I include fuzz_twobit.cpp -lz
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
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

struct Rec {
    std::string name;
    std::vector<uint8_t> codes;                       // 0..3 = T C A G
    std::vector<std::pair<uint32_t, uint32_t>> nb, mb;   // (start, size)
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

static void put32(std::string &s, uint32_t v, bool swap) {
    if (swap) v = __builtin_bswap32(v);
    s.append((const char *)&v, 4);
}

static std::string file_of(const std::vector<Rec> &recs, bool swap, int version, std::mt19937_64 &rng) {
    std::vector<size_t> order(recs.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = i;
    std::shuffle(order.begin(), order.end(), rng);
    size_t at = 16;
    for (const Rec &r : recs) at += 1 + r.name.size() + (version ? 8 : 4);
    std::vector<uint64_t> where(recs.size());
    std::string data;
    for (size_t i : order) {
        const Rec &r = recs[i];
        where[i] = at + data.size();
        put32(data, (uint32_t)r.codes.size(), swap);
        for (int kind = 0; kind < 2; ++kind) {
            const auto &b = kind ? r.mb : r.nb;
            put32(data, (uint32_t)b.size(), swap);
            for (const auto &x : b) put32(data, x.first, swap);
            for (const auto &x : b) put32(data, x.second, swap);
        }
        put32(data, 0, swap);
        for (size_t j = 0; j < r.codes.size(); j += 4) {
            uint8_t byte = 0;
            for (size_t q = 0; q < 4; ++q) byte |= (uint8_t)((j + q < r.codes.size() ? r.codes[j + q] : 0) << (6 - 2 * q));
            data.push_back((char)byte);
        }
    }
    std::string s;
    put32(s, 0x1A412743u, swap);
    put32(s, (uint32_t)version, swap);
    put32(s, (uint32_t)recs.size(), swap);
    put32(s, 0, swap);
    for (size_t i = 0; i < recs.size(); ++i) {
        s.push_back((char)recs[i].name.size());
        s += recs[i].name;
        if (version) {
            uint64_t v = swap ? __builtin_bswap64(where[i]) : where[i];
            s.append((const char *)&v, 8);
        } else {
            put32(s, (uint32_t)where[i], swap);
        }
    }
    return s + data;
}

static std::string twobit_to_fa(const Rec &r) {     // one base at a time
    std::string t;
    for (size_t i = 0; i < r.codes.size(); ++i) {
        bool n = false, m = false;
        for (const auto &b : r.nb) n |= i >= b.first && i < (uint64_t)b.first + b.second;
        for (const auto &b : r.mb) m |= i >= b.first && i < (uint64_t)b.first + b.second;
        char c = n ? 'N' : "TCAG"[r.codes[i]];
        t += m ? (char)(c | 0x20) : c;
    }
    return t;
}

static std::vector<Rec> random_recs(std::mt19937_64 &rng, size_t n, size_t max_len) {
    std::vector<Rec> recs(n);
    for (size_t i = 0; i < n; ++i) {
        Rec &r = recs[i];
        r.name = "seq" + std::to_string(i);
        const size_t len = rng() % 5 == 0 ? rng() % 10 : rng() % (max_len + 1);
        for (size_t j = 0; j < len; ++j) r.codes.push_back((uint8_t)(rng() % 4));
        for (int kind = 0; kind < 2 && len; ++kind) {
            auto &b = kind ? r.mb : r.nb;
            for (int k = (int)(rng() % 5); k > 0; --k) {
                const uint32_t s = (uint32_t)(rng() % (len + 1));
                b.push_back({s, (uint32_t)(rng() % (len - s + 1))});
            }
            if (rng() % 2) b.push_back({(uint32_t)len - 1, 1});
        }
    }
    return recs;
}

static bool read_file(const std::string &path, unsigned threads, crf_fasta **fa) {
    return crf_fasta_open(path.c_str(), threads, 0, fa) == CRF_OK;
}

int main(int argc, char **argv) {
    if (argc < 2) { printf("usage: %s <dir>\n", argv[0]); return 2; }
    const std::string path = std::string(argv[1]) + "/fuzz.2bit";
    std::mt19937_64 rng(2030);
    uint64_t files = 0, flips = 0, writes = 0;
    for (int round = 0; round < 120; ++round) {
        const std::vector<Rec> recs = random_recs(rng, 1 + rng() % 20, round % 6 == 0 ? 300 : 70);
        const bool swap = round & 1;
        const int version = (round >> 1) & 1;
        const std::string blob = file_of(recs, swap, version, rng);
        FILE *f = fopen(path.c_str(), "wb");
        fwrite(blob.data(), 1, blob.size(), f);
        fclose(f);
        for (unsigned threads : {1u, 5u}) {
            crf_fasta *fa = nullptr;
            if (!read_file(path, threads, &fa)) { printf("round %d: %s\n", round, g_err); return 1; }
            const uint8_t *bases;
            const uint64_t *offsets;
            const char *names;
            uint64_t nb;
            crf_fasta_data(fa, &bases, &offsets, &names, &nb);
            for (size_t r = 0; r < recs.size(); ++r) {
                const std::string want = twobit_to_fa(recs[r]);
                if (std::string((const char *)bases + offsets[r], offsets[r + 1] - offsets[r]) != want ||
                    strcmp(names + fa->name_off[r], recs[r].name.c_str()) != 0) {
                    printf("round %d threads %u: record %zu differs\n", round, threads, r);
                    return 1;
                }
            }
            crf_fasta_close(fa);
            ++files;
        }
        // flipped bytes in the header, the index and the record headers (the packed bases are any bytes anyway)
        size_t hdr_end = 16;
        for (const Rec &r : recs) hdr_end += 1 + r.name.size() + (version ? 8 : 4);
        for (int k = 0; k < 40; ++k) {
            std::string bad = blob;
            const size_t at = rng() % 3 == 0 ? rng() % hdr_end : rng() % bad.size();
            bad[at] = (char)(bad[at] ^ (uint8_t)(1u << (rng() % 8)));
            if (rng() % 8 == 0) bad.resize(rng() % bad.size());
            f = fopen(path.c_str(), "wb");
            fwrite(bad.data(), 1, bad.size(), f);
            fclose(f);
            crf_fasta *fa = nullptr;
            const int rc = crf_fasta_open(path.c_str(), 1 + rng() % 4, 0, &fa);
            if (rc == CRF_OK) {
                const uint8_t *bases;
                if (fa->format == 2 && crf_fasta_data(fa, &bases, nullptr, nullptr, nullptr) == CRF_OK && fa->total)
                    for (uint64_t i = 0; i < fa->total; ++i)
                        if (!strchr("TCAGNtcagn", bases[i])) { printf("flip round %d: byte %u\n", round, bases[i]); return 1; }
                crf_fasta_close(fa);
            } else if (rc != CRF_ERR_ARG) {
                printf("flip round %d: status %d (%s)\n", round, rc, g_err);
                return 1;
            }
            ++flips;
        }
    }

    // rows writer: the motif from the packed bytes == from the decoded text
    for (int round = 0; round < 6; ++round) {
        const bool big = round >= 4;
        const std::vector<Rec> recs = random_recs(rng, big ? 30 : 1 + rng() % 10, big ? 40000 : 500);
        const std::string blob = file_of(recs, round & 1, 0, rng);
        FILE *f = fopen(path.c_str(), "wb");
        fwrite(blob.data(), 1, blob.size(), f);
        fclose(f);
        crf_fasta *fa = nullptr;
        if (!read_file(path, 3, &fa)) { printf("writer round %d: %s\n", round, g_err); return 1; }
        const uint8_t *bases, *dna;
        const uint64_t *offsets, *rec_byte, *runs;
        const char *names;
        uint64_t name_bytes, n_runs;
        crf_fasta_data(fa, &bases, &offsets, &names, &name_bytes);
        crf_fasta_twobit(fa, &dna, &rec_byte, &runs, &n_runs);
        std::vector<uint32_t> rec, st, en, k;
        for (int i = 0; i < (big ? 200000 : 300); ++i) {
            const uint32_t r = (uint32_t)(rng() % recs.size());
            const uint64_t len = offsets[r + 1] - offsets[r];
            if (len < 2) continue;
            const uint32_t kk = 1 + (uint32_t)(rng() % std::min<uint64_t>(50, len - 1));
            const uint32_t s = (uint32_t)(rng() % (len - kk + 1));
            rec.push_back(r); st.push_back(s); en.push_back(s + kk); k.push_back(kk);
        }
        std::vector<size_t> idx(rec.size());
        for (size_t i = 0; i < idx.size(); ++i) idx[i] = i;
        std::sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return rec[a] < rec[b]; });
        std::vector<uint32_t> r2, s2, e2, k2;
        for (size_t i : idx) {
            // a motif never holds an N: rows over N or n are left out
            bool has_n = false;
            for (uint32_t j = 0; j < k[i]; ++j) has_n |= (bases[offsets[rec[i]] + st[i] + j] | 0x20) == 'n';
            if (has_n) continue;
            r2.push_back(rec[i]); s2.push_back(st[i]); e2.push_back(en[i]); k2.push_back(k[i]);
        }
        for (int tsv = 0; tsv < 2; ++tsv) {
            uint64_t a = 0, b = 0;
            const std::string pa = std::string(argv[1]) + "/a", pb = std::string(argv[1]) + "/b";
            if (crf_write_rows(pa.c_str(), 0, tsv, names, bases, offsets, r2.data(), s2.data(), e2.data(), k2.data(), r2.size(), &a) ||
                crf_write_rows_twobit(pb.c_str(), 0, tsv, names, dna, rec_byte, r2.data(), s2.data(), e2.data(), k2.data(),
                                      r2.size(), &b)) {
                printf("writer round %d: %s\n", round, g_err);
                return 1;
            }
            if (a != b || slurp(pa) != slurp(pb)) { printf("writer round %d tsv %d: files differ\n", round, tsv); return 1; }
            ++writes;
        }
        crf_fasta_close(fa);
    }
    printf("ok %llu files %llu flips %llu writes\n", (unsigned long long)files, (unsigned long long)flips,
           (unsigned long long)writes);
    return 0;
}
