// Sanitizer harness for the 64-bit origins of the BED / TSV row writer (csrc/crf_rows.h: crf_write_rows_at), compiled
// WITHOUT the CUDA runtime under AddressSanitizer + UBSan.  Seeded random rows (several threads' worth) are written
//   a) by crf_write_rows and by crf_write_rows_at with origin = NULL: the two files must be byte-identical;
//   b) by crf_write_rows_at with per-record origins around 2^32 and 2^33: every line must equal the same row formatted
//      here with snprintf("%llu").
// Prints "ok <rows> rows" and exits 0 when both hold.
//   g++ -std=c++17 -O1 -g -fsanitize=address,undefined -pthread -I csrc -I include fuzz_rows_at.cpp
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <random>
#include <string>
#include <vector>

#include "crf.h"

static thread_local char g_err[512];
static void set_err(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

#include "crf_rows.h"

static std::string slurp(const char *path) {
    std::string out;
    FILE *f = fopen(path, "rb");
    if (!f) return out;
    char buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) out.append(buf, n);
    fclose(f);
    return out;
}

int main(int argc, char **argv) {
    if (argc < 2) { printf("usage: %s <dir> [rows]\n", argv[0]); return 2; }
    const std::string dir = argv[1];
    const uint64_t n_rows = argc > 2 ? strtoull(argv[2], nullptr, 10) : 200000;
    std::mt19937_64 rng(2026);
    const uint32_t n_rec = 5;
    const uint64_t origin[n_rec] = {0, 0xFFFFFFFFull, 0x100000000ull, (1ull << 33) + 12345, 0xFFFFFFFFull * 3};
    std::string names;
    for (uint32_t r = 0; r < n_rec; ++r) names += "unit" + std::to_string(r) + '\0';
    const uint64_t rec_len = 4096;
    std::vector<uint8_t> bases(n_rec * rec_len);
    for (auto &b : bases) b = "ACGTacgtN"[rng() % 9];
    std::vector<uint64_t> offsets(n_rec);
    for (uint32_t r = 0; r < n_rec; ++r) offsets[r] = r * rec_len;
    std::vector<uint32_t> rec(n_rows), st(n_rows), en(n_rows), kk(n_rows);
    for (uint64_t i = 0; i < n_rows; ++i) {
        rec[i] = (uint32_t)(rng() % n_rec);
        kk[i] = 1 + (uint32_t)(rng() % 50);
        st[i] = (uint32_t)(rng() % (rec_len - 64));
        en[i] = (i % 97 == 0) ? 0xFFFFFFFFu : st[i] + 3 * kk[i];          // the largest 32-bit end, shifted past 2^32
    }
    int bad = 0;
    for (int tsv = 0; tsv < 2; ++tsv) {
        const std::string a = dir + "/plain" + std::to_string(tsv), b = dir + "/null" + std::to_string(tsv),
                          c = dir + "/origin" + std::to_string(tsv);
        uint64_t bytes = 0;
        if (crf_write_rows(a.c_str(), 0, tsv, names.data(), bases.data(), offsets.data(), rec.data(), st.data(), en.data(),
                           kk.data(), n_rows, &bytes) != CRF_OK ||
            crf_write_rows_at(b.c_str(), 0, tsv, names.data(), bases.data(), offsets.data(), nullptr, rec.data(), st.data(),
                              en.data(), kk.data(), n_rows, &bytes) != CRF_OK ||
            crf_write_rows_at(c.c_str(), 0, tsv, names.data(), bases.data(), offsets.data(), origin, rec.data(), st.data(),
                              en.data(), kk.data(), n_rows, &bytes) != CRF_OK) {
            printf("write failed: %s\n", g_err);
            return 1;
        }
        if (slurp(a.c_str()) != slurp(b.c_str())) { printf("tsv %d: origin = NULL differs from crf_write_rows\n", tsv); ++bad; }
        std::string want = tsv ? "start_0based\tend\tmotif\n" : "";
        char line[256];
        for (uint64_t i = 0; i < n_rows; ++i) {
            const uint32_t r = rec[i];
            std::string motif;
            for (uint32_t j = 0; j < kk[i]; ++j) {
                char ch = (char)bases[offsets[r] + st[i] + j];
                if (ch >= 'a' && ch <= 'z') ch -= 32;
                motif += ch;
            }
            snprintf(line, sizeof line, "%llu\t%llu\t", (unsigned long long)(origin[r] + st[i]),
                     (unsigned long long)(origin[r] + en[i]));
            if (!tsv) want += "unit" + std::to_string(r) + '\t';
            want += line + motif + '\n';
        }
        if (slurp(c.c_str()) != want) { printf("tsv %d: rows with origins differ from snprintf\n", tsv); ++bad; }
    }
    if (bad) return 1;
    printf("ok %llu rows\n", (unsigned long long)n_rows);
    return 0;
}
