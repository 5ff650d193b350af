// Sanitizer harness for the masked FASTA writer (csrc/crf_fasta_out.h: crf_write_fasta_masked), compiled WITHOUT the CUDA
// runtime under AddressSanitizer + UBSan.  Seeded random files -- empty records, records of every length around the line
// width and the 32-bit mask words, lower case, IUPAC letters and bytes above 127, enough bases for several formatting
// threads and waves -- are written in soft and hard mode and compared byte for byte with the format stated here one base
// at a time.  Prints "ok <files> files <bytes> bytes" and exits 0 when all match.
//   g++ -std=c++17 -O1 -g -fsanitize=address,undefined -pthread -I csrc -I include fuzz_mask_writer.cpp
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

#include "crf_fasta_out.h"

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
    if (argc < 2) { printf("usage: %s <dir>\n", argv[0]); return 2; }
    const std::string path = std::string(argv[1]) + "/masked.fa";
    std::mt19937_64 rng(2027);
    const char alphabet[] = "ACGTacgtNnRYKMswbd-*\xe9";
    uint64_t files = 0, total_bytes = 0;
    for (int round = 0; round < 24; ++round) {
        const bool big = round % 12 == 11;                   // several threads and waves (slices of 2^20 bases)
        const uint64_t n_rec = big ? 3000 + rng() % 3000 : 1 + rng() % 40;
        const uint64_t lead = rng() % 40;                   // offsets[0] > 0: the mask is indexed like bases
        std::vector<uint64_t> offsets{lead};
        std::string names;
        for (uint64_t r = 0; r < n_rec; ++r) {
            const uint64_t kind = rng() % 8;
            const uint64_t len = kind == 0 ? 0 : kind == 1 ? 1 + rng() % 3 : big ? rng() % 12000 : rng() % 700;
            offsets.push_back(offsets.back() + len);
            names += "rec" + std::to_string(r) + (r % 5 == 0 ? "_long_name_of_record" : "") + '\0';
        }
        const uint64_t n = offsets.back() + rng() % 50;     // bases past the last record are never written
        std::vector<uint8_t> bases(n);
        for (auto &b : bases) b = (uint8_t)alphabet[rng() % (sizeof alphabet - 1)];
        std::vector<uint32_t> mask((n + 31) / 32 + 1);
        for (auto &w : mask) w = rng() % 4 == 0 ? 0u : rng() % 4 == 0 ? 0xFFFFFFFFu : (uint32_t)rng();
        const uint32_t width = round % 4 == 0 ? 60 : 1 + (uint32_t)(rng() % 90);
        for (int hard = 0; hard < 2; ++hard) {
            uint64_t bytes = 0;
            if (crf_write_fasta_masked(path.c_str(), names.data(), bases.data(), offsets.data(), n_rec, mask.data(), hard,
                                       width, &bytes) != CRF_OK) {
                printf("write failed: %s\n", g_err);
                return 1;
            }
            std::string want;
            const char *q = names.data();
            for (uint64_t r = 0; r < n_rec; ++r) {
                want += '>';
                want += q;
                want += '\n';
                q += strlen(q) + 1;
                for (uint64_t p = offsets[r]; p < offsets[r + 1]; ++p) {
                    char c = (char)bases[p];
                    if ((mask[p >> 5] >> (p & 31)) & 1) c = hard ? 'N' : (c >= 'A' && c <= 'Z') ? (char)(c + 32) : c;
                    want += c;
                    if ((p - offsets[r] + 1) % width == 0 || p + 1 == offsets[r + 1]) want += '\n';
                }
            }
            const std::string got = slurp(path.c_str());
            if (got != want || bytes != want.size()) {
                printf("round %d hard %d width %u: %zu bytes written, %zu expected\n", round, hard, width, got.size(),
                       want.size());
                return 1;
            }
            ++files;
            total_bytes += got.size();
        }
    }
    printf("ok %llu files %llu bytes\n", (unsigned long long)files, (unsigned long long)total_bytes);
    return 0;
}
