// Sanitizer harness for FASTQ: the reader (csrc/crf_fasta.h, fasta_detail::parse_fastq) and the masked FASTQ writer
// (csrc/crf_fasta_out.h, crf_write_fastq_masked), compiled WITHOUT the CUDA runtime -- the page-locked allocation is
// stubbed to "no device" -- under AddressSanitizer + UBSan.
//  * Reader: seeded random FASTQ texts (empty reads, descriptions, CRLF, quality lines starting with '@', '+' and '>',
//    sometimes a multi-line record or a blank line) are parsed with pieces of 1 to 97 bytes and 8 MiB on 1 and 5 threads,
//    so that piece boundaries land at every offset inside a record, and compared with the records the text was made of.
//    4-line texts must take the threaded path, the others the serial one.
//  * Writer: random reads (enough bases for several formatting threads and waves) written in soft and hard mode and
//    compared byte for byte with the format stated here one base at a time.
// Prints "ok <texts> texts <parses> parses <files> files" and exits 0 when all match.
//   g++ -std=c++17 -O1 -g -fsanitize=address,undefined -pthread -I csrc -I include fuzz_fastq.cpp -lz
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

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

struct Read { std::string name, seq, qual; };

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

static std::vector<Read> random_reads(std::mt19937_64 &rng, size_t n, size_t max_len) {
    const char bases[] = "ACGTNacgtnRYKM";
    std::vector<Read> reads(n);
    for (size_t r = 0; r < n; ++r) {
        Read &rd = reads[r];
        rd.name = "read" + std::to_string(r) + (rng() % 3 == 0 ? ":1:A" : "");
        const size_t len = rng() % 6 == 0 ? 0 : rng() % (max_len + 1);
        for (size_t i = 0; i < len; ++i) rd.seq += bases[rng() % (sizeof bases - 1)];
        for (size_t i = 0; i < len; ++i) {
            const char first[] = "@+>";                 // quality lines that look like headers or '+' lines
            rd.qual += i == 0 && rng() % 2 ? first[rng() % 3] : (char)('!' + rng() % 94);
        }
    }
    return reads;
}

// multi: some records on several lines and a blank line between two records (the serial parser's ground)
static std::string fastq_text(std::mt19937_64 &rng, const std::vector<Read> &reads, bool multi) {
    std::string t;
    const bool crlf = rng() % 4 == 0;
    const char *eol = crlf ? "\r\n" : "\n";
    for (size_t r = 0; r < reads.size(); ++r) {
        const Read &rd = reads[r];
        t += "@" + rd.name + (rng() % 3 == 0 ? " 1:N:0:ACGT extra" : "") + eol;
        const bool split = multi && rd.seq.size() > 2 && rng() % 3 == 0;
        const size_t cut = split ? 1 + rng() % (rd.seq.size() - 1) : rd.seq.size();
        t += rd.seq.substr(0, cut) + eol;
        if (split) t += rd.seq.substr(cut) + eol;
        t += std::string("+") + (rng() % 4 == 0 ? rd.name : "") + eol;
        const size_t qcut = split ? 1 + rng() % (rd.qual.size() - 1) : rd.qual.size();
        t += rd.qual.substr(0, qcut) + eol;
        if (split) t += rd.qual.substr(qcut) + eol;
        if (multi && rng() % 7 == 0) t += eol;
    }
    return t;
}

static bool check_parse(const std::string &text, const std::vector<Read> &reads, unsigned threads, uint64_t piece,
                        bool want_serial) {
    crf_fasta *fa = new crf_fasta;
    bool serial = false;
    const uint8_t *t = (const uint8_t *)text.data();
    const int rc = fasta_detail::parse_fastq("fuzz", t, text.size(), 0, threads, piece, 4, fa, &serial);
    bool ok = rc == CRF_OK && serial == want_serial && fa->offsets.size() == reads.size() + 1 && fa->format == 1 &&
              fa->quals != nullptr;
    for (size_t r = 0; ok && r < reads.size(); ++r) {
        const uint64_t a = fa->offsets[r], b = fa->offsets[r + 1];
        ok = strcmp(fa->names.data() + fa->name_off[r], reads[r].name.c_str()) == 0 &&
             std::string((const char *)fa->bases + a, b - a) == reads[r].seq &&
             std::string((const char *)fa->quals + a, b - a) == reads[r].qual;
    }
    if (!ok)
        printf("parse: %zu bytes, %zu reads, threads %u, piece %llu: status %d serial %d, %zu records (%s)\n", text.size(),
               reads.size(), threads, (unsigned long long)piece, rc, (int)serial, fa->offsets.size() - 1, g_err);
    crf_fasta_close(fa);
    return ok;
}

int main(int argc, char **argv) {
    if (argc < 2) { printf("usage: %s <dir>\n", argv[0]); return 2; }
    std::mt19937_64 rng(2029);
    uint64_t texts = 0, parses = 0, files = 0;
    for (int round = 0; round < 60; ++round) {
        const bool multi = round % 3 == 2;
        const std::vector<Read> reads = random_reads(rng, 1 + rng() % 30, round % 5 == 0 ? 300 : 40);
        const std::string text = fastq_text(rng, reads, multi);
        size_t lines = 0;
        for (char c : text) lines += c == '\n';
        const bool has_multi = lines != 4 * reads.size();    // a record on several lines, or a blank line
        ++texts;
        for (uint64_t piece = 1; piece <= 97; piece += 1 + (round % 4)) {
            for (unsigned threads : {1u, 5u}) {
                if (!check_parse(text, reads, threads, piece, has_multi)) return 1;
                ++parses;
            }
        }
        if (!check_parse(text, reads, 3, 8u << 20, has_multi)) return 1;
        ++parses;
    }

    const std::string path = std::string(argv[1]) + "/masked.fq";
    for (int round = 0; round < 8; ++round) {
        const bool big = round % 4 == 3;                 // several threads and waves (slices of 2^20 bases)
        const std::vector<Read> reads = random_reads(rng, big ? 40000 + rng() % 10000 : 1 + rng() % 50, big ? 300 : 200);
        const uint64_t lead = rng() % 40;                // offsets[0] > 0: mask and qualities are indexed like bases
        std::string bases(lead, 'x'), quals(lead, 'y'), names;
        std::vector<uint64_t> offsets{lead};
        for (const Read &rd : reads) {
            bases += rd.seq;
            quals += rd.qual;
            offsets.push_back(bases.size());
            names += rd.name + '\0';
        }
        std::vector<uint32_t> mask(bases.size() / 32 + 1);
        for (auto &w : mask) w = rng() % 4 == 0 ? 0u : rng() % 4 == 0 ? 0xFFFFFFFFu : (uint32_t)rng();
        for (int hard = 0; hard < 2; ++hard) {
            uint64_t bytes = 0;
            if (crf_write_fastq_masked(path.c_str(), names.data(), (const uint8_t *)bases.data(), (const uint8_t *)quals.data(),
                                       offsets.data(), reads.size(), mask.data(), hard, &bytes) != CRF_OK) {
                printf("write failed: %s\n", g_err);
                return 1;
            }
            std::string want;
            for (size_t r = 0; r < reads.size(); ++r) {
                want += "@" + reads[r].name + "\n";
                for (uint64_t p = offsets[r]; p < offsets[r + 1]; ++p) {
                    char c = bases[p];
                    if ((mask[p >> 5] >> (p & 31)) & 1) c = hard ? 'N' : (c >= 'A' && c <= 'Z') ? (char)(c + 32) : c;
                    want += c;
                }
                want += "\n+\n" + reads[r].qual + "\n";
            }
            const std::string got = slurp(path.c_str());
            if (got != want || bytes != want.size()) {
                printf("write round %d hard %d: %zu bytes written, %zu expected\n", round, hard, got.size(), want.size());
                return 1;
            }
            ++files;
        }
    }
    printf("ok %llu texts %llu parses %llu files\n", (unsigned long long)texts, (unsigned long long)parses,
           (unsigned long long)files);
    return 0;
}
