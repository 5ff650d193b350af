// Host-side packer (no GPU): ASCII bases -> the two 2-bit planes + not-ACGT mask that crf_seq_load_packed uploads
// (0.375 B/bp over PCIe instead of 1 B/bp).  Replaces, together with repack_kernel, what input_sequence.upper()
// (perfect_repeat_finder.py:33) and the per-base str compares of utils/perfect_repeat_tracker.py:53 need from the text.
// Threaded; 32 bases per step with AVX2 when the CPU has it (compare-equal + movemask gives the plane words directly),
// a portable loop otherwise.  Included at the end of crf_api.cu (after crf_fasta.h: shares run_parallel / set_err).
#pragma once
#include <immintrin.h>

namespace pack_detail {

struct Words { uint32_t h, l, nm, is_n; };

static inline Words pack32_scalar(const uint8_t *b, uint32_t n) {   // n <= 32 bases
    Words w = {0, 0, 0xFFFFFFFFu, 0};
    for (uint32_t i = 0; i < n; ++i) {
        uint8_t c = b[i];
        if (c >= 'a' && c <= 'z') c -= 32;
        const uint32_t bit = 1u << i;
        if (c == 'A') { w.nm &= ~bit; }
        else if (c == 'C') { w.l |= bit; w.nm &= ~bit; }
        else if (c == 'G') { w.h |= bit; w.nm &= ~bit; }
        else if (c == 'T') { w.h |= bit; w.l |= bit; w.nm &= ~bit; }
        else if (c == 'N') { w.is_n |= bit; }
    }
    return w;
}

__attribute__((target("avx2"))) static inline Words pack32_avx2(const uint8_t *b) {
    // & 0xDF folds a-z onto A-Z; no other byte value lands on 'A', 'C', 'G', 'T' or 'N'
    const __m256i v = _mm256_and_si256(_mm256_loadu_si256((const __m256i *)b), _mm256_set1_epi8((char)0xDF));
    const uint32_t a = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(v, _mm256_set1_epi8('A')));
    const uint32_t c = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(v, _mm256_set1_epi8('C')));
    const uint32_t g = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(v, _mm256_set1_epi8('G')));
    const uint32_t t = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(v, _mm256_set1_epi8('T')));
    const uint32_t n = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(v, _mm256_set1_epi8('N')));
    return Words{g | t, c | t, ~(a | c | g | t), n};
}

static inline void note_exotic(const uint8_t *bases, uint64_t p0, uint32_t bits, std::vector<uint64_t> &out) {
    while (bits) {
        const uint32_t i = (uint32_t)__builtin_ctz(bits);
        bits &= bits - 1;
        uint8_t c = bases[p0 + i];
        if (c >= 'a' && c <= 'z') c -= 32;
        out.push_back(((p0 + i) << 8) | c);
    }
}

__attribute__((target("avx2"))) static void pack_words_avx2(const uint8_t *bases, uint64_t w_lo, uint64_t w_hi, uint32_t *H,
                                                            uint32_t *L, uint32_t *NM, std::vector<uint64_t> &exo) {
    for (uint64_t w = w_lo; w < w_hi; ++w) {
        const Words x = pack32_avx2(bases + 32 * w);
        H[w] = x.h; L[w] = x.l; NM[w] = x.nm;
        const uint32_t ex = x.nm & ~x.is_n;
        if (ex) note_exotic(bases, 32 * w, ex, exo);
    }
}

static void pack_words_scalar(const uint8_t *bases, uint64_t n, uint64_t w_lo, uint64_t w_hi, uint32_t *H, uint32_t *L,
                              uint32_t *NM, std::vector<uint64_t> &exo) {
    for (uint64_t w = w_lo; w < w_hi; ++w) {
        const uint32_t cnt = (uint32_t)std::min<uint64_t>(32, n - 32 * w);
        const Words x = pack32_scalar(bases + 32 * w, cnt);
        H[w] = x.h; L[w] = x.l; NM[w] = x.nm;
        const uint32_t valid = cnt == 32 ? 0xFFFFFFFFu : ((1u << cnt) - 1u);
        const uint32_t ex = x.nm & ~x.is_n & valid;
        if (ex) note_exotic(bases, 32 * w, ex, exo);
    }
}

// planes of ceil(n / 32) words; positions beyond n are masked.  exotic: ascending (position << 8 | upper-cased byte).
static void pack_all(const uint8_t *bases, uint64_t n, unsigned n_threads, uint32_t *H, uint32_t *L, uint32_t *NM,
                     std::vector<uint64_t> &exotic) {
    const uint64_t n_words = (n + 31) / 32, full = n / 32;
    const bool avx2 = __builtin_cpu_supports("avx2") && !getenv("CRF_PACK_SCALAR");
    const uint64_t PIECE = 1u << 18;                                  // words per work item (8 Mbp)
    const size_t n_items = (size_t)((n_words + PIECE - 1) / PIECE);
    std::vector<std::vector<uint64_t>> exo(n_items);
    fasta_detail::run_parallel(n_threads, n_items, [&](size_t i) {
        const uint64_t lo = i * PIECE, hi = std::min(n_words, lo + PIECE), hi_full = std::min(hi, full);
        if (avx2 && hi_full > lo) pack_words_avx2(bases, lo, hi_full, H, L, NM, exo[i]);
        else if (hi_full > lo) pack_words_scalar(bases, n, lo, hi_full, H, L, NM, exo[i]);
        if (hi > hi_full) pack_words_scalar(bases, n, std::max(lo, hi_full), hi, H, L, NM, exo[i]);   // the ragged last word
    });
    exotic.clear();
    for (auto &v : exo) exotic.insert(exotic.end(), v.begin(), v.end());
}

}  // namespace pack_detail

extern "C" int crf_pack_ascii(const uint8_t *bases, uint64_t n_bases, uint32_t n_threads, uint32_t *H, uint32_t *L,
                              uint32_t *NM, uint64_t *exotic, uint64_t exotic_cap, uint64_t *n_exotic) {
    if ((n_bases && (!bases || !H || !L || !NM)) || !n_exotic) { set_err("crf_pack_ascii: null argument"); return CRF_ERR_ARG; }
    if (n_threads == 0) n_threads = std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    try {
        std::vector<uint64_t> exo;
        pack_detail::pack_all(bases, n_bases, n_threads, H, L, NM, exo);
        *n_exotic = exo.size();
        if (exo.size() > exotic_cap) {
            set_err("crf_pack_ascii: %llu symbols other than A,C,G,T,N; the exotic list holds %llu", (unsigned long long)exo.size(),
                    (unsigned long long)exotic_cap);
            return CRF_ERR_CAPACITY;
        }
        if (!exo.empty()) memcpy(exotic, exo.data(), exo.size() * 8);
    } catch (const std::bad_alloc &) {
        set_err("crf_pack_ascii: out of host memory");
        return CRF_ERR_NOMEM;
    }
    return CRF_OK;
}

// The mask plane as sorted runs of masked positions (what crf_seq_load_packed_runs takes instead of the plane: a genome's N's
// are a few hundred long blocks, so 0.25 instead of 0.375 bytes per base cross PCIe).  Threaded over pieces of the plane.
static void mask_runs(const uint32_t *NM, uint64_t n_bases, unsigned n_threads, std::vector<uint64_t> &runs) {
    const uint64_t n_words = (n_bases + 31) / 32;
    const uint64_t PIECE = 1u << 20;
    const size_t n_items = (size_t)((n_words + PIECE - 1) / PIECE);
    std::vector<std::vector<uint64_t>> part(n_items);
    fasta_detail::run_parallel(n_threads, n_items, [&](size_t it) {
        const uint64_t lo = it * PIECE, hi = std::min(n_words, lo + PIECE);
        std::vector<uint64_t> &out = part[it];
        uint64_t open_at = ~0ull;
        for (uint64_t w = lo; w < hi; ++w) {
            uint32_t m = NM[w];
            if (w == n_words - 1 && (n_bases & 31)) m &= (1u << (n_bases & 31)) - 1u;   // the pad behind the last base is no run
            if (m == 0xFFFFFFFFu) { if (open_at == ~0ull) open_at = 32 * w; continue; }
            if (m == 0) { if (open_at != ~0ull) { out.push_back(open_at); out.push_back(32 * w); open_at = ~0ull; } continue; }
            for (uint32_t b = 0; b < 32;) {                          // a word with both kinds of positions
                if ((m >> b) & 1u) {
                    if (open_at == ~0ull) open_at = 32 * w + b;
                    const uint32_t ones = (uint32_t)__builtin_ctz(~(m >> b) | (b ? (1u << (32 - b)) : 0u));
                    b += ones ? ones : 1;
                    if (b < 32) { out.push_back(open_at); out.push_back(32 * w + b); open_at = ~0ull; }
                } else {
                    if (open_at != ~0ull) { out.push_back(open_at); out.push_back(32 * w + b); open_at = ~0ull; }
                    const uint32_t rest = m >> b;
                    b += rest ? (uint32_t)__builtin_ctz(rest) : 32;
                }
            }
        }
        if (open_at != ~0ull) { out.push_back(open_at); out.push_back(std::min<uint64_t>(32 * hi, n_bases)); }
    });
    runs.clear();
    for (auto &v : part)
        for (size_t i = 0; i + 1 < v.size(); i += 2) {
            if (!runs.empty() && runs.back() == v[i]) runs.back() = v[i + 1];     // a run that continues across pieces
            else { runs.push_back(v[i]); runs.push_back(v[i + 1]); }
        }
}

extern "C" int crf_mask_runs(const uint32_t *NM, uint64_t n_bases, uint32_t n_threads, uint64_t *runs, uint64_t cap,
                             uint64_t *n_runs) {
    if ((n_bases && !NM) || !n_runs) { set_err("crf_mask_runs: null argument"); return CRF_ERR_ARG; }
    if (n_threads == 0) n_threads = std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    try {
        std::vector<uint64_t> r;
        mask_runs(NM, n_bases, n_threads, r);
        *n_runs = r.size() / 2;
        if (r.size() / 2 > cap) {
            set_err("crf_mask_runs: %llu runs; the list holds %llu", (unsigned long long)(r.size() / 2), (unsigned long long)cap);
            return CRF_ERR_CAPACITY;
        }
        if (!r.empty()) memcpy(runs, r.data(), r.size() * 8);
    } catch (const std::bad_alloc &) {
        set_err("crf_mask_runs: out of host memory");
        return CRF_ERR_NOMEM;
    }
    return CRF_OK;
}

// Packed planes of a FASTA file read by crf_fasta_open, made on first use (threaded) and kept with the handle; page-locked
// when crf_fasta_open was asked for it (pinned & 3).
extern "C" int crf_fasta_packed(crf_fasta *fa, uint32_t n_threads, const uint32_t **H, const uint32_t **L, const uint32_t **NM,
                                const uint64_t **exotic, uint64_t *n_exotic) {
    if (!fa || !H || !L || !NM || !exotic || !n_exotic) { set_err("crf_fasta_packed: null argument"); return CRF_ERR_ARG; }
    if (n_threads == 0) n_threads = std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    try {
        if (!fa->planes.p) {
            const int rc = fasta_detail::decode_text(fa);   // (a .2bit or BAM file: its text, decoded on first use)
            if (rc != CRF_OK) return rc;
            const uint64_t n_words = (fa->total + 31) / 32 + 1;
            if (!fa->planes.alloc((size_t)n_words * 12, fa->pinned & 3)) { set_err("crf_fasta_packed: out of host memory"); return CRF_ERR_NOMEM; }
            uint32_t *planes = (uint32_t *)fa->planes.p;
            fa->plane_words = n_words;
            pack_detail::pack_all(fa->bases, fa->total, n_threads, planes, planes + n_words, planes + 2 * n_words, fa->exotic);
            planes[n_words - 1] = 0; planes[2 * n_words - 1] = 0; planes[3 * n_words - 1] = 0xFFFFFFFFu;
        }
    } catch (const std::bad_alloc &) {
        set_err("crf_fasta_packed: out of host memory");
        return CRF_ERR_NOMEM;
    }
    const uint32_t *planes = (const uint32_t *)fa->planes.p;
    *H = planes; *L = planes + fa->plane_words; *NM = planes + 2 * fa->plane_words;
    *exotic = fa->exotic.data();
    *n_exotic = fa->exotic.size();
    return CRF_OK;
}
