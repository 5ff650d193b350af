// crf_api.cu -- host side of libcrf.so: the C ABI declared in include/crf.h.
//
// Product path only: there is no CPU implementation of the scan in this library; every entry
// point either runs the CUDA kernels or fails with a message.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <mutex>
#include <system_error>
#include <thread>
#include <unordered_map>
#include <utility>
#include <new>
#include <vector>

#include "../../include/crf.h"
#include "crf_aux.cuh"
#include "crf_scan.cuh"
#include "crf_scan_warp.cuh"
#include "crf_stop.cuh"
#include "crf_xchg.cuh"
#include "crf_mask.cuh"

using namespace crf;

// ---- error plumbing -----------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static void set_err(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define CU(call)                                                                       \
    do {                                                                               \
        cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess) {                                                       \
            set_err("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return CRF_ERR_CUDA;                                                       \
        }                                                                              \
    } while (0)

#define CHECK(call)            \
    do {                       \
        int rc_ = (call);      \
        if (rc_) return rc_;   \
    } while (0)

// Device buffers freed by a sequence are kept by its context and handed out again to later loads / scans of
// similar size: cudaMalloc / cudaFree of multi-GB buffers cost tens of milliseconds and made the end-to-end
// path (load -> scan -> fetch -> destroy, every step) erratic.
struct crf_ctx {
    int device;
    cudaStream_t own_stream;
    cudaStream_t stream;
    cudaStream_t copy_stream = nullptr;                 // host -> device chunks of a pipelined upload (load_impl)
    cudaEvent_t copy_done = nullptr;
    std::mutex mu;                                      // guards cache / live (sequences of one context may be destroyed
                                                        // from another thread than the one that is loading)
    std::vector<std::pair<void *, size_t>> cache;       // free blocks
    std::unordered_map<void *, size_t> live;            // blocks handed out -> size
    size_t cached_bytes = 0;
    // timing events and the page-locked counter block are per context, not per load: creating them cost more than a
    // small scan (calls on one context are serialised by the caller, crf.h)
    // (a small pool, handed out round robin: a rank of a multi-GPU job keeps several sequences in flight)
    static const int SLOTS = 8;
    cudaEvent_t ev[SLOTS][5] = {};
    unsigned long long *h_counters = nullptr;           // SLOTS x C_COUNT
    int next_slot = 0;
    int n_xchg = 0;                                     // exchange blocks alive on this context (a rank of a multi-GPU job)
    // per-record tables of the load in progress (source start, length, layout offset, owned range): built in page-locked
    // memory that grows and stays -- a reads file has 10^7 records, and fresh pageable vectors for them cost more in page
    // faults and staged copies than the whole upload.  A load is done with it when it returns (it synchronises the stream).
    void *h_tab = nullptr;
    size_t h_tab_bytes = 0;
    bool h_tab_pinned = false;
};
static void *ctx_tables(crf_ctx *c, size_t bytes) {
    if (bytes <= c->h_tab_bytes) return c->h_tab;
    if (c->h_tab) { if (c->h_tab_pinned) cudaFreeHost(c->h_tab); else free(c->h_tab); }
    c->h_tab = nullptr; c->h_tab_bytes = 0;
    size_t want = (size_t)1 << 16;
    while (want < bytes) want <<= 1;
    void *q = nullptr;
    if (cudaHostAlloc(&q, want, cudaHostAllocDefault) == cudaSuccess) c->h_tab_pinned = true;
    else {                                              // no page-locked memory left: pageable works too, only slower
        cudaGetLastError();
        q = malloc(want);
        c->h_tab_pinned = false;
    }
    if (!q) return nullptr;
    c->h_tab = q; c->h_tab_bytes = want;
    return q;
}
static const size_t CACHE_LIMIT_BYTES = 24ull << 30;
static thread_local crf_ctx *g_ctx = nullptr;          // context of the API call in progress

static cudaError_t ctx_malloc(void **p, size_t bytes) {
    bytes = (std::max<size_t>(bytes, 1) + 511) & ~(size_t)511;
    crf_ctx *c = g_ctx;
    std::unique_lock<std::mutex> lock;
    if (c) lock = std::unique_lock<std::mutex>(c->mu);
    if (c) {
        size_t best = (size_t)-1;
        for (size_t i = 0; i < c->cache.size(); ++i) {
            const size_t sz = c->cache[i].second;
            if (sz >= bytes && sz <= bytes + bytes / 4 + (1u << 20) && (best == (size_t)-1 || sz < c->cache[best].second)) best = i;
        }
        if (best != (size_t)-1) {
            *p = c->cache[best].first;
            c->live[*p] = c->cache[best].second;
            c->cached_bytes -= c->cache[best].second;
            c->cache.erase(c->cache.begin() + best);
            return cudaSuccess;
        }
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess && c && !c->cache.empty()) {   // out of memory: give the cached blocks back and retry
        cudaGetLastError();
        for (auto &b : c->cache) cudaFree(b.first);
        c->cache.clear();
        c->cached_bytes = 0;
        e = cudaMalloc(p, bytes);
    }
    if (e == cudaSuccess && c) c->live[*p] = bytes;
    return e;
}
static void ctx_free(void *p) {
    if (!p) return;
    crf_ctx *c = g_ctx;
    std::unique_lock<std::mutex> lock;
    if (c) lock = std::unique_lock<std::mutex>(c->mu);
    if (c) {
        auto it = c->live.find(p);
        if (it != c->live.end()) {
            const size_t sz = it->second;
            c->live.erase(it);
            if (c->cached_bytes + sz <= CACHE_LIMIT_BYTES && c->cache.size() < 256) {
                c->cache.emplace_back(p, sz);
                c->cached_bytes += sz;
                return;
            }
        }
    }
    cudaFree(p);
}

// Everything one scan launch needs; kept with the sequence so that a second assembly pass (long spill list, more
// open-ended rows than the list held) and the statistics can be produced after the counters have come back.
struct ScanPlan {
    crf_scan_params pr;
    int T;
    int warp_ns;                       // 0: block-tiled scan_kernel; 1 / 2: scan_warp_kernel with that many sub-tiles per warp
    int block_ns;                      // block-tiled kernel: strips per thread (1 or 2)
    uint32_t warp_grid;
    uint32_t n_tiles, outcap, ggrid, tgrid, launches;
    size_t smem;
    bool single_copy;
    GatherParams g;
    TranslateParams tp;
};

struct crf_seq {
    crf_ctx *ctx = nullptr;
    uint32_t n_records = 0;
    uint32_t layout_len = 0, n_words = 0, n_words_alloc = 0, cap = 0;
    uint32_t *H = nullptr, *L = nullptr, *NM = nullptr, *X = nullptr;
    uint32_t *d_rec_dev_off = nullptr, *d_own_lo = nullptr, *d_own_hi = nullptr, *d_rec_len = nullptr;
    uint32_t *d_map_rec = nullptr, *d_map_shift = nullptr;
    uint8_t *d_map_open = nullptr;
    uint32_t *d_open_rows = nullptr;
    std::vector<uint32_t> h_rec_dev_off, h_rec_len;     // host copies of the two tables: see host_tables()
    uint64_t *ex_key = nullptr;
    uint32_t n_exotic = 0, ex_cap = 0;
    // scan scratch
    KEntry *d_ktab = nullptr;
    Seg *d_segs = nullptr;
    uint32_t ktab_cap = 0, segs_cap = 0, n_segs = 0, sup_enabled = 0;
    crf_scan_params ktab_for = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t *stage_key = nullptr, *spill_key = nullptr, *fin_key = nullptr;
    uint16_t *stage_k = nullptr, *spill_k = nullptr, *fin_k = nullptr;
    uint32_t res_cap = 0;
    uint32_t *o_rec = nullptr, *o_start = nullptr, *o_end = nullptr, *o_k = nullptr;
    uint32_t *tile_cnt = nullptr, *tile_base = nullptr, *tile_off = nullptr;
    uint32_t tiles_cap = 0;
    unsigned long long *d_counters = nullptr, *h_counters = nullptr;   // h_counters: the context's page-locked block
    cudaEvent_t *ev = nullptr;                                         // the context's events
    uint32_t open_cap = 0;                                             // rows d_open_rows holds
    cudaGraphExec_t graph_exec = nullptr;                              // the whole scan of a small input, captured once
    struct ScanLaunch *graph_key = nullptr;
    uint32_t graph_launches = 0;
    cudaEvent_t side_done = nullptr;                                   // an exchange stream still reads this sequence's rows
    cudaEvent_t pub_done = nullptr;                                    // ... and this one says it is done with the scan counters
    ScanPlan *plan = nullptr;                                          // launch parameters of the scan in flight / last run
    crf_scan_stats_t stats = {};
    crf_seq_info_t info = {};
    uint64_t n_results = 0;
    bool have_results = false;
};

template <typename T>
static int dev_alloc(T **p, size_t n) {
    *p = nullptr;
    CU(ctx_malloc((void **)p, std::max<size_t>(n, 1) * sizeof(T)));
    return CRF_OK;
}
template <typename T>
static void dev_free(T *&p) {
    if (p) ctx_free(p);
    p = nullptr;
}

extern "C" const char *crf_last_error(void) { return g_err; }
extern "C" int crf_abi_version(void) { return 1; }

// ---- context ------------------------------------------------------------------------------------
// CUDA loads a kernel lazily at its first launch, and that load may wait until the kernels already running on the device
// have finished.  A step of the multi-GPU gather has tiny kernels that wait for peers; a first launch must never queue
// up behind one of them, so every kernel of the library is loaded when a context is created.
template <typename K>
static cudaError_t preload(K kernel) {
    cudaFuncAttributes a;
    return cudaFuncGetAttributes(&a, kernel);
}
static cudaError_t preload_kernels();

extern "C" int crf_ctx_create(int device, crf_ctx **out) {
    if (!out) { set_err("crf_ctx_create: null out pointer"); return CRF_ERR_ARG; }
    *out = nullptr;
    int n = 0;
    CU(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) { set_err("crf_ctx_create: device %d not in [0, %d)", device, n); return CRF_ERR_ARG; }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_err("crf_ctx_create: libcrf is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
        return CRF_ERR_UNSUPPORTED;
    }
    crf_ctx *c = new (std::nothrow) crf_ctx;
    if (!c) { set_err("out of host memory"); return CRF_ERR_NOMEM; }
    c->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->copy_done, cudaEventDisableTiming);
    for (auto &set : c->ev)
        for (auto &ev : set)
            if (e == cudaSuccess) e = cudaEventCreate(&ev);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&c->h_counters, crf_ctx::SLOTS * C_COUNT * sizeof(unsigned long long));
    if (e == cudaSuccess) e = preload_kernels();
    if (e != cudaSuccess) { delete c; set_err("cudaStreamCreate failed: %s", cudaGetErrorString(e)); return CRF_ERR_CUDA; }
    c->stream = c->own_stream;
    *out = c;
    return CRF_OK;
}

extern "C" int crf_ctx_destroy(crf_ctx *c) {
    if (!c) return CRF_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto &b : c->cache) cudaFree(b.first);
    if (g_ctx == c) g_ctx = nullptr;
    cudaStreamDestroy(c->own_stream);
    cudaStreamDestroy(c->copy_stream);
    cudaEventDestroy(c->copy_done);
    for (auto &set : c->ev)
        for (auto &ev : set)
            if (ev) cudaEventDestroy(ev);
    if (c->h_counters) cudaFreeHost(c->h_counters);
    if (c->h_tab) { if (c->h_tab_pinned) cudaFreeHost(c->h_tab); else free(c->h_tab); }
    delete c;
    return CRF_OK;
}

extern "C" int crf_ctx_set_stream(crf_ctx *c, void *stream) {
    if (!c) { set_err("null context"); return CRF_ERR_ARG; }
    cudaStream_t next = stream ? (cudaStream_t)stream : c->own_stream;
    if (next != c->stream) {                            // cached device blocks are handed out again without stream ordering:
        CU(cudaSetDevice(c->device));                   // whatever the old stream still does with them finishes first
        CU(cudaStreamSynchronize(c->stream));
    }
    c->stream = next;
    return CRF_OK;
}

extern "C" int crf_ctx_synchronize(crf_ctx *c) {
    if (!c) { set_err("null context"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return CRF_OK;
}

// ---- fallback sort (global bitonic network) -------------------------------------------------
static uint32_t next_pow2(uint32_t n) {
    uint32_t p = 1;
    while (p < n) p <<= 1;
    return p;
}

// sorts key[0..n) (and val) ascending; the arrays must have room for next_pow2(n) elements
static int bitonic_sort(cudaStream_t st, uint64_t *key, uint16_t *val, uint32_t n, uint32_t *launches) {
    if (n < 2) return CRF_OK;
    const uint32_t np = next_pow2(n);
    if (np > n) {
        fill_u64_kernel<<<(np - n + 255) / 256, 256, 0, st>>>(key, ~0ull, n, np);
        if (val) CU(cudaMemsetAsync(val + n, 0xFF, (size_t)(np - n) * 2, st));
        if (launches) ++*launches;
    }
    for (uint32_t kk = 2; kk <= np; kk <<= 1)
        for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
            bitonic_step_kernel<<<(np + 255) / 256, 256, 0, st>>>(key, val, np, j, kk);
            if (launches) ++*launches;
        }
    CU(cudaGetLastError());
    return CRF_OK;
}

// ---- sequence upload ------------------------------------------------------------------------
static void free_graph_key(struct ScanLaunch *k);
static void free_seq(crf_seq *s) {
    if (!s) return;
    if (s->ctx) { cudaSetDevice(s->ctx->device); g_ctx = s->ctx; }
    dev_free(s->H); dev_free(s->L); dev_free(s->NM); dev_free(s->X);
    dev_free(s->d_rec_dev_off); dev_free(s->d_own_lo); dev_free(s->d_own_hi); dev_free(s->d_rec_len);
    dev_free(s->d_map_rec); dev_free(s->d_map_shift); dev_free(s->d_map_open); dev_free(s->d_open_rows); dev_free(s->ex_key); dev_free(s->d_ktab); dev_free(s->d_segs);
    dev_free(s->stage_key); dev_free(s->spill_key); dev_free(s->fin_key);
    dev_free(s->stage_k); dev_free(s->spill_k); dev_free(s->fin_k);
    dev_free(s->o_rec); dev_free(s->o_start); dev_free(s->o_end); dev_free(s->o_k);
    dev_free(s->tile_cnt); dev_free(s->tile_base); dev_free(s->tile_off);
    dev_free(s->d_counters);
    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
    free_graph_key(s->graph_key);
    delete s->plan;
    delete s;
}

#ifndef CRF_DEFAULT_KERNEL
#define CRF_DEFAULT_KERNEL 0           // scan kernel used when neither a flag nor CRF_SCAN_KERNEL says otherwise:
#endif                                 // 0 block-tiled, 1 / 2 warp-tiled (1 / 2 sub-tiles), 3 block-tiled with 2 strips per thread
static const uint32_t EX_CAP = 1u << 22;       // exotic symbols kept per load
static const uint32_t HOST_TABLES_EAGER = 1u << 16;   // record counts up to this keep host copies of their tables from the load on
static const uint32_t TILE_WORDS_MAX = 4096;   // THREADS * 16
static const uint32_t MAX_K = 65535;

static uint64_t layout_limit(uint32_t max_motif_cap) {
    return 0xFFFFFFFFull - 32ull * (2ull * TILE_WORDS_MAX + (max_motif_cap >> 5) + 64);
}
// One load holds at most this many layout positions: sum over records of (length + max_motif_cap).
extern "C" uint64_t crf_load_limit(uint32_t max_motif_cap) { return layout_limit(max_motif_cap); }

// What a load reads: ASCII bytes (one per base), planes packed on the host (crf_pack_ascii), the bytes of a .2bit file, or
// the 4-bit codes of BAM reads.
struct LoadSource {
    const uint8_t *bases = nullptr;                     // ASCII
    const uint32_t *pH = nullptr, *pL = nullptr, *pN = nullptr;   // packed: source position p = bit p & 31 of word p >> 5
    const uint64_t *exotic = nullptr;                   // packed: (source position << 8 | upper-cased byte), ascending
    uint64_t n_exotic = 0;
    const uint64_t *nm_runs = nullptr;                  // packed, instead of pN: the masked positions as sorted runs
    uint64_t n_runs = 0;                                //   [runs[2i], runs[2i+1]) -- 0.25 B/bp cross PCIe instead of 0.375
    bool runs_mode = false;
    const uint8_t *codes = nullptr;                     // .2bit (code_bits 2, runs mode) or BAM (4) codes, crf_codes.h: source
    uint32_t code_bits = 0;                             //   position p = code p % (8 / code_bits) of byte p / (8 / code_bits)
    bool packed() const { return pH != nullptr || codes != nullptr; }
};

// The two passes over the per-record arrays of a load run on a few threads when there are millions of records.
static const uint32_t TABLE_SEGS = 8;
template <class F>
static void for_record_segments(uint32_t n_records, F fn) {               // fn(segment, first, last)
    if (n_records < (1u << 20)) { fn(0u, 0u, n_records); return; }
    std::thread th[TABLE_SEGS];
    for (uint32_t g = 0; g < TABLE_SEGS; ++g) {
        const uint32_t lo = (uint32_t)((uint64_t)n_records * g / TABLE_SEGS), hi = (uint32_t)((uint64_t)n_records * (g + 1) / TABLE_SEGS);
        try {
            th[g] = std::thread([=]() { fn(g, lo, hi); });
        } catch (...) {                                                   // no thread to be had: do the segment here
            fn(g, lo, hi);
        }
    }
    for (auto &t : th)
        if (t.joinable()) t.join();
}

// CRF_LOAD_TRACE=1: host-side stage times of a load on stderr (where does a 10 M-record load spend its time)
struct LoadTrace {
    bool on = getenv("CRF_LOAD_TRACE") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now(), last = t0;
    void mark(const char *what) {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[crf load] %-28s %8.3f ms (at %8.3f)\n", what, std::chrono::duration<double, std::milli>(now - last).count(),
                std::chrono::duration<double, std::milli>(now - t0).count());
        last = now;
    }
};

static int load_impl(crf_ctx *c, const LoadSource &src, const uint64_t *starts, const uint64_t *lengths,
                     const uint64_t *own_lo, const uint64_t *own_hi, uint32_t n_records, uint32_t max_motif_cap,
                     int on_device, crf_seq *s) {
    const char *who = src.code_bits == 2 ? "crf_seq_load_2bit" : src.code_bits == 4 ? "crf_seq_load_nibbles"
                    : src.packed() ? "crf_seq_load_packed" : "crf_seq_load_ascii";
    LoadTrace trace;
    cudaStream_t st = c->stream;
    s->ctx = c;
    s->n_records = n_records;
    s->cap = max_motif_cap;
    {
        std::lock_guard<std::mutex> lock(c->mu);
        const int slot = c->next_slot++ % crf_ctx::SLOTS;
        s->ev = c->ev[slot];
        s->h_counters = c->h_counters + (size_t)slot * C_COUNT;
    }
    CHECK(dev_alloc(&s->d_counters, C_COUNT));
    s->open_cap = OPEN_CAP_INITIAL;
    CHECK(dev_alloc(&s->d_open_rows, 5 * (size_t)s->open_cap));
    trace.mark("slot + small allocs");

    // layout: record r at dev_off[r], followed by a gap of max_motif_cap masked positions.
    // `lengths` may be null: `starts` is then n_records + 1 boundaries (record r = [starts[r], starts[r + 1])).
    // Pass 1 reads the caller's arrays only: checks, the extent of the source, the size of the layout.
    auto len_of = [&](uint32_t r) -> uint64_t { return lengths ? lengths[r] : starts[r + 1] - starts[r]; };
    const bool owned = own_lo && own_hi;
    const uint64_t limit = layout_limit(max_motif_cap);
    struct SegSum {
        uint64_t pos = 0, total = 0, src_lo = ~0ull, src_hi = 0, first_end = 0, last_end = 0;
        bool ends_sorted = true, too_long = false;
        uint32_t bad_offsets = 0xFFFFFFFFu, bad_own = 0xFFFFFFFFu;           // first offending record, if any
    } seg[TABLE_SEGS];
    for_record_segments(n_records, [&](uint32_t g, uint32_t first, uint32_t last) {
        SegSum q;
        uint64_t prev_end = 0;
        for (uint32_t r = first; r < last; ++r) {
            if (!lengths && starts[r + 1] < starts[r]) { q.bad_offsets = std::min(q.bad_offsets, r); continue; }
            const uint64_t len = len_of(r);
            if (len > limit) { q.too_long = true; continue; }
            if (owned && (own_lo[r] > own_hi[r] || own_hi[r] > len)) q.bad_own = std::min(q.bad_own, r);
            q.pos += len + max_motif_cap;
            q.total += len;
            const uint64_t end = starts[r] + len;
            if (r == first) q.first_end = end;
            else q.ends_sorted &= end >= prev_end;
            prev_end = end;
            if (len) {
                q.src_lo = std::min(q.src_lo, starts[r]);
                q.src_hi = std::max(q.src_hi, end);
            }
        }
        q.last_end = prev_end;
        seg[g] = q;
    });
    uint64_t pos = 0, total = 0, src_lo = ~0ull, src_hi = 0;
    uint64_t seg_pos[TABLE_SEGS];                                        // layout position where each segment starts
    bool ends_sorted = true, too_long = false;                           // starts[r] + len non-decreasing in r
    uint32_t bad_offsets = 0xFFFFFFFFu, bad_own = 0xFFFFFFFFu;
    const uint32_t n_segs_used = n_records < (1u << 20) ? 1 : TABLE_SEGS;
    for (uint32_t g = 0; g < n_segs_used; ++g) {
        seg_pos[g] = pos;
        pos += seg[g].pos; total += seg[g].total;
        src_lo = std::min(src_lo, seg[g].src_lo); src_hi = std::max(src_hi, seg[g].src_hi);
        ends_sorted &= seg[g].ends_sorted && (g == 0 || seg[g].first_end >= seg[g - 1].last_end);
        too_long |= seg[g].too_long;
        bad_offsets = std::min(bad_offsets, seg[g].bad_offsets); bad_own = std::min(bad_own, seg[g].bad_own);
    }
    if (bad_offsets != 0xFFFFFFFFu) { set_err("%s: offsets must be non-decreasing", who); return CRF_ERR_ARG; }
    if (too_long) pos = limit + 1;
    if (pos <= limit && bad_own != 0xFFFFFFFFu) {
        set_err("%s_ranges: own range of record %u is not inside the record", who, bad_own);
        return CRF_ERR_ARG;
    }
    if (pos > limit) {
        set_err("%s: the records need more than %llu layout positions (per-load limit, crf_load_limit); split them "
                "over several loads", who, (unsigned long long)limit);
        return CRF_ERR_UNSUPPORTED;
    }
    if (src_lo > src_hi) src_lo = src_hi = 0;
    trace.mark("layout loop");
    s->layout_len = (uint32_t)pos;
    s->n_words = (s->layout_len + 31) / 32;
    s->n_words_alloc = (s->n_words + TILE_WORDS_MAX - 1) / TILE_WORDS_MAX * TILE_WORDS_MAX + (max_motif_cap >> 5) + 16;

    CU(cudaEventRecord(s->ev[0], st));
    // The source span the records cover (units may overlap) goes up in chunks on a second stream while the pack kernel
    // works on the layout words whose source has already arrived (the PCIe copy is ~10x longer than the packing, which
    // then hides behind it).  Unit of the span: bytes (ASCII) or positions rounded out to whole 32-bit words (packed).
    const bool packed = src.packed(), twobit = src.code_bits == 2, nibbles = src.code_bits == 4;
    const uint64_t src_end = src_hi;                                     // .2bit / BAM: bytes up to (src_end + 3) / 4 or
                                                                         // (src_end + 1) / 2 are the caller's
    if (packed) { src_lo &= ~31ull; src_hi = (src_hi + 31) & ~31ull; }
    const uint64_t span = src_hi - src_lo;                               // positions
    const uint64_t UPLOAD_CHUNK = nibbles ? (128ull << 20) : packed ? (512ull << 20) : (64ull << 20);   // positions per chunk
                                                                                                   // (64 MB of planes, bytes or codes)
    const bool pipelined = !on_device && span > 2 * UPLOAD_CHUNK;
    const uint8_t *d_src = src.bases;                                    // device views of the source
    const uint32_t *d_pH = src.pH, *d_pL = src.pL, *d_pN = src.pN;
    uint64_t src_base = 0;                                               // source position of the device view's first element
    uint8_t *d_src_own = nullptr;
    uint32_t *d_planes_own = nullptr;                                    // 3 x (span / 32 + 1) words
    uint32_t *d_mask_own = nullptr;                                      // runs mode with planes on the device: the mask plane
    uint64_t *d_runs = nullptr;
    uint64_t *d_src_start = nullptr;
    const uint64_t span_words = span / 32 + 1;                           // + 1: repack_kernel reads word wi + 1
    const bool runs_mode = packed && src.runs_mode;
    if (!on_device) {
        if (packed) {
            CHECK(dev_alloc(&d_planes_own, (nibbles ? 4 : 3) * (size_t)span_words));
            d_pH = d_planes_own; d_pL = d_planes_own + span_words; d_pN = d_planes_own + 2 * span_words;
        } else {
            CHECK(dev_alloc(&d_src_own, (size_t)span));
            d_src = d_src_own;
        }
        src_base = src_lo;
    } else if (runs_mode) {                                              // H, L stay where they are; the mask is built here
        CHECK(dev_alloc(&d_mask_own, (size_t)((src_hi + 31) / 32 + 1)));
        d_pN = d_mask_own;
    }
    // runs mode: the mask plane of the span is rebuilt on the device from the (few) runs that touch it
    uint64_t run_first = 0, run_last = 0;                                // runs [run_first, run_last) of the caller's list
    const uint64_t run_lo = on_device ? 0 : src_lo, run_hi = src_hi;
    if (runs_mode) {
        const uint64_t *rb = src.nm_runs, nr = src.n_runs;
        uint64_t a = 0, b = nr;                                          // first run that ends after run_lo
        while (a < b) { const uint64_t m = (a + b) / 2; if (rb[2 * m + 1] <= run_lo) a = m + 1; else b = m; }
        run_first = a;
        b = nr;                                                          // first run that starts at or after run_hi
        while (a < b) { const uint64_t m = (a + b) / 2; if (rb[2 * m] < run_hi) a = m + 1; else b = m; }
        run_last = a;
    }
    const uint64_t n_runs_rel = run_last - run_first;
    if (n_runs_rel > 0xFFFFFF00ull) {                                    // mask_runs_kernel takes a 32-bit run count
        if (d_planes_own) ctx_free(d_planes_own);
        if (d_src_own) ctx_free(d_src_own);
        if (d_mask_own) ctx_free(d_mask_own);
        set_err("%s: more than 2^32 masked runs in one load", who);
        return CRF_ERR_UNSUPPORTED;
    }
    trace.mark("source allocs + runs_rel");
    auto copy_span = [&](uint64_t lo, uint64_t n, cudaStream_t cs) -> cudaError_t {    // source positions [src_lo + lo, + n)
        if (!n) return cudaSuccess;
        if (src.codes) {                                                 // (lo is a multiple of 32: whole bytes)
            const uint64_t per = 8 / src.code_bits;
            const uint64_t b0 = (src_lo + lo) / per, b1 = std::min((src_lo + lo + n + per - 1) / per, (src_end + per - 1) / per);
            if (b1 <= b0) return cudaSuccess;
            return cudaMemcpyAsync((uint8_t *)d_planes_own + lo / per, src.codes + b0, b1 - b0, cudaMemcpyHostToDevice, cs);
        }
        if (!packed) return cudaMemcpyAsync(d_src_own + lo, src.bases + src_lo + lo, n, cudaMemcpyHostToDevice, cs);
        const uint64_t w0 = lo / 32, nw = (n + 31) / 32, h0 = src_lo / 32 + w0;
        cudaError_t e = cudaMemcpyAsync(d_planes_own + w0, src.pH + h0, nw * 4, cudaMemcpyHostToDevice, cs);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_planes_own + span_words + w0, src.pL + h0, nw * 4, cudaMemcpyHostToDevice, cs);
        if (e == cudaSuccess && !runs_mode)
            e = cudaMemcpyAsync(d_planes_own + 2 * span_words + w0, src.pN + h0, nw * 4, cudaMemcpyHostToDevice, cs);
        return e;
    };
    auto free_sources = [&]() {
        if (d_src_own) ctx_free(d_src_own);
        if (d_planes_own) ctx_free(d_planes_own);
        if (d_mask_own) ctx_free(d_mask_own);
        if (d_runs) ctx_free(d_runs);
        if (d_src_start) ctx_free(d_src_start);
        d_src_own = nullptr; d_planes_own = nullptr; d_mask_own = nullptr; d_runs = nullptr; d_src_start = nullptr;
    };
    // Pass 2 fills the tables the kernels read, in the context's page-locked arena: source start relative to the device view,
    // length, layout offset, owned range in layout positions
    const size_t n8 = ((size_t)n_records * 4 + 7) & ~(size_t)7;           // bytes of one 32-bit table, 8-byte aligned
    const size_t tab_bytes = (size_t)n_records * 8 + (owned ? 4 : 2) * n8;
    uint8_t *tab = (uint8_t *)ctx_tables(c, tab_bytes + (size_t)n_runs_rel * 16);
    if (!tab) { free_sources(); set_err("out of host memory"); return CRF_ERR_NOMEM; }
    uint64_t *rel = (uint64_t *)tab;
    uint32_t *len32 = (uint32_t *)(tab + (size_t)n_records * 8), *dev_off = (uint32_t *)((uint8_t *)len32 + n8);
    uint32_t *olo = owned ? (uint32_t *)((uint8_t *)dev_off + n8) : nullptr, *ohi = owned ? (uint32_t *)((uint8_t *)olo + n8) : nullptr;
    uint64_t *runs_rel = (uint64_t *)(tab + tab_bytes);                  // the mask runs that touch the span, relative to it
    for_record_segments(n_records, [&](uint32_t g, uint32_t first, uint32_t last) {
        const uint64_t view = packed ? 0 : src_base;
        uint64_t at = seg_pos[g];
        for (uint32_t r = first; r < last; ++r) {
            const uint64_t len = len_of(r);
            rel[r] = len ? starts[r] - view : 0;
            len32[r] = (uint32_t)len;
            dev_off[r] = (uint32_t)at;
            if (owned) { olo[r] = (uint32_t)(at + own_lo[r]); ohi[r] = (uint32_t)(at + own_hi[r]); }
            at += len + max_motif_cap;
        }
    });
    for (uint64_t i = 0; i < n_runs_rel; ++i) {
        const uint64_t *rb = src.nm_runs + 2 * (run_first + i);
        runs_rel[2 * i] = std::max(rb[0], run_lo) - run_lo;
        runs_rel[2 * i + 1] = std::min(rb[1], run_hi) - run_lo;
    }
    // host copies for crf_run_end / crf_seq_set_output_map: now for an ordinary record count, on first use for millions
    if (n_records <= HOST_TABLES_EAGER) {
        s->h_rec_dev_off.assign(dev_off, dev_off + n_records);
        s->h_rec_len.assign(len32, len32 + n_records);
    }
    trace.mark("rel + own tables");
    // exotic symbols of a packed source: source positions -> layout positions (a symbol in the halo two units share
    // appears once per unit); records in ascending source order are walked with one cursor
    std::vector<uint64_t> ex_layout;
    if (packed && src.n_exotic) {
        const uint64_t *ex = src.exotic, ne = src.n_exotic;
        uint64_t cur = 0, prev_start = 0;
        for (uint32_t r = 0; r < n_records; ++r) {
            const uint64_t a = starts[r], b = a + len32[r];
            if (a == b) continue;
            if (a < prev_start || (cur < ne && a > (ex[cur] >> 8) + (1u << 16)))
                cur = (uint64_t)(std::lower_bound(ex, ex + ne, a << 8) - ex);   // out of order, or far ahead: bisect
            while (cur < ne && (ex[cur] >> 8) < a) ++cur;
            prev_start = a;
            for (uint64_t i = cur; i < ne && (ex[i] >> 8) < b; ++i)
                ex_layout.push_back((((ex[i] >> 8) - a + dev_off[r]) << 8) | (ex[i] & 0xFF));
        }
        std::sort(ex_layout.begin(), ex_layout.end());
    }
    trace.mark("exotic layout");
    int rc = dev_alloc(&d_src_start, n_records);
    if (!rc) rc = dev_alloc(&s->d_rec_len, n_records);
    if (!rc) rc = dev_alloc(&s->d_rec_dev_off, n_records);
    if (!rc && owned) rc = dev_alloc(&s->d_own_lo, n_records);
    if (!rc && owned) rc = dev_alloc(&s->d_own_hi, n_records);
    if (!rc) rc = dev_alloc(&s->H, s->n_words_alloc);
    if (!rc) rc = dev_alloc(&s->L, s->n_words_alloc);
    if (!rc) rc = dev_alloc(&s->NM, s->n_words_alloc);
    if (!rc) rc = dev_alloc(&s->X, s->n_words_alloc);
    if (packed) s->ex_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(ex_layout.size(), 16), 0xFFFFFFFFull);
    else s->ex_cap = std::min<uint32_t>(EX_CAP, next_pow2((uint32_t)std::min<uint64_t>(std::max<uint64_t>(total, 16), EX_CAP)));
    if (!rc) rc = dev_alloc(&s->ex_key, s->ex_cap);
    cudaError_t e = cudaSuccess;
    trace.mark("device allocs");
    if (!rc) {
        const size_t n4 = (size_t)n_records * 4;
        e = cudaMemcpyAsync(d_src_start, rel, (size_t)n_records * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(s->d_rec_len, len32, n4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(s->d_rec_dev_off, dev_off, n4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess && owned) e = cudaMemcpyAsync(s->d_own_lo, olo, n4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess && owned) e = cudaMemcpyAsync(s->d_own_hi, ohi, n4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(s->d_counters, 0, C_COUNT * sizeof(unsigned long long), st);
        if (e == cudaSuccess && !ex_layout.empty())
            e = cudaMemcpyAsync(s->ex_key, ex_layout.data(), ex_layout.size() * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess && runs_mode) {                             // mask plane of the span: zero, then the runs
            const size_t mask_words = on_device ? (size_t)((src_hi + 31) / 32 + 1) : (size_t)span_words;
            e = cudaMemsetAsync(const_cast<uint32_t *>(d_pN), 0, mask_words * 4, st);
            const uint32_t nr = (uint32_t)n_runs_rel;
            if (e == cudaSuccess && nr) {
                rc = dev_alloc(&d_runs, (size_t)n_runs_rel * 2);
                if (!rc) e = cudaMemcpyAsync(d_runs, runs_rel, (size_t)n_runs_rel * 16, cudaMemcpyHostToDevice, st);
                if (!rc && e == cudaSuccess) {
                    mask_runs_kernel<<<(nr + 7) / 8, 256, 0, st>>>(d_runs, nr, const_cast<uint32_t *>(d_pN));
                    e = cudaGetLastError();
                }
            }
        }
    }
    trace.mark("table uploads queued");
    // one launch of the packer over layout words [w_lo, w_hi)
    auto launch_pack = [&](uint32_t w_lo, uint32_t w_hi) -> cudaError_t {
        if (w_hi <= w_lo) return cudaSuccess;
        if (twobit) {
            TwoBitParams tp;
            tp.dna = on_device ? src.codes : (const uint8_t *)d_planes_own;
            tp.n_bytes = (src_end + 3) / 4 - (on_device ? 0 : src_lo / 4);
            tp.sN = d_pN; tp.src_base = src_base;
            tp.rec_src_start = d_src_start; tp.rec_len = s->d_rec_len; tp.rec_dev_off = s->d_rec_dev_off;
            tp.n_records = n_records; tp.w_lo = w_lo; tp.w_hi = w_hi;
            tp.H = s->H; tp.L = s->L; tp.NM = s->NM; tp.X = s->X;
            twobit_pack_kernel<<<(w_hi - w_lo + 255) / 256, 256, 0, st>>>(tp);
        } else if (nibbles) {
            NibbleParams np;
            np.nib = on_device ? src.codes : (const uint8_t *)d_planes_own;
            np.n_bytes = (src_end + 1) / 2 - (on_device ? 0 : src_lo / 2);
            np.src_base = src_base;
            np.rec_src_start = d_src_start; np.rec_len = s->d_rec_len; np.rec_dev_off = s->d_rec_dev_off;
            np.n_records = n_records; np.w_lo = w_lo; np.w_hi = w_hi;
            np.H = s->H; np.L = s->L; np.NM = s->NM; np.X = s->X;
            nibble_pack_kernel<<<(w_hi - w_lo + 255) / 256, 256, 0, st>>>(np);
        } else if (packed) {
            RepackParams rp;
            rp.sH = d_pH; rp.sL = d_pL; rp.sN = d_pN; rp.src_base = src_base;
            rp.rec_src_start = d_src_start; rp.rec_len = s->d_rec_len; rp.rec_dev_off = s->d_rec_dev_off;
            rp.n_records = n_records; rp.w_lo = w_lo; rp.w_hi = w_hi;
            rp.H = s->H; rp.L = s->L; rp.NM = s->NM; rp.X = s->X;
            repack_kernel<<<(w_hi - w_lo + 255) / 256, 256, 0, st>>>(rp);
        } else {
            PackParams pp;
            pp.src = d_src; pp.rec_src_start = d_src_start; pp.rec_len = s->d_rec_len; pp.rec_dev_off = s->d_rec_dev_off;
            pp.n_records = n_records;
            pp.H = s->H; pp.L = s->L; pp.NM = s->NM; pp.X = s->X;
            pp.ex_key = s->ex_key; pp.ex_cap = s->ex_cap; pp.ex_count = s->d_counters;
            pp.w_lo = w_lo; pp.w_hi = w_hi;
            pack_kernel<<<(w_hi - w_lo + 255) / 256, 256, 0, st>>>(pp);
        }
        return cudaGetLastError();
    };
    if (!rc && e == cudaSuccess) {
        if (!pipelined) {
            if (!on_device) e = copy_span(0, span, st);
            if (e == cudaSuccess) e = launch_pack(0, s->n_words_alloc);
        } else {
            // "The first record whose source is not all there" bounds the layout words that can be packed.  Records usually end
            // in ascending source order (FASTA records, reads, units with halo): bisect their ends where they lie.  Otherwise
            // src_end[r] = running maximum of where records 0..r end in the source, whatever order they come in.
            std::vector<uint64_t> src_end;
            if (!ends_sorted) {
                src_end.resize(n_records);
                uint64_t run = 0;
                for (uint32_t r = 0; r < n_records; ++r) {
                    if (len32[r]) run = std::max(run, starts[r] - src_lo + len32[r]);
                    src_end[r] = run;
                }
            }
            auto first_incomplete = [&](uint64_t avail) -> uint32_t {     // first r whose source ends beyond src_lo + avail
                if (!ends_sorted) return (uint32_t)(std::upper_bound(src_end.begin(), src_end.end(), avail) - src_end.begin());
                uint32_t lo = 0, hi = n_records;
                while (lo < hi) {
                    const uint32_t mid = lo + (hi - lo) / 2;
                    if (starts[mid] + len32[mid] > src_lo + avail) hi = mid; else lo = mid + 1;
                }
                return lo;
            };
            e = cudaEventRecord(c->copy_done, st);                       // the copies start after what is queued on st
            if (e == cudaSuccess) e = cudaStreamWaitEvent(c->copy_stream, c->copy_done, 0);
            uint32_t w_done = 0;
            for (uint64_t b = 0; b < span && e == cudaSuccess; b += UPLOAD_CHUNK) {
                const uint64_t nb = std::min(UPLOAD_CHUNK, span - b), avail = b + nb;
                e = copy_span(b, nb, c->copy_stream);
                if (e == cudaSuccess) e = cudaEventRecord(c->copy_done, c->copy_stream);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(st, c->copy_done, 0);
                if (e != cudaSuccess) break;
                uint32_t w_hi = s->n_words_alloc;
                if (avail < span) {
                    const uint32_t r = first_incomplete(avail);
                    if (r < n_records) {
                        const uint64_t r0 = starts[r] - src_lo;
                        const uint64_t have = avail > r0 ? std::min<uint64_t>(avail - r0, len32[r]) : 0;
                        w_hi = (uint32_t)((dev_off[r] + have) >> 5);
                    }
                }
                if (w_hi > w_done) {
                    e = launch_pack(w_done, w_hi);
                    w_done = w_hi;
                }
            }
            if (e != cudaSuccess) cudaStreamSynchronize(c->copy_stream);   // nothing may still write the buffer freed below
        }
        if (e == cudaSuccess && packed && !ex_layout.empty()) {
            exotic_apply_kernel<<<((uint32_t)ex_layout.size() + 255) / 256, 256, 0, st>>>(s->ex_key, (uint32_t)ex_layout.size(),
                                                                                          s->H, s->L, s->X);
            e = cudaGetLastError();
        }
        trace.mark("copies + pack queued");
        if (e == cudaSuccess) e = cudaMemcpyAsync(s->h_counters, s->d_counters, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);   // also keeps rel/len32/olo/ex_layout alive long enough
        trace.mark("stream synchronised");
    }
    if (rc) { free_sources(); return rc; }
    if (e != cudaSuccess) { free_sources(); set_err("%s: %s", who, cudaGetErrorString(e)); return CRF_ERR_CUDA; }

    unsigned long long nex = packed ? ex_layout.size() : s->h_counters[0];
    if (!packed && nex > s->ex_cap) {
        // more symbols other than A,C,G,T,N than the list held: size it to the count and pack once more (the source is
        // still on the device)
        if (nex > 0x7FFFFFFFull) { free_sources(); set_err("%s: more than 2^31 symbols other than A,C,G,T,N", who); return CRF_ERR_UNSUPPORTED; }
        dev_free(s->ex_key);
        s->ex_cap = next_pow2((uint32_t)nex);
        rc = dev_alloc(&s->ex_key, s->ex_cap);
        if (!rc) {
            e = cudaMemsetAsync(s->d_counters, 0, sizeof(unsigned long long), st);
            if (e == cudaSuccess) e = launch_pack(0, s->n_words_alloc);
            if (e == cudaSuccess) e = cudaMemcpyAsync(s->h_counters, s->d_counters, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        }
        if (rc) { free_sources(); return rc; }
        if (e != cudaSuccess) { free_sources(); set_err("%s: %s", who, cudaGetErrorString(e)); return CRF_ERR_CUDA; }
        nex = s->h_counters[0];
    }
    free_sources();
    s->n_exotic = (uint32_t)nex;
    if (!packed && s->n_exotic > 1) CHECK(bitonic_sort(st, s->ex_key, nullptr, s->n_exotic, nullptr));
    CU(cudaEventRecord(s->ev[1], st));
    CU(cudaStreamSynchronize(st));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, s->ev[0], s->ev[1]));

    s->info.n_records = n_records;
    s->info.total_bases = total;
    s->info.layout_bases = s->layout_len;
    s->info.packed_bytes = (uint64_t)((total + 3) / 4) + (total + 7) / 8;
    s->info.n_exotic = s->n_exotic;
    s->info.max_motif_cap = max_motif_cap;
    s->info.load_ms = ms;
    trace.mark("done");
    return CRF_OK;
}

// Host copies of the layout offset and length tables (crf_run_end, crf_seq_set_output_map): filled by the load for an ordinary
// record count, read back from the device on first use when there are millions of records.
static int host_tables(crf_seq *s) {
    if (s->h_rec_dev_off.size() == s->n_records && s->h_rec_len.size() == s->n_records) return CRF_OK;
    try {
        s->h_rec_dev_off.resize(s->n_records);
        s->h_rec_len.resize(s->n_records);
    } catch (const std::bad_alloc &) { set_err("out of host memory"); return CRF_ERR_NOMEM; }
    CU(cudaMemcpy(s->h_rec_dev_off.data(), s->d_rec_dev_off, (size_t)s->n_records * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(s->h_rec_len.data(), s->d_rec_len, (size_t)s->n_records * 4, cudaMemcpyDeviceToHost));
    return CRF_OK;
}

static int load_checked(crf_ctx *c, const LoadSource &src, const uint64_t *starts, const uint64_t *lengths,
                        const uint64_t *own_lo, const uint64_t *own_hi, uint32_t n_records, uint32_t max_motif_cap,
                        int on_device, crf_seq **out, const char *who) {
    if (!c || !out || !starts) { set_err("%s: null argument", who); return CRF_ERR_ARG; }   // lengths == null: starts are boundaries
    *out = nullptr;
    if (n_records == 0) { set_err("%s: n_records must be >= 1", who); return CRF_ERR_ARG; }
    if ((own_lo == nullptr) != (own_hi == nullptr)) { set_err("%s_ranges: own_lo and own_hi go together", who); return CRF_ERR_ARG; }
    if (max_motif_cap < 1 || max_motif_cap > MAX_K) {
        set_err("%s: max_motif_cap %u not in [1, %u]", who, max_motif_cap, MAX_K);
        return max_motif_cap < 1 ? CRF_ERR_ARG : CRF_ERR_UNSUPPORTED;
    }
    const bool have_src = src.codes ? true : src.packed() ? (src.pL && src.pN) : (src.bases != nullptr);
    if (!have_src) {
        for (uint32_t r = 0; r < n_records; ++r)
            if (lengths ? lengths[r] : starts[r + 1] - starts[r]) { set_err("%s: null %s", who, src.packed() ? "plane" : "bases"); return CRF_ERR_ARG; }
    }
    if (src.n_exotic && !src.exotic) { set_err("%s: null exotic list", who); return CRF_ERR_ARG; }
    CU(cudaSetDevice(c->device));
    g_ctx = c;
    crf_seq *s = new (std::nothrow) crf_seq;
    if (!s) { set_err("out of host memory"); return CRF_ERR_NOMEM; }
    int rc;
    try {
        rc = load_impl(c, src, starts, lengths, own_lo, own_hi, n_records, max_motif_cap, on_device, s);
    } catch (const std::bad_alloc &) {
        set_err("out of host memory");
        rc = CRF_ERR_NOMEM;
    }
    if (rc) { free_seq(s); return rc; }
    *out = s;
    return CRF_OK;
}

// The entry points that take n_records + 1 boundaries hand them to load_impl as they are (lengths == null): no per-record
// array is built for them on the way.
static int check_offsets(const uint64_t *offsets, uint32_t n_records, const char *who) {
    if (!offsets) { set_err("%s: null argument", who); return CRF_ERR_ARG; }
    if (n_records == 0) { set_err("%s: n_records must be >= 1", who); return CRF_ERR_ARG; }
    return CRF_OK;
}

extern "C" int crf_seq_load_ascii_ranges(crf_ctx *c, const uint8_t *bases, const uint64_t *starts,
                                         const uint64_t *lengths, const uint64_t *own_lo, const uint64_t *own_hi,
                                         uint32_t n_records, uint32_t max_motif_cap, int bases_on_device, crf_seq **out) {
    if (!lengths) { set_err("crf_seq_load_ascii_ranges: null argument"); return CRF_ERR_ARG; }
    LoadSource src;
    src.bases = bases;
    return load_checked(c, src, starts, lengths, own_lo, own_hi, n_records, max_motif_cap, bases_on_device, out, "crf_seq_load_ascii");
}

extern "C" int crf_seq_load_ascii(crf_ctx *c, const uint8_t *bases, const uint64_t *offsets, uint32_t n_records,
                                  uint32_t max_motif_cap, int bases_on_device, crf_seq **out) {
    CHECK(check_offsets(offsets, n_records, "crf_seq_load_ascii"));
    LoadSource src;
    src.bases = bases;
    return load_checked(c, src, offsets, nullptr, nullptr, nullptr, n_records, max_motif_cap, bases_on_device, out, "crf_seq_load_ascii");
}

static int check_runs(const uint64_t *runs, uint64_t n_runs, const char *who) {
    for (uint64_t i = 0; i < n_runs; ++i)
        if (runs[2 * i] >= runs[2 * i + 1] || (i && runs[2 * i] < runs[2 * i - 1])) {
            set_err("%s: runs must be non-empty, ascending and disjoint (run %llu)", who, (unsigned long long)i);
            return CRF_ERR_ARG;
        }
    return CRF_OK;
}

static int packed_load(crf_ctx *c, const uint32_t *H, const uint32_t *L, const uint32_t *NM, const uint64_t *exotic,
                       uint64_t n_exotic, const uint64_t *starts, const uint64_t *lengths, const uint64_t *own_lo,
                       const uint64_t *own_hi, uint32_t n_records, uint32_t max_motif_cap, int planes_on_device, crf_seq **out) {
    if (!H) {
        set_err("crf_seq_load_packed: null plane");
        return CRF_ERR_ARG;
    }
    LoadSource src;
    src.pH = H; src.pL = L; src.pN = NM; src.exotic = exotic; src.n_exotic = n_exotic;
    return load_checked(c, src, starts, lengths, own_lo, own_hi, n_records, max_motif_cap, planes_on_device, out, "crf_seq_load_packed");
}

static int packed_runs_load(crf_ctx *c, const uint32_t *H, const uint32_t *L, const uint64_t *runs, uint64_t n_runs,
                            const uint64_t *exotic, uint64_t n_exotic, const uint64_t *starts, const uint64_t *lengths,
                            const uint64_t *own_lo, const uint64_t *own_hi, uint32_t n_records, uint32_t max_motif_cap,
                            int planes_on_device, crf_seq **out) {
    if (!H || !L) { set_err("crf_seq_load_packed_runs: null plane"); return CRF_ERR_ARG; }
    if (n_runs && !runs) { set_err("crf_seq_load_packed_runs: null run list"); return CRF_ERR_ARG; }
    CHECK(check_runs(runs, n_runs, "crf_seq_load_packed_runs"));
    LoadSource src;
    src.pH = H; src.pL = L; src.pN = H;      // (pN is not read in runs mode; non-null for the argument check)
    src.exotic = exotic; src.n_exotic = n_exotic;
    src.nm_runs = runs; src.n_runs = n_runs; src.runs_mode = true;
    return load_checked(c, src, starts, lengths, own_lo, own_hi, n_records, max_motif_cap, planes_on_device, out, "crf_seq_load_packed_runs");
}

extern "C" int crf_seq_load_packed_ranges(crf_ctx *c, const uint32_t *H, const uint32_t *L, const uint32_t *NM,
                                          const uint64_t *exotic, uint64_t n_exotic, const uint64_t *starts,
                                          const uint64_t *lengths, const uint64_t *own_lo, const uint64_t *own_hi,
                                          uint32_t n_records, uint32_t max_motif_cap, int planes_on_device, crf_seq **out) {
    if (!lengths) { set_err("crf_seq_load_packed_ranges: null argument"); return CRF_ERR_ARG; }
    return packed_load(c, H, L, NM, exotic, n_exotic, starts, lengths, own_lo, own_hi, n_records, max_motif_cap, planes_on_device, out);
}

extern "C" int crf_seq_load_packed_runs_ranges(crf_ctx *c, const uint32_t *H, const uint32_t *L, const uint64_t *runs,
                                               uint64_t n_runs, const uint64_t *exotic, uint64_t n_exotic,
                                               const uint64_t *starts, const uint64_t *lengths, const uint64_t *own_lo,
                                               const uint64_t *own_hi, uint32_t n_records, uint32_t max_motif_cap,
                                               int planes_on_device, crf_seq **out) {
    if (!lengths) { set_err("crf_seq_load_packed_runs_ranges: null argument"); return CRF_ERR_ARG; }
    return packed_runs_load(c, H, L, runs, n_runs, exotic, n_exotic, starts, lengths, own_lo, own_hi, n_records, max_motif_cap,
                            planes_on_device, out);
}

extern "C" int crf_seq_load_packed_runs(crf_ctx *c, const uint32_t *H, const uint32_t *L, const uint64_t *runs, uint64_t n_runs,
                                        const uint64_t *exotic, uint64_t n_exotic, const uint64_t *offsets, uint32_t n_records,
                                        uint32_t max_motif_cap, int planes_on_device, crf_seq **out) {
    CHECK(check_offsets(offsets, n_records, "crf_seq_load_packed_runs"));
    return packed_runs_load(c, H, L, runs, n_runs, exotic, n_exotic, offsets, nullptr, nullptr, nullptr, n_records, max_motif_cap,
                            planes_on_device, out);
}

// What crf_seq_load_2bit and crf_seq_load_nibbles share: the checks, and record r = offsets[r + 1] - offsets[r] bases coded
// from byte rec_byte[r] of src.codes, which the load sees at source position (8 / code_bits) rec_byte[r] (the position of its
// first code in the bytes).  null_list: the entry point's list is missing.
static int code_records(const LoadSource &src, const uint64_t *rec_byte, const uint64_t *offsets, uint32_t n_records,
                        bool null_list, const char *who, std::vector<uint64_t> &starts, std::vector<uint64_t> &lengths) {
    CHECK(check_offsets(offsets, n_records, who));
    if (!src.codes || !rec_byte || null_list) { set_err("%s: null argument", who); return CRF_ERR_ARG; }
    for (uint32_t r = 0; r < n_records; ++r)
        if (offsets[r + 1] < offsets[r]) { set_err("%s: offsets must be non-decreasing", who); return CRF_ERR_ARG; }
    try {
        starts.resize(n_records);
        lengths.resize(n_records);
    } catch (const std::bad_alloc &) {
        set_err("out of host memory");
        return CRF_ERR_NOMEM;
    }
    const uint64_t per_byte = 8 / src.code_bits;
    for (uint32_t r = 0; r < n_records; ++r) {
        starts[r] = per_byte * rec_byte[r];
        lengths[r] = offsets[r + 1] - offsets[r];
    }
    return CRF_OK;
}

// .2bit records (code_records), their N blocks among the runs of offsets' position space: the load sees the runs moved to
// the records' source positions, split at record ends.
extern "C" int crf_seq_load_2bit(crf_ctx *c, const uint8_t *dna, const uint64_t *rec_byte, const uint64_t *offsets,
                                 uint32_t n_records, const uint64_t *runs, uint64_t n_runs, uint32_t max_motif_cap,
                                 int dna_on_device, crf_seq **out) {
    const char *who = "crf_seq_load_2bit";
    LoadSource src;
    src.codes = dna; src.code_bits = 2;
    std::vector<uint64_t> starts, lengths, moved;
    CHECK(code_records(src, rec_byte, offsets, n_records, n_runs && !runs, who, starts, lengths));
    CHECK(check_runs(runs, n_runs, who));
    try {
        const uint64_t pos0 = offsets[0], pos1 = offsets[n_records];
        uint64_t a_i = 0, b_i = n_runs;                                  // first run that ends after pos0
        while (a_i < b_i) { const uint64_t m = (a_i + b_i) / 2; if (runs[2 * m + 1] <= pos0) a_i = m + 1; else b_i = m; }
        bool sorted = true;
        uint32_t r = 0;
        for (uint64_t k = a_i; k < n_runs && runs[2 * k] < pos1; ++k) {
            uint64_t a = std::max(runs[2 * k], pos0);
            const uint64_t b = std::min(runs[2 * k + 1], pos1);
            while (a < b) {
                while (offsets[r + 1] <= a) ++r;
                const uint64_t e = std::min(b, offsets[r + 1]);
                const uint64_t m0 = starts[r] + (a - offsets[r]), m1 = starts[r] + (e - offsets[r]);
                if (!moved.empty() && m0 < moved.back()) sorted = false;
                moved.push_back(m0);
                moved.push_back(m1);
                a = e;
            }
        }
        if (!sorted) {                                                   // records not in file order
            std::vector<std::pair<uint64_t, uint64_t>> pairs(moved.size() / 2);
            for (size_t j = 0; j < pairs.size(); ++j) pairs[j] = {moved[2 * j], moved[2 * j + 1]};
            std::sort(pairs.begin(), pairs.end());
            for (size_t j = 0; j < pairs.size(); ++j) {
                moved[2 * j] = pairs[j].first;
                moved[2 * j + 1] = pairs[j].second;
                if (j && pairs[j].first < pairs[j - 1].second) { set_err("%s: records share bytes of dna", who); return CRF_ERR_ARG; }
            }
        }
    } catch (const std::bad_alloc &) {
        set_err("out of host memory");
        return CRF_ERR_NOMEM;
    }
    src.nm_runs = moved.data(); src.n_runs = moved.size() / 2; src.runs_mode = true;
    return load_checked(c, src, starts.data(), lengths.data(), nullptr, nullptr, n_records, max_motif_cap, dna_on_device, out, who);
}

// BAM reads (code_records), their exotic codes among the list in offsets' position space: the load sees the list moved to
// the records' source positions.
extern "C" int crf_seq_load_nibbles(crf_ctx *c, const uint8_t *nib, const uint64_t *rec_byte, const uint64_t *offsets,
                                    uint32_t n_records, const uint64_t *exotic, uint64_t n_exotic, uint32_t max_motif_cap,
                                    int nib_on_device, crf_seq **out) {
    const char *who = "crf_seq_load_nibbles";
    LoadSource src;
    src.codes = nib; src.code_bits = 4;
    std::vector<uint64_t> starts, lengths, moved;
    CHECK(code_records(src, rec_byte, offsets, n_records, n_exotic && !exotic, who, starts, lengths));
    for (uint64_t i = 1; i < n_exotic; ++i)
        if (exotic[i] >> 8 <= exotic[i - 1] >> 8) { set_err("%s: the exotic list must be ascending (entry %llu)", who, (unsigned long long)i); return CRF_ERR_ARG; }
    try {
        const uint64_t pos0 = offsets[0], pos1 = offsets[n_records];
        const uint64_t *e0 = std::lower_bound(exotic, exotic + n_exotic, pos0 << 8), *e1 = std::lower_bound(e0, exotic + n_exotic, pos1 << 8);
        bool sorted = true;
        uint32_t r = 0;
        for (const uint64_t *e = e0; e < e1; ++e) {
            const uint64_t q = *e >> 8;
            while (offsets[r + 1] <= q) ++r;
            const uint64_t m = ((starts[r] + (q - offsets[r])) << 8) | (*e & 0xFF);
            if (!moved.empty() && m < moved.back()) sorted = false;
            moved.push_back(m);
        }
        if (!sorted) std::sort(moved.begin(), moved.end());            // records not in the order of their bytes
    } catch (const std::bad_alloc &) {
        set_err("out of host memory");
        return CRF_ERR_NOMEM;
    }
    src.exotic = moved.data(); src.n_exotic = moved.size();
    return load_checked(c, src, starts.data(), lengths.data(), nullptr, nullptr, n_records, max_motif_cap, nib_on_device, out, who);
}

extern "C" int crf_seq_load_packed(crf_ctx *c, const uint32_t *H, const uint32_t *L, const uint32_t *NM,
                                   const uint64_t *exotic, uint64_t n_exotic, const uint64_t *offsets, uint32_t n_records,
                                   uint32_t max_motif_cap, int planes_on_device, crf_seq **out) {
    CHECK(check_offsets(offsets, n_records, "crf_seq_load_packed"));
    return packed_load(c, H, L, NM, exotic, n_exotic, offsets, nullptr, nullptr, nullptr, n_records, max_motif_cap, planes_on_device, out);
}

extern "C" int crf_seq_destroy(crf_seq *s) {
    if (!s) return CRF_OK;
    g_ctx = s->ctx;
    cudaSetDevice(s->ctx->device);
    if (s->side_done) cudaEventSynchronize(s->side_done);
    cudaStreamSynchronize(s->ctx->stream);
    free_seq(s);
    return CRF_OK;
}

extern "C" int crf_seq_set_output_map(crf_seq *s, const uint32_t *out_record, const uint64_t *out_shift,
                                      const uint8_t *open_ended) {
    if (!s) { set_err("crf_seq_set_output_map: null sequence"); return CRF_ERR_ARG; }
    g_ctx = s->ctx;
    CU(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    CU(cudaStreamSynchronize(st));
    dev_free(s->d_map_rec); dev_free(s->d_map_shift); dev_free(s->d_map_open);
    const uint32_t n = s->n_records;
    if (out_record) {
        CHECK(dev_alloc(&s->d_map_rec, n));
        CU(cudaMemcpy(s->d_map_rec, out_record, (size_t)n * 4, cudaMemcpyHostToDevice));
    }
    if (out_shift) {
        CHECK(host_tables(s));
        std::vector<uint32_t> sh(n);
        for (uint32_t r = 0; r < n; ++r) {
            if (out_shift[r] > 0xFFFFFFFFull - s->h_rec_len[r]) { set_err("crf_seq_set_output_map: shifted coordinates exceed 32 bits"); return CRF_ERR_UNSUPPORTED; }
            sh[r] = (uint32_t)out_shift[r];
        }
        CHECK(dev_alloc(&s->d_map_shift, n));
        CU(cudaMemcpy(s->d_map_shift, sh.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
    }
    if (open_ended) {
        CHECK(dev_alloc(&s->d_map_open, n));
        CU(cudaMemcpy(s->d_map_open, open_ended, n, cudaMemcpyHostToDevice));
    }
    return CRF_OK;
}

extern "C" int crf_seq_info(const crf_seq *s, crf_seq_info_t *info) {
    if (!s || !info) { set_err("crf_seq_info: null argument"); return CRF_ERR_ARG; }
    *info = s->info;
    return CRF_OK;
}

// ---- scan ---------------------------------------------------------------------------------------
static void build_ktab(const crf_scan_params &pr, bool allow_sup, std::vector<KEntry> &tab, std::vector<Seg> &segs) {
    tab.assign((size_t)pr.max_motif_size + 1, KEntry{});
    for (uint32_t k = 1; k <= pr.max_motif_size; ++k) {
        KEntry &e = tab[k];
        // r_min: trk:86 and trk:91 in closed form (SURVEY Appendix A.2)
        const uint64_t a = pr.min_span > k ? (uint64_t)pr.min_span - k : 0;
        // min_repeats == 1: a shorter run cannot fill its own motif (Appendix A.4 reduces to r >= k-1 away from position 0)
        const uint64_t b = pr.min_repeats > 1 ? (uint64_t)(pr.min_repeats - 1) * k : k - 1;
        const uint64_t rmin = std::max<uint64_t>(std::max(a, b), 1);
        e.rmin = (uint32_t)std::min<uint64_t>(rmin, 0xFFFFFF00u);
        e.re = (uint8_t)std::min<uint32_t>(e.rmin, 32);
        {
            int n = 0;
            for (uint32_t covered = 1; covered < e.re;) {
                const uint32_t sh = std::min<uint32_t>(covered, e.re - covered);
                e.esh[n++] = (uint8_t)sh;
                covered += sh;
            }
        }
        if (e.rmin >= 63) e.mode = MODE_WORD;
        else if (e.rmin >= 31) e.mode = MODE_HALF;
        else if (e.rmin >= 15) e.mode = MODE_BYTE;
        else {
            e.mode = MODE_ERODE;
            const uint32_t r = std::min<uint32_t>(e.rmin, 8);
            int n = 0;
            for (uint32_t covered = 1; covered < r;) {
                const uint32_t sh = std::min(covered, r - covered);
                e.sh[n++] = (uint8_t)sh;
                covered += sh;
            }
        }
        int nd = 0;
        uint32_t m = k;
        for (uint32_t p = 2; p * p <= m; ++p)
            if (m % p == 0) {
                e.div[nd++] = (uint16_t)(k / p);
                while (m % p == 0) m /= p;
            }
        if (m > 1 && m < k) e.div[nd++] = (uint16_t)(k / m);  // m == k: k itself is prime -> d = 1
        else if (m > 1 && k > 1) e.div[nd++] = 1;
        if (pr.flags & CRF_SCAN_NO_PRIMITIVITY)
            for (int j = 0; j < 6; ++j) e.div[j] = 0;
    }
    // segments: maximal k ranges with the same k >> 5, the same fast-phase filter and the same homopolymer
    // suppression level (2 <= k <= 8: stretches of > 8 equal bases; 9 <= k <= 16: > 16; none for the H-plane
    // filters, for k = 1 itself, and when the load has exotic symbols, whose filler codes may collide)
    segs.clear();
    for (uint32_t k = pr.min_motif_size; k <= pr.max_motif_size; ++k) {
        const KEntry &e = tab[k];
        uint8_t sup = 0;
        if (allow_sup && (e.mode == MODE_ERODE || e.mode == MODE_BYTE) && k >= 2 && k <= 16) sup = k <= 8 ? 1 : 2;
        const uint8_t mode = (uint8_t)(e.mode | (sup << 4));
        if (!segs.empty()) {
            Seg &g = segs.back();
            if ((uint32_t)(g.k_hi >> 5) == (k >> 5) && g.mode == mode && g.sh0 == e.sh[0] && g.sh1 == e.sh[1] &&
                g.sh2 == e.sh[2]) {
                g.k_hi = (uint16_t)k;
                continue;
            }
        }
        segs.push_back(Seg{(uint16_t)k, (uint16_t)k, mode, e.sh[0], e.sh[1], e.sh[2]});
    }
}

static int ensure_result_buffers(crf_seq *s, uint32_t cap) {
    if (cap <= s->res_cap) return CRF_OK;
    dev_free(s->stage_key); dev_free(s->spill_key); dev_free(s->fin_key);
    dev_free(s->stage_k); dev_free(s->spill_k); dev_free(s->fin_k);
    dev_free(s->o_rec); dev_free(s->o_start); dev_free(s->o_end); dev_free(s->o_k);
    s->res_cap = 0;
    CHECK(dev_alloc(&s->stage_key, cap)); CHECK(dev_alloc(&s->stage_k, cap));
    CHECK(dev_alloc(&s->spill_key, next_pow2(cap))); CHECK(dev_alloc(&s->spill_k, next_pow2(cap)));
    CHECK(dev_alloc(&s->fin_key, cap)); CHECK(dev_alloc(&s->fin_k, cap));
    CHECK(dev_alloc(&s->o_rec, cap)); CHECK(dev_alloc(&s->o_start, cap));
    CHECK(dev_alloc(&s->o_end, cap)); CHECK(dev_alloc(&s->o_k, cap));
    s->res_cap = cap;
    return CRF_OK;
}

// default scan kernel of this process: CRF_SCAN_KERNEL=block|warp1|warp2 (tuning / A-B runs), else the library default
static int default_warp_ns() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("CRF_SCAN_KERNEL");
        if (e && !strcmp(e, "block")) v = 0;
        else if (e && !strcmp(e, "warp1")) v = 1;
        else if (e && !strcmp(e, "warp2")) v = 2;
        else if (e && !strcmp(e, "block2")) v = 3;
        else v = CRF_DEFAULT_KERNEL;
    }
    return v;
}

static int scan_validate(const crf_seq *s, const crf_scan_params *pr) {
    // the four checks of perfect_repeat_finder.py:23-30
    if (pr->min_motif_size < 1) { set_err("min_motif_size is set to %u. It must be at least 1.", pr->min_motif_size); return CRF_ERR_ARG; }
    if (pr->max_motif_size < pr->min_motif_size) { set_err("max_motif_size is set to %u. It must be at least min_motif_size.", pr->max_motif_size); return CRF_ERR_ARG; }
    if (pr->min_repeats < 1) { set_err("min_repeats is set to %u. It must be at least 1.", pr->min_repeats); return CRF_ERR_ARG; }
    if (pr->min_span < 1) { set_err("min_span is set to %u. It must be at least 1.", pr->min_span); return CRF_ERR_ARG; }
    if (pr->min_repeats == 1 && pr->min_motif_size == 1 && pr->min_span <= 1) {
        set_err("min_repeats == 1 with min_motif_size == 1 and min_span == 1 reports every single base as a repeat "
                "(perfect_repeat_tracker.py:86-91); this degenerate setting is not implemented on the GPU path");
        return CRF_ERR_UNSUPPORTED;
    }
    if (pr->max_motif_size > s->cap) {
        set_err("max_motif_size %u exceeds the max_motif_cap %u this sequence was loaded with", pr->max_motif_size, s->cap);
        return CRF_ERR_ARG;
    }
    const int T = pr->words_per_thread ? (int)pr->words_per_thread : 8;
    if (T != 1 && T != 2 && T != 4 && T != 8 && T != 16) { set_err("words_per_thread must be 1, 2, 4, 8 or 16"); return CRF_ERR_ARG; }
    const uint32_t outcap = pr->tile_out_cap ? pr->tile_out_cap : 1024;
    if (outcap > 4096) { set_err("tile_out_cap must be <= 4096"); return CRF_ERR_ARG; }
    return CRF_OK;
}

// per-k table, tile arrays, launch geometry (no kernel launches; one blocking upload when the filters changed)
static int scan_prepare(crf_seq *s, const crf_scan_params *pr, ScanPlan &pl) {
    crf_ctx *c = s->ctx;
    cudaStream_t st = c->stream;
    pl.pr = *pr;
    pl.T = pr->words_per_thread ? (int)pr->words_per_thread : 8;
    if (s->ktab_cap < pr->max_motif_size + 1) {
        dev_free(s->d_ktab);
        s->ktab_cap = 0;
        CHECK(dev_alloc(&s->d_ktab, (size_t)pr->max_motif_size + 1));
        s->ktab_cap = pr->max_motif_size + 1;
        s->ktab_for.max_motif_size = 0;
    }
    if (s->ktab_for.max_motif_size != pr->max_motif_size || s->ktab_for.min_repeats != pr->min_repeats ||
        s->ktab_for.min_span != pr->min_span || s->ktab_for.flags != pr->flags ||
        s->ktab_for.min_motif_size != pr->min_motif_size) {
        std::vector<KEntry> tab;
        std::vector<Seg> segs;
        // the suppression relies on the primitivity rule dropping what it hides: not with CRF_SCAN_NO_PRIMITIVITY
        build_ktab(*pr, s->n_exotic == 0 && pr->min_repeats > 1 && !(pr->flags & (CRF_SCAN_DEBUG_NO_SUP | CRF_SCAN_NO_PRIMITIVITY)),
                   tab, segs);
        s->sup_enabled = 0;
        for (const Seg &g : segs) s->sup_enabled |= (g.mode >> 4) ? 1u : 0u;
        if (s->segs_cap < segs.size()) {
            dev_free(s->d_segs);
            s->segs_cap = 0;
            CHECK(dev_alloc(&s->d_segs, segs.size()));
            s->segs_cap = (uint32_t)segs.size();
        }
        s->n_segs = (uint32_t)segs.size();
        CU(cudaMemcpyAsync(s->d_ktab, tab.data(), tab.size() * sizeof(KEntry), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(s->d_segs, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));  // tab / segs are locals
        s->ktab_for = *pr;
    }
    // which kernel: the warp-tiled one (CRF_SCAN_WARP_TILES, two sub-tiles per warp) or the block-tiled one; T != 8 exists
    // only block-tiled.  CRF_SCAN_KERNEL=block|warp1|warp2 overrides the default (tuning).
    pl.warp_ns = default_warp_ns();
    pl.block_ns = 1;
    if (pl.warp_ns == 3) { pl.warp_ns = 0; pl.block_ns = 2; }
    if (pr->flags & CRF_SCAN_BLOCK_TILES) pl.warp_ns = 0;
    if (pr->flags & CRF_SCAN_WARP_TILES) pl.warp_ns = std::max(pl.warp_ns, 1);
    if (pr->flags & CRF_SCAN_TWO_STRIPS) { pl.warp_ns = 0; pl.block_ns = 2; }
    if (pl.T != 8 || pr->max_motif_size > 1024) { pl.warp_ns = 0; pl.block_ns = 1; }   // (other shapes: the plain block kernel)
    const uint32_t TW = pl.warp_ns ? 32u * pl.T * pl.warp_ns : (uint32_t)THREADS * pl.T * pl.block_ns;
    pl.n_tiles = (s->n_words + TW - 1) / TW;
    if (s->tiles_cap < pl.n_tiles + 1) {
        dev_free(s->tile_cnt); dev_free(s->tile_base); dev_free(s->tile_off);
        s->tiles_cap = 0;
        CHECK(dev_alloc(&s->tile_cnt, (size_t)pl.n_tiles + 8));   // slack: tile_offsets_kernel reads uint4
        CHECK(dev_alloc(&s->tile_base, (size_t)pl.n_tiles + 1));
        CHECK(dev_alloc(&s->tile_off, (size_t)pl.n_tiles + 1));
        s->tiles_cap = pl.n_tiles + 1;
    }
    if (pl.warp_ns) {
        pl.outcap = pr->tile_out_cap ? std::min<uint32_t>(pr->tile_out_cap, 256) : 48u * pl.warp_ns;
        pl.smem = WARPS_PER_CTA * warp_smem_bytes(pl.T, pl.warp_ns, pr->max_motif_size, pl.outcap);
        int per_sm = 0, n_sm = 0;
        CU(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, c->device));
        if (pl.warp_ns == 1) {
            CU(cudaFuncSetAttribute(scan_warp_kernel<8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, scan_warp_kernel<8, 1>, 32 * WARPS_PER_CTA, pl.smem));
        } else {
            CU(cudaFuncSetAttribute(scan_warp_kernel<8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, scan_warp_kernel<8, 2>, 32 * WARPS_PER_CTA, pl.smem));
        }
        if (per_sm < 1) { set_err("crf_scan: the warp-tiled kernel does not fit an SM (%zu bytes of shared memory)", pl.smem); return CRF_ERR_UNSUPPORTED; }
        pl.warp_grid = std::min<uint32_t>((uint32_t)per_sm * n_sm, (pl.n_tiles + WARPS_PER_CTA - 1) / WARPS_PER_CTA);
        pl.warp_grid = std::max(pl.warp_grid, 1u);
    } else {
        pl.outcap = pr->tile_out_cap ? pr->tile_out_cap : 1024;
        pl.smem = scan_smem_bytes(pl.T, pr->max_motif_size, pl.outcap, pl.block_ns);
        const int smem = (int)pl.smem;
        if (pl.block_ns == 2) CU(cudaFuncSetAttribute(scan_kernel<8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        else if (pl.T == 1) CU(cudaFuncSetAttribute(scan_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        else if (pl.T == 2) CU(cudaFuncSetAttribute(scan_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        else if (pl.T == 4) CU(cudaFuncSetAttribute(scan_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        else if (pl.T == 8) CU(cudaFuncSetAttribute(scan_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        else CU(cudaFuncSetAttribute(scan_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
    pl.single_copy = pr->min_repeats == 1;    // see single_copy_filter_kernel
    return CRF_OK;
}

static uint32_t default_result_cap(const crf_seq *s, const crf_scan_params *pr) {
    const uint32_t cap = pr->result_cap ? pr->result_cap : std::max<uint32_t>(1u << 16, s->layout_len / 96);
    return std::max(cap, s->res_cap);
}

static int launch_translate(crf_seq *s, ScanPlan &pl, cudaStream_t st) {
    pl.tp.open_rows = s->d_open_rows;
    pl.tp.open_cap = s->open_cap;
    translate_kernel<<<pl.tgrid, 256, 0, st>>>(pl.tp);
    CU(cudaGetLastError());
    ++pl.launches;
    return CRF_OK;
}

// Everything the kernels of one scan are launched with; doubles as the key of the captured CUDA graph.
struct ScanLaunch {
    ScanParams sp;
    GatherParams g;
    TranslateParams tp;
    uint32_t T, warp_ns, block_ns, warp_grid, n_tiles, ggrid, tgrid, single_copy;
    unsigned long long smem;
    uint32_t *tile_off;
    uint32_t n_words_alloc, res_cap;
};

// memset -> scan -> tile offsets -> spill sort -> gather -> (single-copy filter) -> translate on `st`; ev[0] .. ev[3] bracket
// the whole / the scan kernel (ev_flags = cudaEventRecordExternal while the stream is being captured into a graph).
static int scan_launch_all(crf_seq *s, const ScanLaunch &L, cudaStream_t st, unsigned ev_flags, uint32_t *launches,
                           cudaEvent_t rows_free = nullptr) {
    CU(cudaEventRecordWithFlags(s->ev[0], st, ev_flags));
    CU(cudaMemsetAsync(s->d_counters, 0, C_COUNT * sizeof(unsigned long long), st));
    CU(cudaEventRecordWithFlags(s->ev[1], st, ev_flags));
    const uint32_t n_tiles = L.n_tiles;
    const size_t smem = (size_t)L.smem;
    if (L.warp_ns == 1) scan_warp_kernel<8, 1><<<L.warp_grid, 32 * WARPS_PER_CTA, smem, st>>>(L.sp);
    else if (L.warp_ns == 2) scan_warp_kernel<8, 2><<<L.warp_grid, 32 * WARPS_PER_CTA, smem, st>>>(L.sp);
    else if (L.block_ns == 2) scan_kernel<8, 2><<<n_tiles, THREADS, smem, st>>>(L.sp);
    else if (L.T == 1) scan_kernel<1><<<n_tiles, THREADS, smem, st>>>(L.sp);
    else if (L.T == 2) scan_kernel<2><<<n_tiles, THREADS, smem, st>>>(L.sp);
    else if (L.T == 4) scan_kernel<4><<<n_tiles, THREADS, smem, st>>>(L.sp);
    else if (L.T == 8) scan_kernel<8><<<n_tiles, THREADS, smem, st>>>(L.sp);
    else scan_kernel<16><<<n_tiles, THREADS, smem, st>>>(L.sp);
    CU(cudaGetLastError());
    CU(cudaEventRecordWithFlags(s->ev[2], st, ev_flags));
    tile_offsets_kernel<<<1, 1024, 0, st>>>(s->tile_cnt, L.tile_off, n_tiles, s->d_counters);
    spill_sort_small_kernel<<<1, 1024, 0, st>>>(L.sp.spill_key, L.sp.spill_k, L.res_cap, s->d_counters);
    gather_kernel<<<L.ggrid, 256, 0, st>>>(L.g);
    *launches = 4;
    if (L.single_copy) {
        single_copy_filter_kernel<<<1, 1024, 0, st>>>(L.g.fin_key, L.g.fin_k, L.sp.NM, L.sp.X, L.n_words_alloc, L.res_cap,
                                                      s->d_counters);
        ++*launches;
    }
    if (rows_free) CU(cudaStreamWaitEvent(st, rows_free, 0));   // the previous step's rows may still be travelling to rank 0
    translate_kernel<<<L.tgrid, 256, 0, st>>>(L.tp);
    ++*launches;
    CU(cudaGetLastError());
    CU(cudaEventRecordWithFlags(s->ev[3], st, ev_flags));
    return CRF_OK;
}

// A scan of a small input (a chromosome, a batch of reads) is a handful of short kernels: launching them as one captured
// graph takes the per-launch gaps out of a step that is otherwise ~100 us.  The graph is re-captured whenever anything it
// was built from changes (buffers grown, other filters, another output map).
static const uint32_t GRAPH_MAX_TILES = 8192;
static void free_graph_key(ScanLaunch *k) { delete k; }

static int scan_enqueue(crf_seq *s, ScanPlan &pl, bool allow_graph = true) {
    cudaStream_t st = s->ctx->stream;
    const crf_scan_params *pr = &pl.pr;
    ScanLaunch L;
    memset(&L, 0, sizeof(L));                      // (the struct is compared byte-wise: padding must be defined)
    ScanParams &sp = L.sp;
    sp.H = s->H; sp.L = s->L; sp.NM = s->NM; sp.X = s->X;
    sp.ktab = s->d_ktab; sp.segs = s->d_segs; sp.n_segs = s->n_segs;
    sp.ex_key = s->ex_key; sp.n_exotic = s->n_exotic;
    sp.rec_dev_off = s->d_rec_dev_off; sp.own_lo = s->d_own_lo; sp.own_hi = s->d_own_hi; sp.n_records = s->n_records;
    sp.n_words = s->n_words;
    sp.kmin = pr->min_motif_size; sp.kmax = pr->max_motif_size;
    sp.outcap = pl.outcap;
    sp.walk_limit = pr->walk_limit_words ? pr->walk_limit_words : 64;
    sp.debug_flags = (pr->flags >> 16) & 0xFFFFu;
    sp.sup_enabled = s->sup_enabled;
    sp.stage_key = s->stage_key; sp.stage_k = s->stage_k; sp.stage_cap = s->res_cap;
    sp.tile_cnt = s->tile_cnt; sp.tile_base = s->tile_base;
    sp.spill_key = s->spill_key; sp.spill_k = s->spill_k; sp.spill_cap = s->res_cap;
    sp.counters = s->d_counters;
    const uint32_t n_tiles = pl.n_tiles;
    GatherParams &g = L.g;
    g.stage_key = s->stage_key; g.stage_k = s->stage_k;
    g.tile_cnt = s->tile_cnt; g.tile_base = s->tile_base; g.tile_off = s->tile_off;
    g.spill_key = s->spill_key; g.spill_k = s->spill_k;
    g.fin_key = s->fin_key; g.fin_k = s->fin_k;
    g.n_tiles = n_tiles; g.fin_cap = s->res_cap; g.stage_cap = s->res_cap; g.spill_cap = s->res_cap;
    g.tile_words = pl.warp_ns ? 32u * pl.T * pl.warp_ns : (uint32_t)THREADS * pl.T * pl.block_ns; g.spill_sorted = 0;
    g.counters = s->d_counters;
    pl.ggrid = (n_tiles * 32 + 255) / 256;
    pl.tgrid = std::min<uint32_t>(148 * 8, (s->res_cap + 255) / 256);
    TranslateParams &tp = L.tp;
    tp.fin_key = s->fin_key; tp.fin_k = s->fin_k; tp.rec_dev_off = s->d_rec_dev_off; tp.rec_len = s->d_rec_len;
    tp.map_rec = s->d_map_rec; tp.map_shift = s->d_map_shift; tp.map_open = s->d_map_open;
    tp.n_records = s->n_records; tp.fin_cap = s->res_cap; tp.counters = s->d_counters;
    tp.o_rec = s->o_rec; tp.o_start = s->o_start; tp.o_end = s->o_end; tp.o_k = s->o_k;
    tp.open_rows = s->d_open_rows; tp.open_cap = s->open_cap;
    pl.g = g;
    pl.tp = tp;
    L.T = (uint32_t)pl.T; L.warp_ns = (uint32_t)pl.warp_ns; L.block_ns = (uint32_t)pl.block_ns; L.warp_grid = pl.warp_grid;
    L.n_tiles = n_tiles; L.ggrid = pl.ggrid; L.tgrid = pl.tgrid; L.single_copy = pl.single_copy ? 1u : 0u;
    L.smem = pl.smem; L.tile_off = s->tile_off; L.n_words_alloc = s->n_words_alloc; L.res_cap = s->res_cap;

    // The previous push of this sequence's rows (on the exchange's own stream) comes first -- for the kernels that overwrite
    // what it reads: the scan counters (read by its first kernel) and the rows (until its last).  With CRF_XCHG_OVERLAP=0 the
    // whole scan waits for the whole push.
    static const bool overlap_off = getenv("CRF_XCHG_OVERLAP") != nullptr && atoi(getenv("CRF_XCHG_OVERLAP")) == 0;
    cudaEvent_t rows_free = nullptr;
    if (s->side_done) {
        if (s->pub_done && !overlap_off) {
            CU(cudaStreamWaitEvent(st, s->pub_done, 0));
            rows_free = s->side_done;
        } else {
            CU(cudaStreamWaitEvent(st, s->side_done, 0));
        }
        s->side_done = s->pub_done = nullptr;
    }
    static const bool graphs_off = getenv("CRF_NO_GRAPH") != nullptr;
    // (not on a rank of a multi-GPU job: instantiating a graph may wait for kernels that are themselves waiting for peers)
    if (allow_graph && s->ctx->n_xchg == 0 && n_tiles <= GRAPH_MAX_TILES && !graphs_off) {
        if (rows_free) { CU(cudaStreamWaitEvent(st, rows_free, 0)); rows_free = nullptr; }   // (a captured scan waits as a whole)
        if (!s->graph_exec || !s->graph_key || memcmp(s->graph_key, &L, sizeof(L)) != 0) {
            if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
            if (!s->graph_key) s->graph_key = new (std::nothrow) ScanLaunch;
            if (!s->graph_key) { set_err("out of host memory"); return CRF_ERR_NOMEM; }
            cudaGraph_t graph = nullptr;
            CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            const int rc = scan_launch_all(s, L, st, cudaEventRecordExternal, &s->graph_launches);
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            if (e == cudaSuccess) e = cudaGraphInstantiate(&s->graph_exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (e != cudaSuccess) { s->graph_exec = nullptr; set_err("crf_scan: graph capture failed: %s", cudaGetErrorString(e)); return CRF_ERR_CUDA; }
            memcpy(s->graph_key, &L, sizeof(L));
        }
        CU(cudaGraphLaunch(s->graph_exec, st));
        pl.launches = s->graph_launches;
        return CRF_OK;
    }
    return scan_launch_all(s, L, st, cudaEventRecordDefault, &pl.launches, rows_free);
}

// after the counters of a completed scan are on the host
static int scan_fill_stats(crf_seq *s, const ScanPlan &pl, uint32_t reruns) {
    const unsigned long long n_total = s->h_counters[C_STAGE] + s->h_counters[C_SPILL];
    float ms_all = 0, ms_k = 0;
    CU(cudaEventElapsedTime(&ms_all, s->ev[0], s->ev[3]));
    CU(cudaEventElapsedTime(&ms_k, s->ev[1], s->ev[2]));
    const unsigned long long n_kept = pl.single_copy ? s->h_counters[C_TOTAL] : n_total;
    s->n_results = n_kept;
    s->have_results = true;
    s->stats.scan_ms = ms_all;
    s->stats.kernel_ms = ms_k;
    s->stats.n_results = n_kept;
    s->stats.n_tiles = pl.n_tiles;
    s->stats.n_spilled = s->h_counters[C_SPILL];
    s->stats.n_long = s->h_counters[C_LONG];
    s->stats.n_open = s->h_counters[C_OPEN];
    s->stats.n_candidates = s->h_counters[C_CAND];
    s->stats.word_k_pairs = (uint64_t)s->n_words * (pl.pr.max_motif_size - pl.pr.min_motif_size + 1);
    s->stats.reruns = reruns;
    s->stats.launches = pl.launches;
    return CRF_OK;
}

extern "C" int crf_scan(crf_seq *s, const crf_scan_params *pr, uint64_t *n_results) {
    if (!s || !pr) { set_err("crf_scan: null argument"); return CRF_ERR_ARG; }
    CHECK(scan_validate(s, pr));
    crf_ctx *c = s->ctx;
    cudaStream_t st = c->stream;
    CU(cudaSetDevice(c->device));
    g_ctx = c;
    s->have_results = false;
    if (!s->plan) s->plan = new (std::nothrow) ScanPlan;
    if (!s->plan) { set_err("out of host memory"); return CRF_ERR_NOMEM; }
    ScanPlan &pl = *s->plan;
    CHECK(scan_prepare(s, pr, pl));
    uint32_t cap = default_result_cap(s, pr);

    uint32_t reruns = 0;
    for (;;) {
        CHECK(ensure_result_buffers(s, cap));
        CHECK(scan_enqueue(s, pl));
        CU(cudaMemcpyAsync(s->h_counters, s->d_counters, C_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));

        const unsigned long long n_stage = s->h_counters[C_STAGE], n_spill = s->h_counters[C_SPILL];
        const unsigned long long n_total = n_stage + n_spill;
        if (n_stage > s->res_cap || n_spill > s->res_cap || n_total > s->res_cap) {
            if (n_total + 1024 > 0xFFFFFFF0ull) { set_err("crf_scan: more than 2^32 results"); return CRF_ERR_UNSUPPORTED; }
            cap = (uint32_t)(n_total + n_total / 16 + 1024);
            ++reruns;
            continue;
        }
        bool again = false;
        if (n_spill > SPILL_SMALL) {  // a long spill list: sort it with the global network, then gather again
            CHECK(bitonic_sort(st, s->spill_key, s->spill_k, (uint32_t)n_spill, &pl.launches));
            pl.g.spill_sorted = 1;
            gather_kernel<<<pl.ggrid, 256, 0, st>>>(pl.g);
            ++pl.launches;
            if (pl.single_copy) {
                single_copy_filter_kernel<<<1, 1024, 0, st>>>(s->fin_key, s->fin_k, s->NM, s->X, s->n_words_alloc,
                                                              s->res_cap, s->d_counters);
                ++pl.launches;
            }
            again = true;
        }
        if (s->h_counters[C_OPEN] > s->open_cap) {   // more open-ended rows than the list held: grow it, translate again
            uint32_t *bigger = nullptr;
            const uint32_t want = (uint32_t)std::min<unsigned long long>(s->h_counters[C_OPEN] + 64, 0x0FFFFFFFull);
            CHECK(dev_alloc(&bigger, 5 * (size_t)want));
            dev_free(s->d_open_rows);
            s->d_open_rows = bigger;
            s->open_cap = want;
            again = true;
        }
        if (again) {
            CU(cudaMemsetAsync(s->d_counters + C_OPEN, 0, sizeof(unsigned long long), st));
            CHECK(launch_translate(s, pl, st));
            CU(cudaEventRecord(s->ev[3], st));
            CU(cudaMemcpyAsync(s->h_counters, s->d_counters, C_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
        }
        CHECK(scan_fill_stats(s, pl, reruns));
        break;
    }
    if (n_results) *n_results = s->n_results;
    return CRF_OK;
}

extern "C" int crf_fetch(crf_seq *s, uint32_t *record, uint32_t *start, uint32_t *end, uint32_t *motif_size,
                         uint64_t capacity, int dst_on_device) {
    if (!s) { set_err("crf_fetch: null sequence"); return CRF_ERR_ARG; }
    if (!s->have_results) { set_err("crf_fetch: no scan results to fetch"); return CRF_ERR_ARG; }
    if (capacity < s->n_results) {
        set_err("crf_fetch: capacity %llu < %llu results", (unsigned long long)capacity, (unsigned long long)s->n_results);
        return CRF_ERR_CAPACITY;
    }
    if (!s->n_results) return CRF_OK;
    if (!record || !start || !end || !motif_size) { set_err("crf_fetch: null output array"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    const cudaMemcpyKind kind = dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const size_t bytes = (size_t)s->n_results * 4;
    CU(cudaMemcpyAsync(record, s->o_rec, bytes, kind, st));
    CU(cudaMemcpyAsync(start, s->o_start, bytes, kind, st));
    CU(cudaMemcpyAsync(end, s->o_end, bytes, kind, st));
    CU(cudaMemcpyAsync(motif_size, s->o_k, bytes, kind, st));
    CU(cudaStreamSynchronize(st));
    return CRF_OK;
}

extern "C" int crf_scan_stats(const crf_seq *s, crf_scan_stats_t *stats) {
    if (!s || !stats) { set_err("crf_scan_stats: null argument"); return CRF_ERR_ARG; }
    *stats = s->stats;
    return CRF_OK;
}

extern "C" int crf_fetch_open(crf_seq *s, uint32_t *rows, uint32_t cap, uint32_t *n_open) {
    if (!s || !n_open) { set_err("crf_fetch_open: null argument"); return CRF_ERR_ARG; }
    if (!s->have_results) { set_err("crf_fetch_open: no scan results"); return CRF_ERR_ARG; }
    *n_open = (uint32_t)std::min<uint64_t>(s->stats.n_open, 0xFFFFFFFFull);
    const uint32_t n = std::min<uint32_t>(std::min<uint32_t>(*n_open, cap), s->open_cap);
    if (!n) return CRF_OK;
    if (!rows) { set_err("crf_fetch_open: null rows"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(s->ctx->device));
    const uint32_t have = std::min<uint32_t>(*n_open, s->open_cap);   // rows the device list holds (crf_scan grew it to fit)
    std::vector<uint32_t> tmp(5 * (size_t)have);
    CU(cudaMemcpyAsync(tmp.data(), s->d_open_rows, tmp.size() * 4, cudaMemcpyDeviceToHost, s->ctx->stream));
    CU(cudaStreamSynchronize(s->ctx->stream));
    std::vector<uint32_t> order(have);
    for (uint32_t i = 0; i < have; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return tmp[5 * a] < tmp[5 * b]; });  // result order
    for (uint32_t i = 0; i < n; ++i) memcpy(rows + 5 * i, &tmp[5 * order[i]], 20);
    return CRF_OK;
}

extern "C" int crf_patch_end(crf_seq *s, uint64_t row, uint32_t new_end) {
    if (!s || !s->have_results || row >= s->n_results) { set_err("crf_patch_end: no such result row"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(s->ctx->device));
    CU(cudaMemcpyAsync(s->o_end + row, &new_end, 4, cudaMemcpyHostToDevice, s->ctx->stream));
    CU(cudaStreamSynchronize(s->ctx->stream));
    return CRF_OK;
}

extern "C" int crf_run_end(crf_seq *s, uint32_t record, uint32_t pos, uint32_t k, uint32_t *run_end) {
    if (!s || !run_end) { set_err("crf_run_end: null argument"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(s->ctx->device));
    CHECK(host_tables(s));
    if (record >= s->n_records || pos >= s->h_rec_len[record]) { set_err("crf_run_end: position out of range"); return CRF_ERR_ARG; }
    if (k < 1 || k > s->cap) { set_err("crf_run_end: k %u not in [1, max_motif_cap %u]", k, s->cap); return CRF_ERR_ARG; }
    cudaStream_t st = s->ctx->stream;
    ScanParams sp = {};
    sp.H = s->H; sp.L = s->L; sp.NM = s->NM; sp.X = s->X;
    sp.ex_key = s->ex_key; sp.n_exotic = s->n_exotic; sp.n_words = s->n_words;
    uint32_t *d_out = reinterpret_cast<uint32_t *>(s->d_counters + C_COUNT - 1);
    const uint32_t d0 = s->h_rec_dev_off[record];
    run_end_kernel<<<1, THREADS, 0, st>>>(sp, k, d0 + pos, d_out);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(s->h_counters, d_out, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *run_end = *reinterpret_cast<uint32_t *>(s->h_counters) - d0;
    return CRF_OK;
}

extern "C" int crf_interval_stop(crf_seq *s, uint32_t min_motif_size, uint32_t max_motif_size, const uint64_t *end_pos,
                                 const uint64_t *full_len, int64_t *stop) {
    if (!s) { set_err("crf_interval_stop: null sequence"); return CRF_ERR_ARG; }
    if (min_motif_size < 1 || max_motif_size < min_motif_size || max_motif_size > s->cap) {
        set_err("crf_interval_stop: motif sizes [%u, %u] not inside [1, max_motif_cap %u]", min_motif_size, max_motif_size, s->cap);
        return CRF_ERR_ARG;
    }
    const uint32_t n = s->n_records;
    if (!n) return CRF_OK;
    if (!end_pos || !full_len || !stop) { set_err("crf_interval_stop: null argument"); return CRF_ERR_ARG; }
    const size_t per_warp = (size_t)(max_motif_size - min_motif_size + 1) * sizeof(uint32_t);
    uint32_t warps = STOP_WARPS;
    while (warps > 1 && warps * per_warp > (48u << 10)) warps /= 2;
    const size_t smem = warps * per_warp;
    if (smem > (227u << 10)) {
        set_err("crf_interval_stop: %u motif sizes need more shared memory than a block has", max_motif_size - min_motif_size + 1);
        return CRF_ERR_UNSUPPORTED;
    }
    crf_ctx *c = s->ctx;
    CU(cudaSetDevice(c->device));
    g_ctx = c;
    cudaStream_t st = c->stream;
    if (smem > (48u << 10)) CU(cudaFuncSetAttribute(interval_stop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uint64_t *d_buf = nullptr;                            // end_pos | full_len | stop
    CHECK(dev_alloc(&d_buf, 3 * (size_t)n));
    StopParams p = {};
    p.H = s->H; p.L = s->L; p.NM = s->NM; p.X = s->X;
    p.ex_key = s->ex_key; p.n_exotic = s->n_exotic;
    p.rec_dev_off = s->d_rec_dev_off; p.rec_len = s->d_rec_len; p.n_records = n;
    p.kmin = min_motif_size; p.kmax = max_motif_size;
    p.end_pos = d_buf; p.full_len = d_buf + n; p.stop = reinterpret_cast<int64_t *>(d_buf + 2 * (size_t)n);
    cudaError_t e = cudaMemcpyAsync(d_buf, end_pos, (size_t)n * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_buf + n, full_len, (size_t)n * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        interval_stop_kernel<<<(n + warps - 1) / warps, 32 * warps, smem, st>>>(p);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(stop, p.stop, (size_t)n * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    dev_free(d_buf);
    if (e != cudaSuccess) { set_err("crf_interval_stop: %s", cudaGetErrorString(e)); return CRF_ERR_CUDA; }
    for (uint32_t r = 0; r < n; ++r)
        if (stop[r] == STOP_BAD_ARG) {
            set_err("crf_interval_stop: record %u of the load is longer than its full_len %llu", r, (unsigned long long)full_len[r]);
            return CRF_ERR_ARG;
        }
    return CRF_OK;
}

// ---- per-base masks (crf_mask.cuh) ------------------------------------------------------------------
static int mask_rows_impl(crf_ctx *c, const uint32_t *record, const uint32_t *start, const uint32_t *end, uint64_t n_rows,
                          int rows_on_device, const uint64_t *dst_offset, uint32_t n_records, uint32_t *mask,
                          uint64_t mask_bits, int mask_on_device, void **scratch) {
    cudaStream_t st = c->stream;
    const uint64_t n_words = (mask_bits + 31) / 32;
    const uint64_t batch = std::min<uint64_t>(n_rows, MASK_BATCH_ROWS);
    // scratch: queue counter, error flag | dst_offset | queue slots | device mask (host mask) | rows (host rows)
    size_t off = 16;
    const size_t at_dst = off;   off += (size_t)n_records * 8;
    const size_t at_first = off; off += (size_t)batch * 8;
    const size_t at_slot = off;  off += ((size_t)batch * 4 + 7) & ~(size_t)7;
    const size_t at_mask = off;  if (!mask_on_device) off += (size_t)n_words * 4;
    const size_t at_rows = off;  if (!rows_on_device) off += 3 * (size_t)n_rows * 4;
    CU(ctx_malloc(scratch, off));
    uint8_t *base = (uint8_t *)*scratch;
    MaskParams p = {};
    p.dst_offset = (const uint64_t *)(base + at_dst);
    p.n_records = n_records;
    p.mask_bits = mask_bits;
    p.mask = mask_on_device ? mask : (uint32_t *)(base + at_mask);
    p.queue_ctr = (unsigned long long *)base;
    p.err = (uint32_t *)(base + 8);
    p.queue_first = (uint64_t *)(base + at_first);
    p.queue_row = (uint32_t *)(base + at_slot);
    if (!rows_on_device) {
        uint32_t *rows = (uint32_t *)(base + at_rows);
        CU(cudaMemcpyAsync(rows, record, n_rows * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(rows + n_rows, start, n_rows * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(rows + 2 * n_rows, end, n_rows * 4, cudaMemcpyHostToDevice, st));
        record = rows; start = rows + n_rows; end = rows + 2 * n_rows;
    }
    if (n_records) CU(cudaMemcpyAsync((void *)p.dst_offset, dst_offset, (size_t)n_records * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(base + 8, 0, 8, st));
    CU(cudaMemsetAsync(p.mask, 0, n_words * 4, st));
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    for (uint64_t first = 0; first < n_rows; first += MASK_BATCH_ROWS) {
        p.n_rows = (uint32_t)std::min<uint64_t>(MASK_BATCH_ROWS, n_rows - first);
        p.record = record + first; p.start = start + first; p.end = end + first;
        CU(cudaMemsetAsync(p.queue_ctr, 0, 8, st));
        mask_rows_kernel<<<(p.n_rows + 255) / 256, 256, 0, st>>>(p);
        mask_long_rows_kernel<<<8 * sms, 256, 0, st>>>(p);
        CU(cudaGetLastError());
    }
    uint32_t err = 0;
    CU(cudaMemcpyAsync(&err, p.err, 4, cudaMemcpyDeviceToHost, st));
    if (!mask_on_device) CU(cudaMemcpyAsync(mask, p.mask, n_words * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (err) {
        set_err("crf_mask_rows: %s", err & MASK_ERR_ORDER ? "a row ends before it starts"
                                     : err & MASK_ERR_RECORD ? "a row's record is not below n_records"
                                                             : "a row reaches past mask_bits");
        return CRF_ERR_ARG;
    }
    return CRF_OK;
}

extern "C" int crf_mask_rows(crf_ctx *c, const uint32_t *record, const uint32_t *start, const uint32_t *end, uint64_t n_rows,
                             int rows_on_device, const uint64_t *dst_offset, uint32_t n_records, uint32_t *mask,
                             uint64_t mask_bits, int mask_on_device) {
    if (!c) { set_err("crf_mask_rows: null context"); return CRF_ERR_ARG; }
    if ((n_rows && (!record || !start || !end)) || (n_records && !dst_offset) || (mask_bits && !mask)) {
        set_err("crf_mask_rows: null argument");
        return CRF_ERR_ARG;
    }
    if (mask_bits > (1ull << 62)) { set_err("crf_mask_rows: mask_bits %llu too large", (unsigned long long)mask_bits); return CRF_ERR_ARG; }
    if (!mask_bits && !n_rows) return CRF_OK;
    CU(cudaSetDevice(c->device));
    g_ctx = c;
    void *scratch = nullptr;
    const int rc = mask_rows_impl(c, record, start, end, n_rows, rows_on_device, dst_offset, n_records, mask, mask_bits,
                                  mask_on_device, &scratch);
    if (rc == CRF_ERR_CUDA) cudaStreamSynchronize(c->stream);   // nothing queued may still use the block when it is handed out again
    ctx_free(scratch);
    return rc;
}

// ---- multi-GPU gather over peer memory (crf_xchg.cuh) ---------------------------------------------
static const size_t XCHG_ROWS_OFFSET = (sizeof(XchgBlock) + 255) & ~(size_t)255;
static const uint32_t XCHG_RING = 64;

struct crf_xchg {
    crf_ctx *ctx = nullptr;
    uint32_t rank = 0, world = 1;
    uint64_t row_cap = 0;
    void *base = nullptr;                        // this rank's block (+ the row buffer on the root)
    size_t bytes = 0;
    void *peer_base[XCHG_MAX_WORLD] = {};
    bool peer_ipc[XCHG_MAX_WORLD] = {};
    bool connected[XCHG_MAX_WORLD] = {};
    uint32_t step = 0, first_unchecked = 1;      // steps are numbered from 1
    unsigned long long *h_ring = nullptr;        // page-locked: XCHG_RING x XCHG_RESULT_WORDS
    unsigned long long timeout_ns = 20ull * 1000 * 1000 * 1000;
    std::vector<crf_seq *> pending;              // sequences whose asynchronous scans feed the steps in flight
    // the exchange kernels run on their own stream behind the scan that feeds them, so the next phase's scan (another
    // sequence, the context's stream) overlaps the push of this one
    cudaStream_t xstream = nullptr;
    cudaEvent_t ev_main = nullptr, ev_side = nullptr, ev_pub = nullptr;
    bool compact = false;                        // 12-byte rows over NVLink (crf_xchg_set_compact)
};

extern "C" int crf_xchg_create(crf_ctx *c, uint32_t rank, uint32_t world, uint64_t row_cap, crf_xchg **out) {
    if (!c || !out) { set_err("crf_xchg_create: null argument"); return CRF_ERR_ARG; }
    *out = nullptr;
    if (world < 1 || world > XCHG_MAX_WORLD || rank >= world) {
        set_err("crf_xchg_create: rank %u / world %u (at most %u ranks)", rank, world, XCHG_MAX_WORLD);
        return CRF_ERR_ARG;
    }
    if (row_cap > 0xFFFFFFF0ull) { set_err("crf_xchg_create: row_cap must be below 2^32"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(c->device));
    crf_xchg *x = new (std::nothrow) crf_xchg;
    if (!x) { set_err("out of host memory"); return CRF_ERR_NOMEM; }
    x->ctx = c; x->rank = rank; x->world = world; x->row_cap = row_cap;
    x->bytes = XCHG_ROWS_OFFSET + (rank == 0 ? (size_t)row_cap * 16 : 0);
    // a plain cudaMalloc (not the context's block cache): the block is exported to other processes
    cudaError_t e = cudaMalloc(&x->base, x->bytes);
    if (e == cudaSuccess) e = cudaMemset(x->base, 0, XCHG_ROWS_OFFSET);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&x->h_ring, (size_t)XCHG_RING * XCHG_RESULT_WORDS * 8);
    // (highest priority: when the rows of one step travel while the next step's scan runs, the copy blocks take the first
    // SM slots that come free instead of queueing behind thousands of scan tiles)
    int prio_lo = 0, prio_hi = 0;
    if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&x->xstream, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&x->ev_main, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&x->ev_side, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&x->ev_pub, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        if (x->xstream) cudaStreamDestroy(x->xstream);
        if (x->ev_main) cudaEventDestroy(x->ev_main);
        if (x->ev_side) cudaEventDestroy(x->ev_side);
        if (x->ev_pub) cudaEventDestroy(x->ev_pub);
        if (x->h_ring) cudaFreeHost(x->h_ring);
        if (x->base) cudaFree(x->base);
        delete x;
        set_err("crf_xchg_create: %s", cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? CRF_ERR_NOMEM : CRF_ERR_CUDA;
    }
    memset(x->h_ring, 0, (size_t)XCHG_RING * XCHG_RESULT_WORDS * 8);
    x->peer_base[rank] = x->base;
    x->connected[rank] = true;
    ++c->n_xchg;
    *out = x;
    return CRF_OK;
}

extern "C" int crf_xchg_export(crf_xchg *x, uint8_t *handle) {
    if (!x || !handle) { set_err("crf_xchg_export: null argument"); return CRF_ERR_ARG; }
    static_assert(sizeof(cudaIpcMemHandle_t) == CRF_IPC_HANDLE_BYTES, "IPC handle size");
    CU(cudaSetDevice(x->ctx->device));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, x->base));
    memcpy(handle, &h, sizeof(h));
    return CRF_OK;
}

extern "C" int crf_xchg_connect_ipc(crf_xchg *x, uint32_t peer, const uint8_t *handle) {
    if (!x || !handle || peer >= x->world || peer == x->rank) { set_err("crf_xchg_connect_ipc: bad argument"); return CRF_ERR_ARG; }
    if (x->connected[peer]) { set_err("crf_xchg_connect_ipc: rank %u is already connected", peer); return CRF_ERR_ARG; }
    CU(cudaSetDevice(x->ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void *ptr = nullptr;
    CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    x->peer_base[peer] = ptr;
    x->peer_ipc[peer] = true;
    x->connected[peer] = true;
    return CRF_OK;
}

extern "C" int crf_xchg_connect_local(crf_xchg *x, uint32_t peer, crf_xchg *other) {
    if (!x || !other || peer >= x->world || peer == x->rank || other->rank != peer) {
        set_err("crf_xchg_connect_local: bad argument");
        return CRF_ERR_ARG;
    }
    if (x->connected[peer]) { set_err("crf_xchg_connect_local: rank %u is already connected", peer); return CRF_ERR_ARG; }
    CU(cudaSetDevice(x->ctx->device));
    if (other->ctx->device != x->ctx->device) {
        int can = 0;
        CU(cudaDeviceCanAccessPeer(&can, x->ctx->device, other->ctx->device));
        if (!can) { set_err("crf_xchg_connect_local: device %d cannot access device %d", x->ctx->device, other->ctx->device); return CRF_ERR_UNSUPPORTED; }
        cudaError_t e = cudaDeviceEnablePeerAccess(other->ctx->device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) { set_err("cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e)); return CRF_ERR_CUDA; }
    }
    x->peer_base[peer] = other->base;
    x->connected[peer] = true;
    return CRF_OK;
}

extern "C" int crf_xchg_destroy(crf_xchg *x) {
    if (!x) return CRF_OK;
    cudaSetDevice(x->ctx->device);
    cudaStreamSynchronize(x->ctx->stream);
    cudaStreamSynchronize(x->xstream);
    for (crf_seq *s : x->pending) s->side_done = s->pub_done = nullptr;
    cudaStreamDestroy(x->xstream);
    cudaEventDestroy(x->ev_main);
    cudaEventDestroy(x->ev_side);
    cudaEventDestroy(x->ev_pub);
    for (uint32_t r = 0; r < x->world; ++r)
        if (x->peer_ipc[r] && x->peer_base[r]) cudaIpcCloseMemHandle(x->peer_base[r]);
    if (x->base) cudaFree(x->base);
    if (x->h_ring) cudaFreeHost(x->h_ring);
    --x->ctx->n_xchg;
    delete x;
    return CRF_OK;
}

extern "C" int crf_xchg_set_compact(crf_xchg *x, int on) {
    if (!x) { set_err("crf_xchg_set_compact: null exchange"); return CRF_ERR_ARG; }
    x->compact = on != 0;
    return CRF_OK;
}

extern "C" int crf_xchg_set_timeout(crf_xchg *x, double seconds) {
    if (!x || !(seconds > 0)) { set_err("crf_xchg_set_timeout: bad argument"); return CRF_ERR_ARG; }
    x->timeout_ns = (unsigned long long)(seconds * 1e9);
    return CRF_OK;
}

// push + settle of the rows the sequence holds (results of the scan queued before it on the stream)
static int xchg_enqueue(crf_seq *s, crf_xchg *x, bool trusted, bool append) {
    for (uint32_t r = 0; r < x->world; ++r)
        if (!x->connected[r]) { set_err("crf_xchg: rank %u is not connected", r); return CRF_ERR_ARG; }
    if (x->step + 1 - x->first_unchecked >= XCHG_RING) {
        set_err("crf_xchg: %u steps in flight without crf_xchg_wait (at most %u)", XCHG_RING, XCHG_RING);
        return CRF_ERR_ARG;
    }
    cudaStream_t xs = x->xstream;
    CU(cudaEventRecord(x->ev_main, x->ctx->stream));          // the scan + assembly queued so far
    CU(cudaStreamWaitEvent(xs, x->ev_main, 0));
    ++x->step;
    PushParams pp = {};
    pp.self = (XchgBlock *)x->base;
    for (uint32_t r = 0; r < x->world; ++r) pp.peer[r] = (XchgBlock *)x->peer_base[r];
    pp.root_rows = (uint32_t *)((char *)x->peer_base[0] + XCHG_ROWS_OFFSET);
    pp.row_cap = x->row_cap;
    pp.rank = x->rank; pp.world = x->world; pp.step = x->step;
    pp.o_rec = s->o_rec; pp.o_start = s->o_start; pp.o_end = s->o_end; pp.o_k = s->o_k;
    pp.counters = s->d_counters;
    pp.res_cap = s->res_cap; pp.open_cap = s->open_cap;
    pp.trusted = trusted ? 1u : 0u;
    pp.append = append ? 1u : 0u;
    pp.compact = x->compact ? 1u : 0u;
    pp.timeout_ns = x->timeout_ns;
    publish_kernel<<<1, 32, 0, xs>>>(pp);
    CU(cudaEventRecord(x->ev_pub, xs));                       // the scan counters have been read: the next scan may clear them
    push_kernel<<<148 * 2, 256, 0, xs>>>(pp);
    SettleParams sp = {};
    sp.self = (XchgBlock *)x->base;
    sp.row_cap = x->row_cap; sp.rank = x->rank; sp.world = x->world; sp.step = x->step; sp.append = pp.append;
    sp.timeout_ns = x->timeout_ns;
    settle_kernel<<<1, 32, 0, xs>>>(sp);
    if (x->compact && x->rank == 0)
        unpack_kernel<<<148 * 4, 256, 0, xs>>>((XchgBlock *)x->base, (uint32_t *)((char *)x->base + XCHG_ROWS_OFFSET), x->row_cap);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(x->h_ring + (size_t)(x->step % XCHG_RING) * XCHG_RESULT_WORDS, ((XchgBlock *)x->base)->result,
                       XCHG_RESULT_WORDS * 8, cudaMemcpyDeviceToHost, xs));
    CU(cudaEventRecord(x->ev_side, xs));
    s->side_done = x->ev_side;                                // the next scan of this sequence waits for its rows to be gone
    s->pub_done = x->ev_pub;                                  // (only before it overwrites them; its kernel starts after this one)
    return CRF_OK;
}

extern "C" int crf_scan_gather(crf_seq *s, const crf_scan_params *pr, crf_xchg *x, int append) {
    if (!s || !pr || !x) { set_err("crf_scan_gather: null argument"); return CRF_ERR_ARG; }
    if (s->ctx != x->ctx) { set_err("crf_scan_gather: sequence and exchange belong to different contexts"); return CRF_ERR_ARG; }
    CHECK(scan_validate(s, pr));
    crf_ctx *c = s->ctx;
    CU(cudaSetDevice(c->device));
    g_ctx = c;
    s->have_results = false;
    if (!s->plan) s->plan = new (std::nothrow) ScanPlan;
    if (!s->plan) { set_err("out of host memory"); return CRF_ERR_NOMEM; }
    CHECK(scan_prepare(s, pr, *s->plan));
    CHECK(ensure_result_buffers(s, default_result_cap(s, pr)));
    CHECK(scan_enqueue(s, *s->plan, false));      // (no graph: instantiating one may wait for kernels that wait for peers)
    CU(cudaMemcpyAsync(s->h_counters, s->d_counters, C_COUNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    CHECK(xchg_enqueue(s, x, false, append != 0));
    if (std::find(x->pending.begin(), x->pending.end(), s) == x->pending.end()) x->pending.push_back(s);
    s->plan->launches += 3;
    return CRF_OK;
}

extern "C" int crf_xchg_push(crf_seq *s, crf_xchg *x, int append) {
    if (!s || !x) { set_err("crf_xchg_push: null argument"); return CRF_ERR_ARG; }
    if (s->ctx != x->ctx) { set_err("crf_xchg_push: sequence and exchange belong to different contexts"); return CRF_ERR_ARG; }
    if (!s->have_results) { set_err("crf_xchg_push: no scan results"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(s->ctx->device));
    CHECK(xchg_enqueue(s, x, true, append != 0));
    return CRF_OK;
}

extern "C" int crf_xchg_wait(crf_xchg *x, crf_xchg_result_t *res) {
    if (!x || !res) { set_err("crf_xchg_wait: null argument"); return CRF_ERR_ARG; }
    if (x->step == 0) { set_err("crf_xchg_wait: nothing was pushed"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(x->ctx->device));
    CU(cudaStreamSynchronize(x->xstream));                    // (behind everything the context's stream had queued)
    uint32_t worst = XCHG_OK;
    for (uint32_t st = x->first_unchecked; st <= x->step; ++st)
        worst = std::max<uint32_t>(worst, (uint32_t)x->h_ring[(size_t)(st % XCHG_RING) * XCHG_RESULT_WORDS]);
    res->steps_checked = x->step + 1 - x->first_unchecked;
    x->first_unchecked = x->step + 1;
    const unsigned long long *r = x->h_ring + (size_t)(x->step % XCHG_RING) * XCHG_RESULT_WORDS;
    res->status = (uint32_t)r[0];
    res->worst_status = worst;
    res->total_rows = r[1];
    res->total_open = r[2];
    res->my_offset = r[3];
    res->any_open = (uint32_t)r[4];
    res->base_rows = r[5];
    res->step = x->step;
    for (uint32_t q = 0; q < XCHG_MAX_WORLD; ++q) res->rows_of_rank[q] = q < x->world ? r[8 + q] : 0;
    if (res->status == XCHG_TIMEOUT) {
        set_err("crf_xchg_wait: a peer rank did not arrive within %.1f s", x->timeout_ns * 1e-9);
        return CRF_ERR_CUDA;
    }
    for (crf_seq *s : x->pending) {                           // the asynchronous scans behind these steps: their counters
        s->side_done = s->pub_done = nullptr;                 // are on the host now
        if (worst == XCHG_OK) CHECK(scan_fill_stats(s, *s->plan, 0));
    }
    x->pending.clear();
    return CRF_OK;
}

extern "C" int crf_xchg_step_result(crf_xchg *x, uint32_t step, crf_xchg_result_t *res) {
    if (!x || !res) { set_err("crf_xchg_step_result: null argument"); return CRF_ERR_ARG; }
    if (step == 0 || step >= x->first_unchecked || step + XCHG_RING <= x->step) {
        set_err("crf_xchg_step_result: step %u is not among the last %u completed steps", step, XCHG_RING);
        return CRF_ERR_ARG;
    }
    const unsigned long long *r = x->h_ring + (size_t)(step % XCHG_RING) * XCHG_RESULT_WORDS;
    memset(res, 0, sizeof(*res));
    res->status = res->worst_status = (uint32_t)r[0];
    res->steps_checked = 1;
    res->step = step;
    res->total_rows = r[1];
    res->total_open = r[2];
    res->my_offset = r[3];
    res->any_open = (uint32_t)r[4];
    res->base_rows = r[5];
    for (uint32_t q = 0; q < XCHG_MAX_WORLD; ++q) res->rows_of_rank[q] = q < x->world ? r[8 + q] : 0;
    return CRF_OK;
}

extern "C" int crf_xchg_fetch(crf_xchg *x, uint32_t *record, uint32_t *start, uint32_t *end, uint32_t *motif_size,
                              uint64_t first_row, uint64_t n_rows, int dst_on_device) {
    if (!x) { set_err("crf_xchg_fetch: null exchange"); return CRF_ERR_ARG; }
    if (x->rank != 0) { set_err("crf_xchg_fetch: the gathered rows live on rank 0"); return CRF_ERR_ARG; }
    if (first_row + n_rows > x->row_cap) { set_err("crf_xchg_fetch: rows beyond the buffer"); return CRF_ERR_ARG; }
    if (!n_rows) return CRF_OK;
    if (!record || !start || !end || !motif_size) { set_err("crf_xchg_fetch: null output array"); return CRF_ERR_ARG; }
    CU(cudaSetDevice(x->ctx->device));
    cudaStream_t st = x->ctx->stream;
    const cudaMemcpyKind kind = dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const uint32_t *rows = (const uint32_t *)((char *)x->base + XCHG_ROWS_OFFSET) + first_row;
    uint32_t *dst[4] = {record, start, end, motif_size};
    for (int j = 0; j < 4; ++j) CU(cudaMemcpyAsync(dst[j], rows + (size_t)j * x->row_cap, (size_t)n_rows * 4, kind, st));
    CU(cudaStreamSynchronize(st));
    return CRF_OK;
}

extern "C" int crf_xchg_patch_end(crf_xchg *x, const uint64_t *rows, const uint32_t *new_end, uint32_t n) {
    if (!x || (n && (!rows || !new_end))) { set_err("crf_xchg_patch_end: null argument"); return CRF_ERR_ARG; }
    if (x->rank != 0) { set_err("crf_xchg_patch_end: the gathered rows live on rank 0"); return CRF_ERR_ARG; }
    if (!n) return CRF_OK;
    CU(cudaSetDevice(x->ctx->device));
    g_ctx = x->ctx;
    cudaStream_t st = x->ctx->stream;
    uint64_t *d_idx = nullptr;
    uint32_t *d_end = nullptr;
    CHECK(dev_alloc(&d_idx, n));
    int rc = dev_alloc(&d_end, n);
    cudaError_t e = cudaSuccess;
    if (!rc) {
        e = cudaMemcpyAsync(d_idx, rows, (size_t)n * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_end, new_end, (size_t)n * 4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) {
            patch_rows_kernel<<<(n + 255) / 256, 256, 0, st>>>((uint32_t *)((char *)x->base + XCHG_ROWS_OFFSET), x->row_cap, d_idx, d_end, n);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    dev_free(d_idx);
    dev_free(d_end);
    if (rc) return rc;
    if (e != cudaSuccess) { set_err("crf_xchg_patch_end: %s", cudaGetErrorString(e)); return CRF_ERR_CUDA; }
    return CRF_OK;
}

static cudaError_t preload_kernels() {
    cudaError_t e = preload(scan_kernel<1>);
    if (e == cudaSuccess) e = preload(scan_kernel<8, 2>);
    if (e == cudaSuccess) e = preload(scan_warp_kernel<8, 1>);
    if (e == cudaSuccess) e = preload(scan_warp_kernel<8, 2>);
    if (e == cudaSuccess) e = preload(scan_kernel<2>);
    if (e == cudaSuccess) e = preload(scan_kernel<4>);
    if (e == cudaSuccess) e = preload(scan_kernel<8>);
    if (e == cudaSuccess) e = preload(scan_kernel<16>);
    if (e == cudaSuccess) e = preload(pack_kernel);
    if (e == cudaSuccess) e = preload(repack_kernel);
    if (e == cudaSuccess) e = preload(twobit_pack_kernel);
    if (e == cudaSuccess) e = preload(nibble_pack_kernel);
    if (e == cudaSuccess) e = preload(mask_runs_kernel);
    if (e == cudaSuccess) e = preload(exotic_apply_kernel);
    if (e == cudaSuccess) e = preload(tile_offsets_kernel);
    if (e == cudaSuccess) e = preload(spill_sort_small_kernel);
    if (e == cudaSuccess) e = preload(gather_kernel);
    if (e == cudaSuccess) e = preload(translate_kernel);
    if (e == cudaSuccess) e = preload(single_copy_filter_kernel);
    if (e == cudaSuccess) e = preload(bitonic_step_kernel);
    if (e == cudaSuccess) e = preload(fill_u64_kernel);
    if (e == cudaSuccess) e = preload(run_end_kernel);
    if (e == cudaSuccess) e = preload(interval_stop_kernel);
    if (e == cudaSuccess) e = preload(publish_kernel);
    if (e == cudaSuccess) e = preload(push_kernel);
    if (e == cudaSuccess) e = preload(settle_kernel);
    if (e == cudaSuccess) e = preload(patch_rows_kernel);
    if (e == cudaSuccess) e = preload(unpack_kernel);
    if (e == cudaSuccess) e = preload(mask_rows_kernel);
    if (e == cudaSuccess) e = preload(mask_long_rows_kernel);
    return e;
}

#include "crf_rows.h"
#include "crf_fasta_out.h"

#include "crf_fasta.h"
#include "crf_pack.h"
