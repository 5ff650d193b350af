// crf_mask.cuh -- per-base repeat masks: the union of result rows as a bit mask (crf_mask_rows).
//
// Row i sets bits [dst_offset[record[i]] + start[i], dst_offset[record[i]] + end[i]) of the mask.  A genome's rows are
// millions of 9-100 bp repeats and a few satellites of several Mbp, so the work is cut in two:
//   mask_rows_kernel       one thread per row: checks it, paints a row of at most MASK_SHORT_WORDS words itself and
//                          queues a longer one together with its number of MASK_CHUNK_WORDS-word chunks;
//   mask_long_rows_kernel  one warp per chunk of the queued rows, its lanes on consecutive words.
// One 64-bit atomic per queued row hands out both its queue slot (high bits) and its first chunk (low bits), so the queue
// is sorted by first chunk and a chunk finds its row by binary search; no prefix-sum pass is needed.  Edge words (shared
// with other rows) are set with atomicOr, inner words with plain all-ones stores, as mask_runs_kernel does; the result is
// the same in any row order.
#pragma once
#include <stdint.h>

namespace crf {

constexpr uint32_t MASK_SHORT_WORDS = 8;       // rows spanning at most this many words are painted by their own thread
constexpr uint32_t MASK_CHUNK_WORDS = 256;     // words one warp paints per work item (8 kbp)
constexpr uint32_t MASK_SLOT_SHIFT = 40;       // queue counter: slot << 40 | chunks handed out so far
constexpr uint64_t MASK_BATCH_ROWS = 1u << 20; // rows per launch pair: slots < 2^20, chunks < 2^20 * 2^19 < 2^40
// error bits of the flag word (the host turns any of them into CRF_ERR_ARG)
constexpr uint32_t MASK_ERR_ORDER = 1, MASK_ERR_RECORD = 2, MASK_ERR_RANGE = 4;

struct MaskParams {
    const uint32_t *record, *start, *end;      // this batch's rows
    uint32_t n_rows;
    const uint64_t *dst_offset;                // per record
    uint32_t n_records;
    uint64_t mask_bits;
    uint32_t *mask;
    unsigned long long *queue_ctr;             // slot << MASK_SLOT_SHIFT | chunks
    uint64_t *queue_first;                     // per slot: first chunk (ascending with the slot)
    uint32_t *queue_row;                       // per slot: row of this batch
    uint32_t *err;
};

// the bits of word w that [a, b) covers (w inside [a >> 5, (b - 1) >> 5])
__device__ __forceinline__ uint32_t mask_word_bits(uint64_t w, uint64_t a, uint64_t b) {
    uint32_t m = 0xFFFFFFFFu;
    if (w == a >> 5) m &= 0xFFFFFFFFu << (uint32_t)(a & 31);
    if (w == (b - 1) >> 5 && (b & 31)) m &= (1u << (uint32_t)(b & 31)) - 1u;
    return m;
}

// [a, b) of row i, or false for an empty or invalid row (an invalid one also raises its error bit)
__device__ __forceinline__ bool mask_row_range(const MaskParams &p, uint32_t i, uint64_t &a, uint64_t &b) {
    const uint32_t r = p.record[i], s = p.start[i], e = p.end[i];
    uint32_t bad = 0;
    if (e < s) bad |= MASK_ERR_ORDER;
    if (r >= p.n_records) bad |= MASK_ERR_RECORD;
    else if (e > p.mask_bits || p.dst_offset[r] > p.mask_bits - e) bad |= MASK_ERR_RANGE;
    if (bad) { atomicOr(p.err, bad); return false; }
    a = p.dst_offset[r] + s;
    b = p.dst_offset[r] + e;
    return a < b;
}

__global__ void __launch_bounds__(256) mask_rows_kernel(const MaskParams p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_rows) return;
    uint64_t a, b;
    if (!mask_row_range(p, i, a, b)) return;
    const uint64_t w0 = a >> 5, w1 = (b - 1) >> 5;
    if (w1 - w0 < MASK_SHORT_WORDS) {
        for (uint64_t w = w0; w <= w1; ++w) atomicOr(&p.mask[w], mask_word_bits(w, a, b));
        return;
    }
    const uint64_t chunks = (w1 - w0 + MASK_CHUNK_WORDS) / MASK_CHUNK_WORDS;
    const unsigned long long old = atomicAdd(p.queue_ctr, (1ull << MASK_SLOT_SHIFT) | chunks);
    const uint32_t slot = (uint32_t)(old >> MASK_SLOT_SHIFT);
    p.queue_first[slot] = old & ((1ull << MASK_SLOT_SHIFT) - 1);
    p.queue_row[slot] = i;
}

// grid-stride over the chunks of the queued rows (a fixed grid: the counts stay on the device)
__global__ void __launch_bounds__(256) mask_long_rows_kernel(const MaskParams p) {
    const unsigned long long ctr = *p.queue_ctr;
    const uint32_t n_slots = (uint32_t)(ctr >> MASK_SLOT_SHIFT);
    const uint64_t n_chunks = ctr & ((1ull << MASK_SLOT_SHIFT) - 1);
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n_warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t c = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5; c < n_chunks; c += n_warps) {
        uint32_t lo = 0, hi = n_slots;                     // last slot whose first chunk is <= c
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (p.queue_first[mid] <= c) lo = mid; else hi = mid;
        }
        const uint32_t i = p.queue_row[lo];
        const uint32_t r = p.record[i];
        const uint64_t a = p.dst_offset[r] + p.start[i], b = p.dst_offset[r] + p.end[i];
        const uint64_t w0 = a >> 5, w1 = (b - 1) >> 5;
        const uint64_t from = w0 + (c - p.queue_first[lo]) * MASK_CHUNK_WORDS;
        const uint64_t to = min(w1 + 1, from + MASK_CHUNK_WORDS);
        for (uint64_t w = from + lane; w < to; w += 32) {
            if (w == w0 || w == w1) atomicOr(&p.mask[w], mask_word_bits(w, a, b));   // shared with neighbouring rows
            else p.mask[w] = 0xFFFFFFFFu;
        }
    }
}

}  // namespace crf
