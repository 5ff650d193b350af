// crf_stop.cuh -- interval mode: where the reference's lock-step loop breaks (crf_interval_stop).
//
// prf:70-74 advances one tracker per motif size k over the interval's sequence s (length L = full_len) and breaks at the
// first t > end_pos at which no tracker is mid-repeat.  Tracker k is mid-repeat at t iff the k compares of M_k ending at
// j = min(t, L-k-1) are all ones (trk:63-65; a tracker stops at L-k-1, trk:50, and keeps its state).  A record of the
// load is the loaded prefix s[0 .. W) of s.  One warp per record: lane l owns the motif sizes k = kmin + l + 32 i, walks
// the layout words from a little before end_pos + 1 and carries, per k, the run of ones of M_k that ends at the previous
// word (in shared memory) -- so each word of M_k is read once, whatever k is.
#pragma once
#include "crf_device.cuh"

namespace crf {

constexpr int64_t STOP_TO_END = -1;       // CRF_STOP_TO_END
constexpr int64_t STOP_UNDECIDED = -2;    // CRF_STOP_UNDECIDED
constexpr int64_t STOP_BAD_ARG = -3;      // the record is longer than its full_len (the host turns it into CRF_ERR_ARG)
constexpr uint32_t STOP_WARPS = 4;        // warps per block (fewer when the per-k state of four does not fit)
// per-k state: the run of ones of M_k that ends at the last word walked, capped at k; or, once the tracker has stopped
// (L-k-1 lies behind), whether it stopped mid-repeat
constexpr uint32_t FROZEN_OFF = 0xFFFFFFFEu, FROZEN_ON = 0xFFFFFFFFu;

struct StopParams {
    const uint32_t *H, *L, *NM, *X;
    const uint64_t *ex_key;
    uint32_t n_exotic;
    const uint32_t *rec_dev_off, *rec_len;
    uint32_t n_records;
    uint32_t kmin, kmax;
    const uint64_t *end_pos, *full_len;   // per record (device copies of the caller's arrays)
    int64_t *stop;
};

// bits b of m with m[b-k+1 .. b] all ones, the window inside the word (k <= 32)
__device__ __forceinline__ uint32_t erode_in_word(uint32_t m, uint32_t k) {
    uint32_t len = 1;
    while (2 * len <= k) { m &= m << len; len *= 2; }
    if (len < k) m &= m << (k - len);
    return m;
}

__device__ __forceinline__ uint32_t bits_from(uint32_t lo) { return lo >= 32 ? 0u : 0xFFFFFFFFu << lo; }   // [lo, 32)

__global__ void __launch_bounds__(32 * STOP_WARPS) interval_stop_kernel(const StopParams p) {
    extern __shared__ uint32_t stop_state[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t r = blockIdx.x * (blockDim.x >> 5) + warp;
    if (r >= p.n_records) return;
    const uint32_t nk = p.kmax - p.kmin + 1;
    uint32_t *state = stop_state + (size_t)warp * nk;
    const int64_t W = p.rec_len[r], F = (int64_t)p.full_len[r];
    const uint64_t E = p.end_pos[r];
    if (W > F) { if (lane == 0) p.stop[r] = STOP_BAD_ARG; return; }
    if (F == 0 || E + 1 >= (uint64_t)F) { if (lane == 0) p.stop[r] = STOP_TO_END; return; }   // no t > end_pos left
    const int64_t e = (int64_t)E, kmax = p.kmax;
    // last t this prefix decides: with W < F a tracker k at t reads s[t + k], so t <= W - 1 - kmax
    const int64_t t_hi = W < F ? W - 1 - kmax : F - 1;
    if (t_hi < e + 1) { if (lane == 0) p.stop[r] = STOP_UNDECIDED; return; }
    // the walk starts k before the first compare it needs: before e + 1, or up to 2k before the end for a tracker that
    // stops before e + 1 (L - k - 1 < e + 1)
    const int64_t s0 = max((int64_t)0, min(e + 1 - kmax, F - 2 * kmax));
    const uint32_t d0 = p.rec_dev_off[r];
    for (uint32_t i = lane; i < nk; i += 32) {
        const int64_t j_end = F - (int64_t)(p.kmin + i) - 1;
        state[i] = j_end < 0 ? FROZEN_OFF : 0u;     // a tracker with no compare at all never is mid-repeat
    }
    __syncwarp();
    const uint32_t t_lo_pos = d0 + (uint32_t)(e + 1), t_hi_pos = d0 + (uint32_t)t_hi;   // layout positions of the t range
    const uint32_t w_first = (d0 + (uint32_t)s0) >> 5, w_last = t_hi_pos >> 5;
    for (uint32_t w = w_first; w <= w_last; ++w) {
        const uint32_t base = w << 5;
        uint32_t cov = 0;
        for (uint32_t i = lane; i < nk; i += 32) {
            const uint32_t k = p.kmin + i;
            uint32_t st = state[i];
            if (st == FROZEN_ON) { cov = 0xFFFFFFFFu; continue; }
            if (st == FROZEN_OFF) continue;
            const uint32_t m = exact_mask_global(p.H, p.L, p.NM, p.X, p.ex_key, p.n_exotic, k, w);
            const uint32_t fz = m == 0xFFFFFFFFu ? 32u : (uint32_t)__ffs(~m) - 1;   // first zero of the word
            // runs that reach back into earlier words (carry + b + 1 >= k, no zero in [0, b]) ...
            const uint32_t need = k - 1 > st ? k - 1 - st : 0u;
            uint32_t mid = need < fz ? bits_from(need) & ~bits_from(fz) : 0u;
            if (k <= 32) mid |= erode_in_word(m, k);                               // ... and those inside the word
            st = m == 0xFFFFFFFFu ? min(st + 32, k) : min((uint32_t)__clz(~m), k);
            // the tracker stops at L-k-1 and keeps the state it had there (layout positions past it are the gap)
            const int64_t j_end = (int64_t)d0 + F - (int64_t)k - 1;
            if (j_end >= (int64_t)base && j_end < (int64_t)base + 32) {
                const uint32_t b = (uint32_t)(j_end - base);
                const bool on = (mid >> b) & 1u;
                mid = (mid & ~bits_from(b + 1)) | (on ? bits_from(b + 1) : 0u);
                st = on ? FROZEN_ON : FROZEN_OFF;
            }
            state[i] = st;
            cov |= mid;
        }
        cov = __reduce_or_sync(0xFFFFFFFFu, cov);
        uint32_t in_range = 0xFFFFFFFFu;
        if (base < t_lo_pos) in_range &= bits_from(t_lo_pos - base);
        if (t_hi_pos - base < 31) in_range &= ~bits_from(t_hi_pos - base + 1);
        const uint32_t free = ~cov & in_range;
        if (free) {
            if (lane == 0) p.stop[r] = (int64_t)(base + (uint32_t)__ffs(free) - 1) - d0;
            return;
        }
    }
    if (lane == 0) p.stop[r] = W < F ? STOP_UNDECIDED : STOP_TO_END;
}

}  // namespace crf
