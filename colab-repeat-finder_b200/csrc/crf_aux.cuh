// crf_aux.cuh -- kernels around the scan: packing, result assembly, fallback sort, run-end query.
#pragma once
#include "crf_device.cuh"

namespace crf {

// ---- pack: ASCII records -> H/L/NM/X planes (replaces input_sequence.upper(), prf:33, and the
// per-base str compares of trk:53 by a 2-bit code + mask) ---------------------------------------
struct PackParams {
    const uint8_t *src;           // source bytes; record r = src[rec_src_start[r] .. + rec_len[r])
    const uint64_t *rec_src_start;
    const uint32_t *rec_len;
    const uint32_t *rec_dev_off;  // n_records (layout position of each record's first base)
    uint32_t n_records;
    uint32_t w_lo, w_hi;          // layout words this launch packs (the upload is pipelined chunk by chunk)
    uint32_t *H, *L, *NM, *X;
    uint64_t *ex_key;
    uint32_t ex_cap;
    unsigned long long *ex_count;
};

__global__ void __launch_bounds__(256) pack_kernel(const PackParams p) {
    const uint32_t w = p.w_lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= p.w_hi) return;
    const uint32_t p0 = w << 5;
    // record containing (or preceding) p0: last r with rec_dev_off[r] <= p0
    uint32_t lo = 0, hi = p.n_records ? p.n_records - 1 : 0;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (p.rec_dev_off[mid] <= p0) lo = mid; else hi = mid - 1;
    }
    uint32_t r = lo;
    uint64_t src0 = 0;
    uint32_t dev0 = 0, rec_end = 0, next_start = NOPOS;
    if (p.n_records) {
        src0 = p.rec_src_start[r];
        dev0 = p.rec_dev_off[r];
        rec_end = dev0 + p.rec_len[r];
        next_start = (r + 1 < p.n_records) ? p.rec_dev_off[r + 1] : NOPOS;
    }
    uint32_t h = 0, l = 0, nm = 0, x = 0;
#pragma unroll 4
    for (uint32_t b = 0; b < 32; ++b) {
        const uint32_t pos = p0 + b;
        if (pos >= next_start) {
            ++r;
            src0 = p.rec_src_start[r];
            dev0 = p.rec_dev_off[r];
            rec_end = dev0 + p.rec_len[r];
            next_start = (r + 1 < p.n_records) ? p.rec_dev_off[r + 1] : NOPOS;
        }
        uint32_t code, masked = 1, exo = 0;
        if (pos >= dev0 && pos < rec_end) {
            uint32_t c = p.src[src0 + (pos - dev0)];
            if (c >= 'a' && c <= 'z') c -= 32;  // upper() for ASCII (prf:33)
            if (c == 'A') { code = 0; masked = 0; }
            else if (c == 'C') { code = 1; masked = 0; }
            else if (c == 'G') { code = 2; masked = 0; }
            else if (c == 'T') { code = 3; masked = 0; }
            else if (c == 'N') { code = hash32(pos) & 3; }
            else {
                code = hash32(c * 0x9E3779B1u) & 3;  // equal letters -> equal filler code
                exo = 1;
                const unsigned long long idx = atomicAdd(p.ex_count, 1ull);
                if (idx < p.ex_cap) p.ex_key[idx] = ((uint64_t)pos << 8) | c;
            }
        } else {
            code = hash32(pos) & 3;  // inter-record gap / tail pad: masked, aperiodic filler
        }
        h |= (code >> 1) << b;
        l |= (code & 1) << b;
        nm |= masked << b;
        x |= exo << b;
    }
    p.H[w] = h;
    p.L[w] = l;
    p.NM[w] = nm;
    p.X[w] = x;
}

// ---- repack: 2-bit planes + mask as packed on the HOST (crf_pack_ascii: all records back to back, position p of the
// source = bit p & 31 of word p >> 5) -> the device layout (records separated by masked gaps, filler codes at masked
// positions).  Same result as pack_kernel on the ASCII bytes, at 0.375 B/bp of input instead of 1 B/bp. ----------------
struct RepackParams {
    const uint32_t *sH, *sL, *sN;   // source planes; word 0 holds source positions [src_base, src_base + 32)
    uint64_t src_base;              // multiple of 32
    const uint64_t *rec_src_start;  // source position of each record's first base
    const uint32_t *rec_len;
    const uint32_t *rec_dev_off;
    uint32_t n_records;
    uint32_t w_lo, w_hi;            // layout words this launch packs
    uint32_t *H, *L, *NM, *X;
};

__global__ void __launch_bounds__(256) repack_kernel(const RepackParams p) {
    const uint32_t w = p.w_lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= p.w_hi) return;
    const uint32_t p0 = w << 5;
    uint32_t h = 0, l = 0, nm = 0xFFFFFFFFu;                 // gaps and pads are masked
    if (p.n_records) {
        uint32_t lo = 0, hi = p.n_records - 1;               // last record that starts at or before p0
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (p.rec_dev_off[mid] <= p0) lo = mid; else hi = mid - 1;
        }
        const uint64_t p1 = (uint64_t)p0 + 32;
        for (uint32_t r = lo; r < p.n_records; ++r) {
            const uint32_t dev0 = p.rec_dev_off[r];
            if ((uint64_t)dev0 >= p1) break;
            const uint64_t rec_end = (uint64_t)dev0 + p.rec_len[r];
            const uint64_t a = max((uint64_t)p0, (uint64_t)dev0), b = min(p1, rec_end);
            if (a >= b) continue;
            const uint32_t nbits = (uint32_t)(b - a), place = (uint32_t)(a - p0);
            const uint64_t sbit = p.rec_src_start[r] - p.src_base + (a - dev0);
            const uint64_t wi = sbit >> 5;
            const uint32_t sh = (uint32_t)sbit & 31u;
            const uint32_t mask = nbits == 32 ? 0xFFFFFFFFu : ((1u << nbits) - 1u);
            const uint64_t wj = (sh && nbits > 32u - sh) ? wi + 1 : wi;   // never read beyond the last word that holds data
            const uint32_t eh = __funnelshift_r(p.sH[wi], p.sH[wj], sh) & mask;
            const uint32_t el = __funnelshift_r(p.sL[wi], p.sL[wj], sh) & mask;
            const uint32_t en = __funnelshift_r(p.sN[wi], p.sN[wj], sh) & mask;
            h |= eh << place;
            l |= el << place;
            nm = (nm & ~(mask << place)) | (en << place);
        }
    }
    h &= ~nm;
    l &= ~nm;
    for (uint32_t m = nm; m;) {                               // aperiodic filler at masked positions (see pack_kernel)
        const uint32_t b = __ffs(m) - 1;
        m &= m - 1;
        const uint32_t code = hash32(p0 + b) & 3;
        h |= (code >> 1) << b;
        l |= (code & 1) << b;
    }
    p.H[w] = h;
    p.L[w] = l;
    p.NM[w] = nm;
    p.X[w] = 0;
}

// ---- .2bit: the packed bases of a .2bit file -> the device layout.  Source position q is base q & 3 of byte q >> 2, the
// first base in the top two bits, T=0 C=1 A=2 G=3: with (h, l) its two bits, the planes are H = ~(h ^ l), L = ~h.  The
// N blocks arrive as the mask plane of the source positions (runs mode).  Same structure and result as repack_kernel, with
// the source planes of a word made from its 8 bytes; X = 0 (a .2bit file holds only A, C, G, T and N). ---------------------
struct TwoBitParams {
    const uint8_t *dna;             // byte 0 holds source positions [src_base, src_base + 4)
    uint64_t n_bytes;               // bytes of dna that may be read
    const uint32_t *sN;             // mask plane; word 0 = source positions [src_base, src_base + 32)
    uint64_t src_base;              // multiple of 32
    const uint64_t *rec_src_start;  // source position of each record's first base
    const uint32_t *rec_len;
    const uint32_t *rec_dev_off;
    uint32_t n_records;
    uint32_t w_lo, w_hi;            // layout words this launch packs
    uint32_t *H, *L, *NM, *X;
};

__device__ __forceinline__ uint32_t even_bits(uint64_t v) {     // bits 0, 2, 4, ... of v -> bits 0, 1, 2, ...
    v &= 0x5555555555555555ull;
    v = (v | (v >> 1)) & 0x3333333333333333ull;
    v = (v | (v >> 2)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v >> 4)) & 0x00FF00FF00FF00FFull;
    v = (v | (v >> 8)) & 0x0000FFFF0000FFFFull;
    return (uint32_t)(v | (v >> 16));
}

// the H / L planes of source word wi (bytes 8 wi .. 8 wi + 7)
__device__ __forceinline__ void twobit_planes(const TwoBitParams &p, uint64_t wi, uint32_t &H, uint32_t &L) {
    const uint64_t b0 = 8 * wi;
    const uint8_t *s = p.dna + b0;
    uint64_t x = 0;
    if (b0 + 8 <= p.n_bytes && ((uintptr_t)s & 7) == 0) {
        x = *reinterpret_cast<const uint64_t *>(s);
    } else {
        for (uint32_t j = 0; j < 8; ++j)
            if (b0 + j < p.n_bytes) x |= (uint64_t)s[j] << (8 * j);
    }
    x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);   // base j of the word -> bits 2j + 1, 2j
    x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
    const uint32_t h = even_bits(x >> 1), l = even_bits(x);
    H = ~(h ^ l);
    L = ~h;
}

__global__ void __launch_bounds__(256) twobit_pack_kernel(const TwoBitParams p) {
    const uint32_t w = p.w_lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= p.w_hi) return;
    const uint32_t p0 = w << 5;
    uint32_t h = 0, l = 0, nm = 0xFFFFFFFFu;                 // gaps and pads are masked
    if (p.n_records) {
        uint32_t lo = 0, hi = p.n_records - 1;               // last record that starts at or before p0
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (p.rec_dev_off[mid] <= p0) lo = mid; else hi = mid - 1;
        }
        const uint64_t p1 = (uint64_t)p0 + 32;
        for (uint32_t r = lo; r < p.n_records; ++r) {
            const uint32_t dev0 = p.rec_dev_off[r];
            if ((uint64_t)dev0 >= p1) break;
            const uint64_t rec_end = (uint64_t)dev0 + p.rec_len[r];
            const uint64_t a = max((uint64_t)p0, (uint64_t)dev0), b = min(p1, rec_end);
            if (a >= b) continue;
            const uint32_t nbits = (uint32_t)(b - a), place = (uint32_t)(a - p0);
            const uint64_t sbit = p.rec_src_start[r] - p.src_base + (a - dev0);
            const uint64_t wi = sbit >> 5;
            const uint32_t sh = (uint32_t)sbit & 31u;
            const uint32_t mask = nbits == 32 ? 0xFFFFFFFFu : ((1u << nbits) - 1u);
            const uint64_t wj = (sh && nbits > 32u - sh) ? wi + 1 : wi;
            uint32_t hi_, li_, hj, lj;
            twobit_planes(p, wi, hi_, li_);
            if (wj != wi) twobit_planes(p, wj, hj, lj); else { hj = hi_; lj = li_; }
            const uint32_t eh = __funnelshift_r(hi_, hj, sh) & mask;
            const uint32_t el = __funnelshift_r(li_, lj, sh) & mask;
            const uint32_t en = __funnelshift_r(p.sN[wi], p.sN[wj], sh) & mask;
            h |= eh << place;
            l |= el << place;
            nm = (nm & ~(mask << place)) | (en << place);
        }
    }
    h &= ~nm;
    l &= ~nm;
    for (uint32_t m = nm; m;) {                               // aperiodic filler at masked positions (see pack_kernel)
        const uint32_t b = __ffs(m) - 1;
        m &= m - 1;
        const uint32_t code = hash32(p0 + b) & 3;
        h |= (code >> 1) << b;
        l |= (code & 1) << b;
    }
    p.H[w] = h;
    p.L[w] = l;
    p.NM[w] = nm;
    p.X[w] = 0;
}

// ---- BAM: 4-bit codes (=ACMGRSVTWYHKDBN) -> the device layout.  Source position q is nibble q & 1 of byte q >> 1, high
// nibble first.  A code c gives H = (c & 0b1100) != 0, L = (c & 0b1010) != 0 (A = 1, C = 2, G = 4, T = 8 -> codes 0..3),
// and NM wherever c is not 1, 2, 4 or 8, so N and the other codes are masked without a list from the host (the exotic ones
// then get their letters from exotic_apply_kernel).  Same structure and result as twobit_pack_kernel. -------------------
struct NibbleParams {
    const uint8_t *nib;             // byte 0 holds source positions [src_base, src_base + 2)
    uint64_t n_bytes;               // bytes of nib that may be read
    uint64_t src_base;              // multiple of 32
    const uint64_t *rec_src_start;  // source position of each record's first base
    const uint32_t *rec_len;
    const uint32_t *rec_dev_off;
    uint32_t n_records;
    uint32_t w_lo, w_hi;            // layout words this launch packs
    uint32_t *H, *L, *NM, *X;
};

__device__ __forceinline__ uint32_t fourth_bits(uint64_t v) {   // bits 0, 4, 8, ... of v -> bits 0, 1, 2, ...
    v &= 0x1111111111111111ull;
    v = (v | (v >> 3)) & 0x0303030303030303ull;
    v = (v | (v >> 6)) & 0x000F000F000F000Full;
    v = (v | (v >> 12)) & 0x000000FF000000FFull;
    return (uint32_t)((v | (v >> 24)) & 0xFFFFu);
}

// H, L and NM of 16 source positions from their 8 bytes (x: byte j in bits 8j..8j+7)
__device__ __forceinline__ void nibble_planes16(uint64_t x, uint32_t &H, uint32_t &L, uint32_t &NM) {
    x = ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);   // position i -> bits 4i .. 4i + 3
    const uint64_t b0 = x, b1 = x >> 1, b2 = x >> 2, b3 = x >> 3;
    const uint64_t any = b0 | b1 | b2 | b3, two = (b0 & (b1 | b2 | b3)) | (b1 & (b2 | b3)) | (b2 & b3);
    H = fourth_bits(b2 | b3);
    L = fourth_bits(b1 | b3);
    NM = fourth_bits(~(any & ~two));
}

// the H / L / NM planes of source word wi (bytes 16 wi .. 16 wi + 15); bytes past n_bytes read as code 0 (masked)
__device__ __forceinline__ void nibble_planes(const NibbleParams &p, uint64_t wi, uint32_t &H, uint32_t &L, uint32_t &NM) {
    const uint64_t b0 = 16 * wi;
    const uint8_t *s = p.nib + b0;
    uint64_t x0 = 0, x1 = 0;
    if (b0 + 16 <= p.n_bytes && ((uintptr_t)s & 15) == 0) {
        const uint4 v = *reinterpret_cast<const uint4 *>(s);
        x0 = ((uint64_t)v.y << 32) | v.x;
        x1 = ((uint64_t)v.w << 32) | v.z;
    } else {
        for (uint32_t j = 0; j < 16; ++j)
            if (b0 + j < p.n_bytes) (j < 8 ? x0 : x1) |= (uint64_t)s[j] << (8 * (j & 7));
    }
    uint32_t h0, l0, n0, h1, l1, n1;
    nibble_planes16(x0, h0, l0, n0);
    nibble_planes16(x1, h1, l1, n1);
    H = h0 | (h1 << 16);
    L = l0 | (l1 << 16);
    NM = n0 | (n1 << 16);
}

__global__ void __launch_bounds__(256) nibble_pack_kernel(const NibbleParams p) {
    const uint32_t w = p.w_lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= p.w_hi) return;
    const uint32_t p0 = w << 5;
    uint32_t h = 0, l = 0, nm = 0xFFFFFFFFu;                 // gaps and pads are masked
    if (p.n_records) {
        uint32_t lo = 0, hi = p.n_records - 1;               // last record that starts at or before p0
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (p.rec_dev_off[mid] <= p0) lo = mid; else hi = mid - 1;
        }
        const uint64_t p1 = (uint64_t)p0 + 32;
        for (uint32_t r = lo; r < p.n_records; ++r) {
            const uint32_t dev0 = p.rec_dev_off[r];
            if ((uint64_t)dev0 >= p1) break;
            const uint64_t rec_end = (uint64_t)dev0 + p.rec_len[r];
            const uint64_t a = max((uint64_t)p0, (uint64_t)dev0), b = min(p1, rec_end);
            if (a >= b) continue;
            const uint32_t nbits = (uint32_t)(b - a), place = (uint32_t)(a - p0);
            const uint64_t sbit = p.rec_src_start[r] - p.src_base + (a - dev0);
            const uint64_t wi = sbit >> 5;
            const uint32_t sh = (uint32_t)sbit & 31u;
            const uint32_t mask = nbits == 32 ? 0xFFFFFFFFu : ((1u << nbits) - 1u);
            const uint64_t wj = (sh && nbits > 32u - sh) ? wi + 1 : wi;
            uint32_t hi_, li_, ni_, hj, lj, nj;
            nibble_planes(p, wi, hi_, li_, ni_);
            if (wj != wi) nibble_planes(p, wj, hj, lj, nj); else { hj = hi_; lj = li_; nj = ni_; }
            const uint32_t eh = __funnelshift_r(hi_, hj, sh) & mask;
            const uint32_t el = __funnelshift_r(li_, lj, sh) & mask;
            const uint32_t en = __funnelshift_r(ni_, nj, sh) & mask;
            h |= eh << place;
            l |= el << place;
            nm = (nm & ~(mask << place)) | (en << place);
        }
    }
    h &= ~nm;
    l &= ~nm;
    for (uint32_t m = nm; m;) {                               // aperiodic filler at masked positions (see pack_kernel)
        const uint32_t b = __ffs(m) - 1;
        m &= m - 1;
        const uint32_t code = hash32(p0 + b) & 3;
        h |= (code >> 1) << b;
        l |= (code & 1) << b;
    }
    p.H[w] = h;
    p.L[w] = l;
    p.NM[w] = nm;
    p.X[w] = 0;
}

// runs mode of a packed load: the mask plane from the sorted runs of masked positions [runs[2i], runs[2i+1]); one warp per
// run (its lanes stride over the run's words; a genome has a few hundred long N blocks, a read set millions of single N's)
__global__ void __launch_bounds__(256) mask_runs_kernel(const uint64_t *runs, uint32_t n_runs, uint32_t *NM) {
    const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (r >= n_runs) return;
    const uint64_t a = runs[2 * r], b = runs[2 * r + 1];
    const uint64_t w_first = a >> 5, w_last = (b - 1) >> 5;
    for (uint64_t w = w_first + lane; w <= w_last; w += 32) {
        uint32_t m = 0xFFFFFFFFu;
        if (w == w_first) m &= 0xFFFFFFFFu << (uint32_t)(a & 31);
        if (w == w_last && (b & 31)) m &= (1u << (uint32_t)(b & 31)) - 1u;
        if (w == w_first || w == w_last) atomicOr(&NM[w], m);   // an edge word may be shared with the neighbouring run
        else NM[w] = m;
    }
}

// exotic symbols of a packed load: (layout position << 8 | letter), already sorted: mark them in X and give them the
// letter's filler code (equal letters -> equal codes, pack_kernel)
__global__ void __launch_bounds__(256) exotic_apply_kernel(const uint64_t *ex_key, uint32_t n, uint32_t *H, uint32_t *L, uint32_t *X) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t key = ex_key[i];
    const uint32_t pos = (uint32_t)(key >> 8), c = (uint32_t)(key & 0xFF);
    const uint32_t code = hash32(c * 0x9E3779B1u) & 3, w = pos >> 5, bit = 1u << (pos & 31);
    if (code >> 1) atomicOr(&H[w], bit); else atomicAnd(&H[w], ~bit);
    if (code & 1) atomicOr(&L[w], bit); else atomicAnd(&L[w], ~bit);
    atomicOr(&X[w], bit);
}

// ---- assembly: tile segments -> one (start, end)-sorted list --------------------------------
// exclusive prefix sum of tile_cnt (single block, four tiles per thread and step; n_tiles is tens of
// thousands at most, the arrays are allocated with slack for the vector loads)
__global__ void __launch_bounds__(1024) tile_offsets_kernel(const uint32_t *tile_cnt, uint32_t *tile_off,
                                                            uint32_t n_tiles, unsigned long long *counters) {
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_tiles; base += 4096) {
        const uint32_t i = base + 4 * tid;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (i < n_tiles) v = *reinterpret_cast<const uint4 *>(tile_cnt + i);
        if (i + 1 >= n_tiles) v.y = 0;
        if (i + 2 >= n_tiles) v.z = 0;
        if (i + 3 >= n_tiles) v.w = 0;
        if (i >= n_tiles) v.x = 0;
        const uint32_t mine = v.x + v.y + v.z + v.w;
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (uint32_t)o) incl += t;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        uint32_t woff = 0, total = 0;
        for (uint32_t j = 0; j < 32; ++j) {
            const uint32_t t = warp_sum[j];
            if (j < warp) woff += t;
            total += t;
        }
        const uint32_t carry = carry_s;
        const uint32_t e0 = carry + woff + incl - mine;
        if (i < n_tiles) tile_off[i] = e0;
        if (i + 1 < n_tiles) tile_off[i + 1] = e0 + v.x;
        if (i + 2 < n_tiles) tile_off[i + 2] = e0 + v.x + v.y;
        if (i + 3 < n_tiles) tile_off[i + 3] = e0 + v.x + v.y + v.z;
        __syncthreads();
        if (tid == 0) carry_s = carry + total;
        __syncthreads();
    }
    if (tid == 0) {
        tile_off[n_tiles] = carry_s;
        const unsigned long long spill = counters[C_SPILL];
        counters[C_TOTAL] = (unsigned long long)carry_s + spill;
    }
}

// Results that overflowed a tile's sorted-output slots ("spill") are sorted on their own and merged
// with the tile-ordered main list while it is gathered: final index = own index + rank in the other
// list.  Up to SPILL_SMALL rows are sorted by one block in shared memory (no host round trip); more
// than that, the host sorts the spill list with the global bitonic network and gathers again.
constexpr uint32_t SPILL_SMALL = 4096;

__device__ __forceinline__ bool row_less(uint64_t ka, uint16_t va, uint64_t kb, uint16_t vb) {
    return ka < kb || (ka == kb && va < vb);
}

__global__ void __launch_bounds__(1024) spill_sort_small_kernel(uint64_t *spill_key, uint16_t *spill_k, uint32_t spill_cap,
                                                                const unsigned long long *counters) {
    __shared__ uint64_t sk[SPILL_SMALL];
    __shared__ uint16_t sv[SPILL_SMALL];
    const unsigned long long n64 = counters[C_SPILL];
    if (n64 < 2 || n64 > SPILL_SMALL || n64 > spill_cap) return;
    const uint32_t n = (uint32_t)n64;
    uint32_t np = 1;
    while (np < n) np <<= 1;
    for (uint32_t i = threadIdx.x; i < np; i += blockDim.x) {
        sk[i] = i < n ? spill_key[i] : ~0ull;
        sv[i] = i < n ? spill_k[i] : (uint16_t)0xFFFF;
    }
    __syncthreads();
    for (uint32_t kk = 2; kk <= np; kk <<= 1)
        for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
            for (uint32_t i = threadIdx.x; i < np; i += blockDim.x) {
                const uint32_t ixj = i ^ j;
                if (ixj > i) {
                    const bool asc = (i & kk) == 0;
                    const uint64_t a = sk[i], b = sk[ixj];
                    const uint16_t va = sv[i], vb = sv[ixj];
                    if (row_less(b, vb, a, va) == asc) { sk[i] = b; sk[ixj] = a; sv[i] = vb; sv[ixj] = va; }
                }
            }
            __syncthreads();
        }
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        spill_key[i] = sk[i];
        spill_k[i] = sv[i];
    }
}

struct GatherParams {
    const uint64_t *stage_key;
    const uint16_t *stage_k;
    const uint32_t *tile_cnt, *tile_base, *tile_off;
    const uint64_t *spill_key;
    const uint16_t *spill_k;
    uint64_t *fin_key;
    uint16_t *fin_k;
    uint32_t n_tiles, fin_cap, stage_cap, spill_cap;
    uint32_t tile_words;     // words per tile (a spilled row's tile = (start >> 5) / tile_words)
    uint32_t spill_sorted;   // host says: the spill list is sorted even though it is longer than SPILL_SMALL
    const unsigned long long *counters;
};

// one warp per tile copies its sorted segment to its final place, leaving room for the spilled
// rows that sort before each element; the spilled rows are placed by the tail of the grid
__global__ void __launch_bounds__(256) gather_kernel(const GatherParams g) {
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (g.counters[C_STAGE] > g.stage_cap || g.counters[C_TOTAL] > g.fin_cap) return;  // host re-runs
    const unsigned long long nspill64 = g.counters[C_SPILL];
    if (nspill64 > g.spill_cap) return;
    if (nspill64 > SPILL_SMALL && !g.spill_sorted) return;  // host sorts the spill list and gathers again
    const uint32_t m = (uint32_t)nspill64;
    if (warp_global < g.n_tiles) {
        const uint32_t n = g.tile_cnt[warp_global], src = g.tile_base[warp_global], dst = g.tile_off[warp_global];
        for (uint32_t i = lane; i < n; i += 32) {
            const uint64_t key = g.stage_key[src + i];
            const uint16_t kk = g.stage_k[src + i];
            uint32_t lo = 0, hi = m;  // spilled rows that sort before this one
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (row_less(g.spill_key[mid], g.spill_k[mid], key, kk)) lo = mid + 1; else hi = mid;
            }
            g.fin_key[dst + i + lo] = key;
            g.fin_k[dst + i + lo] = kk;
        }
    }
    if (m) {
        const uint32_t stride = gridDim.x * blockDim.x;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
            const uint64_t key = g.spill_key[i];
            const uint16_t kk = g.spill_k[i];
            const uint32_t t = (uint32_t)(key >> 37) / g.tile_words;
            const uint32_t n = g.tile_cnt[t], src = g.tile_base[t];
            uint32_t lo = 0, hi = n;  // rows of its tile's segment that sort before it
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (row_less(g.stage_key[src + mid], g.stage_k[src + mid], key, kk)) lo = mid + 1; else hi = mid;
            }
            g.fin_key[g.tile_off[t] + lo + i] = key;
            g.fin_k[g.tile_off[t] + lo + i] = kk;
        }
    }
}

// layout coordinates -> (record, start, end, k)  (the re-offsetting of prf:81, per record); with an
// output map (partitioned loads) the unit's record id / offset are applied and open-ended results counted
struct TranslateParams {
    const uint64_t *fin_key;
    const uint16_t *fin_k;
    const uint32_t *rec_dev_off, *rec_len;
    const uint32_t *map_rec, *map_shift;   // nullable
    const uint8_t *map_open;               // nullable
    uint32_t n_records, fin_cap;
    unsigned long long *counters;
    uint32_t *o_rec, *o_start, *o_end, *o_k;
    uint32_t *open_rows;                   // open_cap x 5: row, record, start, end, k of open-ended results
    uint32_t open_cap;                     // (the host grows the list and translates again when it was too short)
};

constexpr uint32_t OPEN_CAP_INITIAL = 256;

__global__ void __launch_bounds__(256) translate_kernel(const TranslateParams t) {
    const unsigned long long n = t.counters[C_TOTAL];
    if (n > t.fin_cap) return;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t key = t.fin_key[i];
        const uint32_t st = (uint32_t)(key >> 32), en = (uint32_t)key;
        uint32_t lo = 0, hi = t.n_records - 1;
        while (lo < hi) {
            const uint32_t mid = (lo + hi + 1) >> 1;
            if (t.rec_dev_off[mid] <= st) lo = mid; else hi = mid - 1;
        }
        const uint32_t d0 = t.rec_dev_off[lo];
        const uint32_t shift = t.map_shift ? t.map_shift[lo] : 0u;
        const uint32_t orec = t.map_rec ? t.map_rec[lo] : lo;
        t.o_rec[i] = orec;
        t.o_start[i] = st - d0 + shift;
        t.o_end[i] = en - d0 + shift;
        t.o_k[i] = t.fin_k[i];
        if (t.map_open && t.map_open[lo] && en - d0 == t.rec_len[lo]) {  // reached the end of an open-ended record
            const unsigned long long slot = atomicAdd(t.counters + C_OPEN, 1ull);
            if (slot < t.open_cap) {
                uint32_t *row = t.open_rows + 5 * slot;
                row[0] = i; row[1] = orec; row[2] = st - d0 + shift; row[3] = en - d0 + shift; row[4] = t.fin_k[i];
            }
        }
    }
}

// ---- min_repeats == 1 only: r_min may be k-1, and a run of exactly k-1 matches leaves the motif's last base
// S[st+k-1] (the mismatch position itself) untested; an 'N' there drops the row (trk:83).  The scan kernel never
// sees this case in ordinary scans (r_min >= k), so it is settled here, on the sorted list, by one block that
// compacts in place chunk by chunk (a row only ever moves to a lower index).  Rare mode, not tuned. ---------------
__global__ void __launch_bounds__(1024) single_copy_filter_kernel(uint64_t *key, uint16_t *kk, const uint32_t *NM,
                                                                  const uint32_t *X, uint32_t n_words, uint32_t fin_cap,
                                                                  unsigned long long *counters) {
    __shared__ uint32_t warp_total[32];
    const unsigned long long n64 = counters[C_STAGE] + counters[C_SPILL];
    if (counters[C_STAGE] > fin_cap || counters[C_SPILL] > fin_cap || n64 > fin_cap) return;   // host re-runs
    const uint32_t n = (uint32_t)n64, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t out = 0;
    for (uint32_t chunk = 0; chunk < n; chunk += 1024) {
        const uint32_t i = chunk + threadIdx.x;
        uint64_t key_i = 0;
        uint16_t k_i = 0;
        bool keep = false;
        if (i < n) {
            key_i = key[i];
            k_i = kk[i];
            const uint32_t st = (uint32_t)(key_i >> 32), en = (uint32_t)key_i;
            keep = true;
            if (en - st == 2u * k_i - 1u) {
                const uint32_t q = st + k_i - 1u, w = q >> 5;
                if (w < n_words && (((NM[w] & ~X[w]) >> (q & 31)) & 1u)) keep = false;
            }
        }
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, keep);
        if (lane == 0) warp_total[warp] = __popc(bal);
        __syncthreads();                                  // every row of the chunk is in registers now
        uint32_t before = 0, total = 0;
        for (uint32_t w = 0; w < 32; ++w) {
            const uint32_t c = warp_total[w];
            before += w < warp ? c : 0u;
            total += c;
        }
        if (keep) {
            const uint32_t pos = out + before + __popc(bal & ((1u << lane) - 1u));
            key[pos] = key_i;
            kk[pos] = k_i;
        }
        out += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) counters[C_TOTAL] = out;
}

// ---- fallback ordering: global bitonic network on (key, k); n_pow2 elements, tail padded with
// all-ones keys.  Only used when a tile overflowed its sorted-output slots, and for the (tiny)
// list of exotic symbols. -------------------------------------------------------------------
__global__ void __launch_bounds__(256) bitonic_step_kernel(uint64_t *key, uint16_t *val, uint32_t n_pow2, uint32_t j,
                                                           uint32_t kk) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pow2) return;
    const uint32_t ixj = i ^ j;
    if (ixj <= i) return;
    const bool asc = (i & kk) == 0;
    const uint64_t a = key[i], b = key[ixj];
    const uint16_t va = val ? val[i] : 0, vb = val ? val[ixj] : 0;
    const bool gt = (a > b) || (a == b && va > vb);
    if (gt == asc) {
        key[i] = b;
        key[ixj] = a;
        if (val) { val[i] = vb; val[ixj] = va; }
    }
}
__global__ void __launch_bounds__(256) fill_u64_kernel(uint64_t *dst, uint64_t v, uint32_t from, uint32_t to) {
    const uint32_t i = from + blockIdx.x * blockDim.x + threadIdx.x;
    if (i < to) dst[i] = v;
}

// ---- run-end query (crf_run_end): one block walks 256 words per step ---------------------------
__global__ void __launch_bounds__(THREADS) run_end_kernel(const ScanParams p, uint32_t k, uint32_t pos, uint32_t *out) {
    __shared__ uint32_t minpos;
    const uint32_t tid = threadIdx.x;
    uint32_t wcur = pos >> 5;
    for (;;) {
        if (tid == 0) minpos = NOPOS;
        __syncthreads();
        const uint32_t w = wcur + tid;
        uint32_t m = (w < p.n_words) ? exact_mask(p, k, w) : 0u;
        if (w == (pos >> 5)) m |= (1u << (pos & 31)) - 1u;
        if (m != 0xFFFFFFFFu) atomicMin(&minpos, (w << 5) + (__ffs(~m) - 1));
        __syncthreads();
        const uint32_t r = minpos;
        __syncthreads();
        if (r != NOPOS) {
            if (tid == 0) *out = r;
            return;
        }
        wcur += THREADS;
    }
}

}  // namespace crf
