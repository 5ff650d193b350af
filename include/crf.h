/*
 * crf.h -- C ABI of libcrf.so, the B200 (sm_100a) perfect-tandem-repeat scan.
 *
 * The reference (broadinstitute/colab-repeat-finder) has no FFI of its own: its hot path is the
 * Python function detect_repeats() (perfect_repeat_finder.py:10-81) driving one
 * PerfectRepeatTracker per motif size (utils/perfect_repeat_tracker.py:3-105).  These entry
 * points are what a ctypes binding under that function binds instead of the tracker loop
 * (INTEGRATION.md shows the stub).  Plain C types only, no exceptions cross the boundary, every
 * call returns an int status (0 = ok) and leaves a message for crf_last_error() on failure.
 *
 * Threading: one crf_ctx per GPU; calls on one context (and on its sequences) must be
 * serialised by the caller.  Different contexts may be driven from different threads/processes.
 *
 * Coordinates are 0-based, half-open, per record -- the (start_0based, end) convention of
 * perfect_repeat_finder.py:81.
 */
#ifndef CRF_H
#define CRF_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRF_OK 0
#define CRF_ERR_CUDA 1        /* a CUDA runtime call failed                               */
#define CRF_ERR_ARG 2         /* invalid argument (the ValueError cases of prf:23-30 too)  */
#define CRF_ERR_NOMEM 3
#define CRF_ERR_UNSUPPORTED 4 /* valid for the reference, not implemented here (loud)     */
#define CRF_ERR_CAPACITY 5    /* caller-provided buffer too small                          */
#define CRF_ERR_IO 6          /* a file could not be written in full                       */

typedef struct crf_ctx crf_ctx; /* one CUDA device + stream + scratch                      */
typedef struct crf_seq crf_seq; /* a set of records resident in HBM as packed bit-planes   */

/* Last error message of the calling thread ("" if none). */
const char *crf_last_error(void);
/* ABI version of the library (bumped on incompatible change). */
int crf_abi_version(void);

/* ---- context ---------------------------------------------------------------------------- */
int crf_ctx_create(int device, crf_ctx **ctx);
/* Destroy the context's sequences and exchange blocks first: they keep pointers into it. */
int crf_ctx_destroy(crf_ctx *ctx);
/* Run all work of this context on `cuda_stream` (a cudaStream_t; NULL = the context's own).  Switching waits for the work
 * queued on the previous stream. */
int crf_ctx_set_stream(crf_ctx *ctx, void *cuda_stream);
int crf_ctx_synchronize(crf_ctx *ctx);

/* ---- sequence upload ----------------------------------------------------------------------
 * Replaces the `input_sequence` str handed to detect_repeats (prf:10,33): `bases` holds
 * n_records records back to back, record r = bases[offsets[r] .. offsets[r+1]); any case, any
 * byte value.  Upper-casing (prf:33) happens on the device.  The records are packed into two
 * 2-bit planes plus a not-ACGT mask; runs never cross a record boundary.  `max_motif_cap` is the
 * largest max_motif_size later scans may use (it sizes the inter-record gap and the halo).
 * bases_on_device != 0: `bases` is a device pointer (offsets stay on the host).
 */
int crf_seq_load_ascii(crf_ctx *ctx, const uint8_t *bases, const uint64_t *offsets, uint32_t n_records,
                       uint32_t max_motif_cap, int bases_on_device, crf_seq **seq);
/* Same, with each record given as its own (start, length) range of `bases` (ranges may overlap:
 * partition units share their halo) and, optionally, the sub-range [own_lo, own_hi) of each record
 * whose run STARTS this load reports (NULL, NULL = whole records).  A run that starts in the owned
 * range is followed to its end anywhere in the record.  See DESIGN.md "Multi-GPU". */
int crf_seq_load_ascii_ranges(crf_ctx *ctx, const uint8_t *bases, const uint64_t *starts, const uint64_t *lengths,
                              const uint64_t *own_lo, const uint64_t *own_hi, uint32_t n_records,
                              uint32_t max_motif_cap, int bases_on_device, crf_seq **seq);
/* The same from planes packed on the HOST (crf_pack_ascii, or crf_fasta_packed at ingest): 0.375 bytes per base cross
 * PCIe instead of 1.  All records back to back in one position space: position p = bit p & 31 of word p >> 5 of
 *   H, L : the two bits of the base code (A=00 C=01 G=10 T=11; anything at masked positions),
 *   NM   : 1 = not A/C/G/T after upper-casing (N, IUPAC codes, anything else),
 * ceil(total / 32) words each, plus the list of symbols that are neither ACGT nor N ("exotic": only the literal N never
 * matches, utils/perfect_repeat_tracker.py:53; other letters compare by equality) as (position << 8 | upper-cased byte),
 * ascending.  Record r = positions [offsets[r], offsets[r+1]) resp. [starts[r], starts[r] + lengths[r]).  The device
 * re-lays the bits out with the inter-record gaps and filler codes (repack_kernel); results are identical to the ASCII
 * load of the same text.  planes_on_device != 0: H, L, NM (not exotic / offsets) are device pointers. */
int crf_seq_load_packed(crf_ctx *ctx, const uint32_t *H, const uint32_t *L, const uint32_t *NM, const uint64_t *exotic,
                        uint64_t n_exotic, const uint64_t *offsets, uint32_t n_records, uint32_t max_motif_cap,
                        int planes_on_device, crf_seq **seq);
int crf_seq_load_packed_ranges(crf_ctx *ctx, const uint32_t *H, const uint32_t *L, const uint32_t *NM,
                               const uint64_t *exotic, uint64_t n_exotic, const uint64_t *starts, const uint64_t *lengths,
                               const uint64_t *own_lo, const uint64_t *own_hi, uint32_t n_records, uint32_t max_motif_cap,
                               int planes_on_device, crf_seq **seq);
/* The same with the mask handed over as RUNS instead of a plane: runs[2i], runs[2i+1] = the i-th maximal block of masked
 * positions [from, to), ascending and disjoint (crf_mask_runs makes them from an NM plane).  A genome's N's are a few hundred
 * long blocks, so 0.25 bytes per base cross PCIe; the device rebuilds the plane (mask_runs_kernel). */
int crf_seq_load_packed_runs(crf_ctx *ctx, const uint32_t *H, const uint32_t *L, const uint64_t *runs, uint64_t n_runs,
                             const uint64_t *exotic, uint64_t n_exotic, const uint64_t *offsets, uint32_t n_records,
                             uint32_t max_motif_cap, int planes_on_device, crf_seq **seq);
int crf_seq_load_packed_runs_ranges(crf_ctx *ctx, const uint32_t *H, const uint32_t *L, const uint64_t *runs, uint64_t n_runs,
                                    const uint64_t *exotic, uint64_t n_exotic, const uint64_t *starts,
                                    const uint64_t *lengths, const uint64_t *own_lo, const uint64_t *own_hi,
                                    uint32_t n_records, uint32_t max_motif_cap, int planes_on_device, crf_seq **seq);
/* Records of a .2bit file (crf_fasta_twobit), loaded from the file's packed bytes: record r holds offsets[r + 1] -
 * offsets[r] bases packed from byte rec_byte[r] of dna, its N blocks among the ascending, disjoint runs [runs[2i],
 * runs[2i+1]) of the position space of offsets (runs outside [offsets[0], offsets[n_records]) are ignored, so a load of
 * some of the records takes the whole file's list).  The byte span the records cover (headers between them included) goes
 * up at 0.25 B/bp, in chunks on a second stream while twobit_pack_kernel lays out the words whose bytes have arrived; the
 * records may not share bytes.  The rows equal those of crf_seq_load_ascii on the decoded text (crf_fasta_data).
 * dna_on_device != 0: dna is a device pointer to the file's bytes (rec_byte, offsets and runs stay host arrays). */
int crf_seq_load_2bit(crf_ctx *ctx, const uint8_t *dna, const uint64_t *rec_byte, const uint64_t *offsets, uint32_t n_records,
                      const uint64_t *runs, uint64_t n_runs, uint32_t max_motif_cap, int dna_on_device, crf_seq **seq);
/* Reads of a BAM file (crf_fasta_nibbles), loaded from their 4-bit codes: record r holds offsets[r + 1] - offsets[r] bases,
 * base i in nibble i & 1 (high nibble first) of byte rec_byte[r] + i / 2 of nib, codes =ACMGRSVTWYHKDBN (A = 1, C = 2,
 * G = 4, T = 8, N = 15).  Every code other than A, C, G, T is masked; the exotic list (position in the space of offsets
 * << 8 | letter, ascending; entries outside [offsets[0], offsets[n_records]) are ignored, so a load of some of the records
 * takes the whole file's list) gives the codes other than A, C, G, T and N their letters, as crf_seq_load_packed does.  The
 * byte span the records cover goes up at 0.5 B/bp, in chunks on a second stream while nibble_pack_kernel lays out the
 * words whose bytes have arrived.  The rows equal those of crf_seq_load_ascii on the decoded text (crf_fasta_data).
 * nib_on_device != 0: nib is a device pointer (rec_byte, offsets and exotic stay host arrays). */
int crf_seq_load_nibbles(crf_ctx *ctx, const uint8_t *nib, const uint64_t *rec_byte, const uint64_t *offsets,
                         uint32_t n_records, const uint64_t *exotic, uint64_t n_exotic, uint32_t max_motif_cap,
                         int nib_on_device, crf_seq **seq);
/* Host only: the maximal runs of set bits of an NM plane over [0, n_bases) (threaded).  *n_runs = how many there are
 * (CRF_ERR_CAPACITY if more than cap pairs: call again with a longer list). */
int crf_mask_runs(const uint32_t *NM, uint64_t n_bases, uint32_t n_threads, uint64_t *runs, uint64_t cap, uint64_t *n_runs);
/* Host-only packer for the above (threaded; AVX2 when the CPU has it).  H, L, NM: ceil(n_bases / 32) words each, written
 * in full (positions beyond n_bases are masked).  exotic: room for exotic_cap entries; *n_exotic = how many there are
 * (CRF_ERR_CAPACITY if more than exotic_cap: call again with a longer list).  n_threads = 0: up to 16. */
int crf_pack_ascii(const uint8_t *bases, uint64_t n_bases, uint32_t n_threads, uint32_t *H, uint32_t *L, uint32_t *NM,
                   uint64_t *exotic, uint64_t exotic_cap, uint64_t *n_exotic);
int crf_seq_destroy(crf_seq *seq);
/* Layout positions one load can hold: the sum over its records of (length + max_motif_cap) must not exceed this
 * (positions are 32-bit on the device); callers with more split the records over several loads.  A single record
 * longer than this is cut into units (owned range, one base of left context, a halo of at least one qualifying
 * repeat) that go to several *_ranges loads with own_lo / own_hi; each load maps its units to themselves with
 * crf_seq_set_output_map (out_record = the caller's unit number, out_shift = NULL), so rows stay unit-relative and
 * the caller adds each unit's 64-bit origin; open-ended rows are followed into the next unit with crf_run_end and
 * patched with crf_patch_end (crf_b200/multi.py does this; crf_write_rows_at prints the sums). */
uint64_t crf_load_limit(uint32_t max_motif_cap);
/* Optional, for partitioned loads: report record r of this load as record out_record[r] with start/end
 * shifted by out_shift[r] (a unit's offset inside its chromosome), and count as "open" every result that
 * ends exactly at the end of a record flagged in open_ended[r] (the unit's data stops before the
 * chromosome does, so the run may continue: crf_scan_stats().n_open, see crf_run_end).  NULLs reset.
 * Shifted coordinates must fit 32 bits (CRF_ERR_UNSUPPORTED otherwise): for units of a chromosome longer than
 * 2^32 bases, map every unit to a record number of its own with no shift and add the unit's origin on the host
 * (see crf_load_limit). */
int crf_seq_set_output_map(crf_seq *seq, const uint32_t *out_record, const uint64_t *out_shift,
                           const uint8_t *open_ended);

typedef struct {
    uint64_t n_records;
    uint64_t total_bases;  /* sum of record lengths                                    */
    uint64_t layout_bases; /* device layout incl. inter-record gaps                    */
    uint64_t packed_bytes; /* bytes of the two base planes + mask plane (algorithmic)   */
    uint64_t n_exotic;     /* symbols other than A,C,G,T,N after upper-casing           */
    uint32_t max_motif_cap;
    uint32_t reserved;
    double load_ms;        /* device time of the last upload+pack                       */
} crf_seq_info_t;
int crf_seq_info(const crf_seq *seq, crf_seq_info_t *info);

/* ---- scan ----------------------------------------------------------------------------------
 * One call = the whole of prf:49-81 for every record: all motif sizes in
 * [min_motif_size, max_motif_size], filters min_repeats / min_span (trk:86,91), primitivity
 * (trk:98, 108-142), ordering by (record, start, end) (prf:81).  Results stay in HBM until
 * fetched.  The argument checks and messages of prf:23-30 map to CRF_ERR_ARG.
 * min_repeats == 1 (trk:86-91 then lets a mismatch position with fewer than k-1 matches before it emit only
 * through Python's negative-index wrap-around at position 0): the scan returns every maximal run of at least
 * max(min_span - k, k - 1) matches whose motif is N-free and primitive -- all the reference reports except the
 * (at most one per motif size) wrap-around candidates of position 0 and the early-break selection of interval
 * mode, which the caller adds from the sequence ends (crf_b200/api.py, O(max_motif_size^2) symbol compares).
 * min_repeats == 1 with min_motif_size == 1 and min_span == 1 (every base is a "repeat") is CRF_ERR_UNSUPPORTED.
 */
/* keep runs whose motif is not primitive too (used to find where the reference's interval-mode
 * loop stops, prf:70-74: is_in_middle_of_repeat() does not look at the motif) */
#define CRF_SCAN_NO_PRIMITIVITY 1u
/* which scan kernel (same results, different scheduling; default = the library's choice): tiles owned by warps, no
 * block-wide barrier (csrc/crf_scan_warp.cuh), or tiles owned by 256-thread blocks (csrc/crf_scan.cuh) */
#define CRF_SCAN_WARP_TILES 2u
#define CRF_SCAN_BLOCK_TILES 4u
#define CRF_SCAN_TWO_STRIPS 8u   /* block tiles with two strips per thread (131 kbp tiles) */
/* bits 16..31: profiling switches (results are NOT valid when set): 1<<16 = fast phase only */
#define CRF_SCAN_DEBUG_FAST_ONLY (1u << 16)
#define CRF_SCAN_DEBUG_NO_SUP (1u << 17)   /* tuning: no homopolymer suppression in the filters (results stay valid) */

typedef struct {
    uint32_t min_motif_size;
    uint32_t max_motif_size;
    uint32_t min_repeats;
    uint32_t min_span;
    /* test / tuning knobs; 0 = library default */
    uint32_t words_per_thread; /* tile shape: 8 or 16 32-base words per thread            */
    uint32_t tile_out_cap;     /* per-tile sorted-output slots before spilling           */
    uint32_t walk_limit_words; /* words a single thread walks before the block takes over */
    uint32_t result_cap;       /* initial result capacity (grown and re-run on overflow)  */
    uint32_t flags;            /* CRF_SCAN_* bits                                         */
} crf_scan_params;

int crf_scan(crf_seq *seq, const crf_scan_params *params, uint64_t *n_results);

/* Copy the results of the last scan into caller arrays of `capacity` entries each
 * (dst_on_device != 0: device pointers).  record = index into the load's records;
 * start/end per record; motif_size = k, the motif is record[start:start+k] upper-cased. */
int crf_fetch(crf_seq *seq, uint32_t *record, uint32_t *start, uint32_t *end, uint32_t *motif_size,
              uint64_t capacity, int dst_on_device);

typedef struct {
    double scan_ms;      /* device time, packed planes resident -> sorted results resident  */
    double kernel_ms;    /* the scan kernel alone                                          */
    uint64_t n_results;
    uint64_t n_tiles;
    uint64_t n_spilled;  /* results that left the in-order path (sorted by the fallback)   */
    uint64_t n_long;     /* runs finished by the block-cooperative walker                  */
    uint64_t n_candidates; /* (strip, k) pairs the filter sent to the exact phase          */
    uint64_t word_k_pairs; /* 32-base words x motif sizes evaluated                        */
    uint32_t reruns;     /* scans repeated because the result buffer was too small         */
    uint32_t launches;   /* kernels launched by the last crf_scan                          */
    uint64_t n_open;     /* results that reached the end of an open-ended record (output map) */
} crf_scan_stats_t;
int crf_scan_stats(const crf_seq *seq, crf_scan_stats_t *stats);

/* Results of the last scan that reached the end of an open-ended record (see crf_seq_set_output_map): up to
 * `cap` rows of 5 values (row index in the result list, record, start, end, motif_size) in result order;
 * *n_open = how many there are in total.  crf_patch_end overwrites the end of one result row in HBM (after
 * the run has been followed with crf_run_end on whoever holds the next bases). */
int crf_fetch_open(crf_seq *seq, uint32_t *rows, uint32_t cap, uint32_t *n_open);
int crf_patch_end(crf_seq *seq, uint64_t row, uint32_t new_end);

/* End of the maximal run of period k through position `pos` of `record` (pos must satisfy
 * M_k[pos] == 1, else *run_end = pos).  *run_end = first position >= pos that does not match.
 * Used to stitch runs that leave a partition (chunk/GPU) -- see DESIGN.md "multi-GPU". */
int crf_run_end(crf_seq *seq, uint32_t record, uint32_t pos, uint32_t k, uint32_t *run_end);

/* Interval mode, for every record r of the load: record r is the prefix s_r[0 .. W_r) of a sequence s_r of full_len[r]
 * bases (W_r = the record's loaded length).  stop[r] = the position T after which the reference's lock-step loop breaks
 * (prf:70-74: the first t > end_pos[r] at which no tracker k in [min_motif_size, max_motif_size] is mid-repeat; tracker k
 * is mid-repeat at t iff the k compares of M_k ending at min(t, full_len[r] - k - 1) are all matches),
 * CRF_STOP_TO_END (-1) if the loop runs to the end of s_r (end_pos[r] >= full_len[r] - 1 included), CRF_STOP_UNDECIDED
 * (-2) if W_r < full_len[r] and every t the loaded prefix can decide (t <= W_r - 1 - max_motif_size) is covered: load a
 * longer prefix and ask again.  T is relative to the record.  One warp per record walks from just before end_pos[r] + 1
 * to T, one 32-base word per step: a repeat that straddles end_pos costs a walk over its length.  CRF_ERR_ARG if some
 * W_r > full_len[r] or max_motif_size exceeds the load's max_motif_cap; CRF_ERR_UNSUPPORTED above ~58 000 motif sizes.
 * end_pos, full_len, stop: host arrays of n_records entries.  One stream sync.  crf_b200/intervals.py scans many intervals
 * of one sequence in one load with it (DESIGN.md section 6, "Many intervals"). */
#define CRF_STOP_TO_END (-1)
#define CRF_STOP_UNDECIDED (-2)
int crf_interval_stop(crf_seq *seq, uint32_t min_motif_size, uint32_t max_motif_size, const uint64_t *end_pos,
                      const uint64_t *full_len, int64_t *stop);

/* ---- multi-GPU: gathering the compacted rows of N GPUs on rank 0 over NVLink peer memory -----------------
 * The reference scales out by fanning `--interval` jobs over CPU workers and concatenating their BED files
 * (hail_batch_pipeline/run_hail_batch_pipeline.py:76-77, 115-123, 153).  Here each rank (one GPU: one process
 * under torchrun, or one thread of a single process) scans a contiguous range of (record, chunk) units, so the
 * final list is the concatenation of the ranks' sorted rows in rank order.  An exchange block per rank, mapped
 * into every peer (CUDA IPC between processes, peer access inside one process), lets the GPUs do that
 * concatenation themselves: counts are exchanged with 8-byte peer stores, every rank writes its rows straight
 * into rank 0's buffer at its prefix offset, no host round trip and no collective library inside a step
 * (csrc/crf_xchg.cuh).  All ranks must make the same sequence of crf_scan_gather / crf_xchg_push calls.
 */
typedef struct crf_xchg crf_xchg;
#define CRF_IPC_HANDLE_BYTES 64
#define CRF_XCHG_MAX_WORLD 16
/* row_cap = rows rank 0's buffer holds (16 bytes each; only rank 0 allocates them). */
int crf_xchg_create(crf_ctx *ctx, uint32_t rank, uint32_t world, uint64_t row_cap, crf_xchg **xchg);
int crf_xchg_destroy(crf_xchg *xchg);
/* Ranks in different processes: export a CRF_IPC_HANDLE_BYTES handle, pass it around (any transport), connect. */
int crf_xchg_export(crf_xchg *xchg, uint8_t *handle);
int crf_xchg_connect_ipc(crf_xchg *xchg, uint32_t peer_rank, const uint8_t *handle);
/* Ranks of one process (one context per device, one thread per context). */
int crf_xchg_connect_local(crf_xchg *xchg, uint32_t peer_rank, crf_xchg *peer);
int crf_xchg_set_timeout(crf_xchg *xchg, double seconds); /* how long a kernel waits for a peer (default 20 s) */
/* 12 instead of 16 bytes per row over NVLink (rank 0's ingress bounds the gather): allowed when every record number and every
 * motif size of the job is below 65 536; all ranks must make the same choice.  Rank 0 still ends up with the four columns. */
int crf_xchg_set_compact(crf_xchg *xchg, int on);

/* crf_scan + push in one go, fully asynchronous: nothing is copied back and the host does not wait.  If the scan
 * outgrows a buffer, has a long spill list or more open-ended rows than their list holds, the step is void on
 * every rank (status 1): repeat it with crf_scan (which grows what was too small) followed by crf_xchg_push.
 * A job may be gathered in several PHASES (a rank holds one sequence per phase; genome order = phase-major, rank-minor):
 * append != 0 puts this step's rows after those of the job's earlier steps.  The exchange kernels run on a stream of
 * their own behind the scan that feeds them, so the push of phase p overlaps the scan of phase p + 1. */
int crf_scan_gather(crf_seq *seq, const crf_scan_params *params, crf_xchg *xchg, int append);
/* Push the rows of the last completed crf_scan (asynchronous). */
int crf_xchg_push(crf_seq *seq, crf_xchg *xchg, int append);

typedef struct {
    uint32_t status;        /* of the last step: 0 ok, 1 void (repeat the slow way), 2 rank 0's buffer too small, 3 timeout */
    uint32_t worst_status;  /* over all steps since the previous crf_xchg_wait */
    uint32_t steps_checked;
    uint32_t step;          /* number of the last step (from 1) */
    uint32_t any_open;      /* some rank has open-ended rows (same answer on every rank): stitch before using the rows */
    uint32_t reserved;
    uint64_t total_rows;    /* rows of all ranks so far in this job (they are on rank 0, in genome order) */
    uint64_t base_rows;     /* of which gathered by the job's earlier phases (0 unless the step appended) */
    uint64_t total_open;    /* rank 0 only: open-ended rows of all ranks (runs that left their unit's data) */
    uint64_t my_offset;     /* first row of this rank inside rank 0's buffer */
    uint64_t rows_of_rank[CRF_XCHG_MAX_WORLD];
} crf_xchg_result_t;
/* Wait until this rank's part of every queued step is complete (on rank 0: until all rows have landed). */
int crf_xchg_wait(crf_xchg *xchg, crf_xchg_result_t *result);
/* The result of one of the last 64 steps that crf_xchg_wait has already checked (phased jobs: one per phase). */
int crf_xchg_step_result(crf_xchg *xchg, uint32_t step, crf_xchg_result_t *result);
/* Rank 0: copy gathered rows [first_row, first_row + n_rows) out (see crf_fetch for the columns). */
int crf_xchg_fetch(crf_xchg *xchg, uint32_t *record, uint32_t *start, uint32_t *end, uint32_t *motif_size,
                   uint64_t first_row, uint64_t n_rows, int dst_on_device);
/* Rank 0: overwrite the end of gathered rows (global row numbers) -- stitched open-ended runs. */
int crf_xchg_patch_end(crf_xchg *xchg, const uint64_t *rows, const uint32_t *new_end, uint32_t n);

/* ---- per-base masks --------------------------------------------------------------------------
 * Sets mask to exactly the union over i < n_rows of the bits
 *   [dst_offset[record[i]] + start[i], dst_offset[record[i]] + end[i])
 * (bit p & 31 of word p >> 5; mask holds ceil(mask_bits / 32) words, written in full, every bit no row covers cleared).
 * Rows may overlap and come in any order: the union of a scan's rows is its repeat mask (crf_b200/mask.py), with
 * dst_offset = where each record (or unit of a record longer than one load, crf_load_limit) starts in the mask.
 * dst_offset: host array of n_records uint64 values, so a destination may lie above 2^32.
 * rows_on_device / mask_on_device select device or host pointers for record / start / end and for mask.
 * A row with end < start, record >= n_records, or a range past mask_bits gives CRF_ERR_ARG (the mask is then
 * unspecified).  One stream sync. */
int crf_mask_rows(crf_ctx *ctx, const uint32_t *record, const uint32_t *start, const uint32_t *end, uint64_t n_rows,
                  int rows_on_device, const uint64_t *dst_offset, uint32_t n_records,
                  uint32_t *mask, uint64_t mask_bits, int mask_on_device);

/* ---- output (host only, no GPU) -------------------------------------------------------------
 * Writes result rows as text, replacing the per-row Python of prf:148-149 (BED: chrom, start, end, motif) and
 * prf:166-170 (TSV: start_0based, end, motif, with header).  names = NUL-separated record names in record
 * order; bases/offsets = the host copy of the records (the motif is bases[offsets[r] + start .. + k),
 * upper-cased).  append != 0 appends to an existing file.  Returns the number of bytes written in *bytes. */
int crf_write_rows(const char *path, int append, int tsv, const char *names, const uint8_t *bases,
                   const uint64_t *offsets, const uint32_t *record, const uint32_t *start, const uint32_t *end,
                   const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes);
/* The same with origin[r] (NULL = 0 for every record) added to the printed start and end of record r's rows: the
 * rows of a chromosome longer than 2^32 bases, written unit by unit (names repeated, offsets[u] = the host offset of
 * the unit's origin, start / end relative to it).  crf_write_rows is this call with origin = NULL. */
int crf_write_rows_at(const char *path, int append, int tsv, const char *names, const uint8_t *bases,
                      const uint64_t *offsets, const uint64_t *origin, const uint32_t *record, const uint32_t *start,
                      const uint32_t *end, const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes);
/* crf_write_rows for records read from a .2bit file: the motif is read from the file's packed bases (dna and rec_byte as
 * crf_fasta_twobit gives them: record r's base i is bits 7-6 of byte rec_byte[r] + i / 4 for i % 4 == 0, then 5-4, 3-2,
 * 1-0; T=0 C=1 A=2 G=3) as upper-case A/C/G/T.  A motif never holds an N, so the output is byte-identical to
 * crf_write_rows on the file's decoded text (crf_fasta_data). */
int crf_write_rows_twobit(const char *path, int append, int tsv, const char *names, const uint8_t *dna,
                          const uint64_t *rec_byte, const uint32_t *record, const uint32_t *start, const uint32_t *end,
                          const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes);
/* crf_write_rows for reads of a BAM file: the motif is read from their 4-bit codes (nib and rec_byte as crf_fasta_nibbles
 * gives them: record r's base i is nibble i & 1, high nibble first, of byte rec_byte[r] + i / 2) as the letters
 * =ACMGRSVTWYHKDBN -- byte-identical to crf_write_rows on the file's decoded text (crf_fasta_data). */
int crf_write_rows_nibbles(const char *path, int append, int tsv, const char *names, const uint8_t *nib,
                           const uint64_t *rec_byte, const uint32_t *record, const uint32_t *start, const uint32_t *end,
                           const uint32_t *motif_size, uint64_t n_rows, uint64_t *bytes);
/* A repeat-masked FASTA file: per record a header line ">name" (names NUL-separated, as crf_write_rows takes them), then
 * its bases, line_width per line.  Mask bit p (as crf_mask_rows lays it out) stands for bases[p], with the indexing of
 * offsets (record r = bases[offsets[r] .. offsets[r+1])).  A masked byte is lower-cased when it is an ASCII letter A-Z
 * (hard == 0: soft masking) or becomes 'N' (hard != 0); every other byte is written as it is.  Formatted on up to 16
 * threads.  *bytes = bytes written; a short write is CRF_ERR_IO. */
int crf_write_fasta_masked(const char *path, const char *names, const uint8_t *bases, const uint64_t *offsets,
                           uint64_t n_records, const uint32_t *mask, int hard, uint32_t line_width, uint64_t *bytes);
/* The same as a FASTQ file: per record "@name\n", its bases on one line (masked as above), "+\n" and quals[offsets[r] ..
 * offsets[r+1]) on one line, written as they are (quals is indexed like bases, as crf_fasta_quals gives it). */
int crf_write_fastq_masked(const char *path, const char *names, const uint8_t *bases, const uint8_t *quals,
                           const uint64_t *offsets, uint64_t n_records, const uint32_t *mask, int hard, uint64_t *bytes);

/* ---- input (host only, no GPU) ---------------------------------------------------------------
 * Native FASTA ingest, replacing what the reference takes from pyfastx (prf:117-137: the records in file
 * order, .name = first whitespace-delimited header token, .seq = the lines joined, case preserved).  Plain or
 * gzip (concatenated members too; BGZF/bgzip blocks are inflated in parallel).
 * FASTQ too: a text whose first byte that is not whitespace is '@' is read as FASTQ (records '@name ...', sequence
 * lines up to a line starting with '+', quality lines until they hold as many bytes as the sequence; multi-line records
 * and CRLF line ends are read; a malformed record is CRF_ERR_ARG naming its 1-based number), with the same layout.  The result is laid out as crf_seq_load_ascii and crf_write_rows
 * take it: all records back to back, n_records+1 offsets, NUL-separated names.  n_threads = 0: up to 16.
 * pinned: bit 0 = page-locked base buffer (cudaHostAlloc, when a device is present: a faster upload of the text), bit 1 =
 * page-locked planes only (crf_fasta_packed; bit 0 implies it) -- what a caller that uploads the planes and keeps the text
 * on the host for the motif column wants: page-locking gigabytes it never uploads costs seconds.  Bit 2 (value 4): keep
 * a FASTQ file's qualities (crf_fasta_quals); without it they are checked and dropped.
 * The pointers of crf_fasta_data and crf_fasta_quals stay valid until crf_fasta_close. */
typedef struct crf_fasta crf_fasta;
int crf_fasta_open(const char *path, uint32_t n_threads, int pinned, crf_fasta **fasta);
int crf_fasta_info(const crf_fasta *fasta, uint64_t *n_records, uint64_t *total_bases, int *pinned);
int crf_fasta_data(const crf_fasta *fasta, const uint8_t **bases, const uint64_t **offsets, const char **names,
                   uint64_t *names_bytes);
/* UCSC .2bit too: a file that starts with the signature 0x1A412743 (either byte order; version 0, or 1 with 64-bit index
 * offsets) is read as .2bit.  Only its index and record headers are parsed at open: every count, offset and block is
 * checked against the file size and dnaSize, and a bad file is CRF_ERR_ARG naming the 1-based record.  N blocks and mask
 * blocks may be unsorted or overlap; they are merged per record.  crf_fasta_data then decodes the text on first call (on the
 * reader's threads): what twoBitToFa writes, T/C/A/G, N blocks as 'N', mask blocks lower-cased ('n' inside both).
 * BAM too: a BGZF file whose first inflated bytes are "BAM\1" is read as unaligned reads, giving what `samtools fastq -n`
 * writes from it: the records with (flag & 0x900) == 0 in file order, named by read_name, their bases reverse-complemented
 * when flag & 0x10, qualities + 33 (reversed with them; '"' when absent).  The blocks are inflated on the reader's threads
 * a window of 32 MiB at a time and only the 4-bit codes (crf_fasta_nibbles), the names and, with pinned bit 2, the
 * qualities are kept: host memory peaks at the window, plus the largest record, plus what is kept (with pinned & 3 the
 * codes are then copied into page-locked memory, so for that moment they are held twice).  Every count and length
 * is checked against the record and the stream; a malformed record is CRF_ERR_ARG naming its 1-based number (a missing
 * end-of-file block is accepted), and a BAM compressed as plain gzip rather than BGZF is CRF_ERR_ARG.  crf_fasta_data
 * decodes the text on its first call (on the reader's threads), letters of =ACMGRSVTWYHKDBN.
 * *format = 0 for a FASTA file, 1 for a FASTQ file, 2 for a .2bit file, 3 for a BAM file. */
int crf_fasta_format(const crf_fasta *fasta, int *format);
/* A FASTQ or BAM file's qualities, laid out like the bases (record r = quals[offsets[r] .. offsets[r+1])); NULL for other
 * formats or when crf_fasta_open was not given pinned bit 2. */
int crf_fasta_quals(const crf_fasta *fasta, const uint8_t **quals);
/* Offsets (n_records + 1) and NUL-separated names of any handle, without decoding a .2bit or BAM file's bases. */
int crf_fasta_index(const crf_fasta *fasta, const uint64_t **offsets, const char **names, uint64_t *names_bytes);
/* A .2bit handle's packed form (CRF_ERR_ARG for any other): dna = the file's bytes (page-locked when crf_fasta_open had
 * pinned & 3, else mapped), rec_byte[r] = the byte where record r's packed bases start, runs = its N blocks as n_runs
 * ascending, disjoint runs [runs[2i], runs[2i+1]) of the position space of the offsets (merged within a record, not across
 * records) -- what crf_seq_load_2bit and crf_write_rows_twobit take. */
int crf_fasta_twobit(const crf_fasta *fasta, const uint8_t **dna, const uint64_t **rec_byte, const uint64_t **runs,
                     uint64_t *n_runs);
/* A BAM handle's packed form (CRF_ERR_ARG for any other): nib = the reads' 4-bit codes (page-locked when crf_fasta_open
 * had pinned & 3), record r from byte rec_byte[r] with reverse complements applied (an odd record's last byte has a low
 * nibble 0), exotic = the n_exotic codes other than A, C, G, T and N as (position in the space of the offsets << 8 | letter),
 * ascending -- what crf_seq_load_nibbles and crf_write_rows_nibbles take. */
int crf_fasta_nibbles(const crf_fasta *fasta, const uint8_t **nib, const uint64_t **rec_byte, const uint64_t **exotic,
                      uint64_t *n_exotic);
/* Packed planes of the whole file (all records back to back, as crf_seq_load_packed takes them), made on first call
 * and owned by the handle; page-locked when the base buffer is. */
int crf_fasta_packed(crf_fasta *fasta, uint32_t n_threads, const uint32_t **H, const uint32_t **L, const uint32_t **NM,
                     const uint64_t **exotic, uint64_t *n_exotic);
int crf_fasta_close(crf_fasta *fasta);
/* Host only: all members of a gzip stream -> bytes, with the FASTA reader's own DEFLATE decoder (use_zlib == 0; it hands
 * anything it does not take to zlib, as the reader does), with zlib alone (use_zlib == 1), or with the reader's decoder
 * alone (use_zlib == 2: CRF_ERR_UNSUPPORTED for what it declines -- corrupt input included).  CRF_ERR_CAPACITY with *out_n =
 * the size needed when `cap` is too small; CRF_ERR_ARG for a stream zlib rejects too. */
int crf_gunzip(const uint8_t *gz, uint64_t n, uint8_t *out, uint64_t cap, uint64_t *out_n, int use_zlib);

#ifdef __cplusplus
}
#endif
#endif /* CRF_H */
