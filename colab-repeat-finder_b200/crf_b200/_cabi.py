"""ctypes binding of libcrf.so (the C ABI in include/crf.h).

This is the only way the Python host code reaches the GPU.  There is no CPU fallback: if the
shared library is missing or a call fails, an exception is raised.
"""
import ctypes
import functools
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CRF_LIB_PATH") or os.path.join(_HERE, "libcrf.so")   # override: A/B builds while tuning

SCAN_NO_PRIMITIVITY = 1
SCAN_WARP_TILES = 2
SCAN_BLOCK_TILES = 4
SCAN_TWO_STRIPS = 8

CRF_OK, CRF_ERR_CUDA, CRF_ERR_ARG, CRF_ERR_NOMEM, CRF_ERR_UNSUPPORTED, CRF_ERR_CAPACITY, CRF_ERR_IO = range(7)
STOP_TO_END, STOP_UNDECIDED = -1, -2          # crf_interval_stop
#: most motif sizes (max - min + 1) crf_interval_stop takes: one uint32 of shared memory each, 227 KB per block; it refuses
#: more with CRF_ERR_UNSUPPORTED
STOP_MAX_MOTIF_SIZES = (227 << 10) // 4

#: every symbol include/crf.h declares (tests check the library exports all of them)
EXPORTS = [
    "crf_last_error", "crf_abi_version", "crf_ctx_create", "crf_ctx_destroy", "crf_ctx_set_stream",
    "crf_ctx_synchronize", "crf_load_limit", "crf_seq_load_packed", "crf_seq_load_packed_ranges", "crf_pack_ascii",
    "crf_seq_load_packed_runs", "crf_seq_load_packed_runs_ranges", "crf_mask_runs",
    "crf_fasta_packed", "crf_seq_load_2bit", "crf_seq_load_nibbles", "crf_seq_load_ascii", "crf_seq_load_ascii_ranges", "crf_seq_set_output_map", "crf_seq_destroy", "crf_seq_info", "crf_scan", "crf_fetch",
    "crf_scan_stats", "crf_run_end", "crf_interval_stop", "crf_fetch_open", "crf_patch_end", "crf_write_rows",
    "crf_write_rows_at", "crf_write_rows_twobit", "crf_write_rows_nibbles", "crf_mask_rows", "crf_write_fasta_masked", "crf_write_fastq_masked",
    "crf_fasta_open", "crf_fasta_info", "crf_fasta_data", "crf_fasta_format", "crf_fasta_quals", "crf_fasta_index",
    "crf_fasta_twobit", "crf_fasta_nibbles", "crf_fasta_close",
    "crf_gunzip",
    "crf_xchg_create", "crf_xchg_destroy", "crf_xchg_export", "crf_xchg_connect_ipc", "crf_xchg_connect_local",
    "crf_xchg_set_timeout", "crf_xchg_set_compact", "crf_scan_gather", "crf_xchg_push", "crf_xchg_wait", "crf_xchg_step_result", "crf_xchg_fetch",
    "crf_xchg_patch_end",
]

IPC_HANDLE_BYTES = 64
XCHG_MAX_WORLD = 16
XCHG_OK, XCHG_VOID_STEP, XCHG_ROOT_FULL, XCHG_TIMEOUT = range(4)


class CrfError(RuntimeError):
    """A libcrf call failed (CUDA error, out of memory, capacity)."""


class ScanParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint32) for n in (
        "min_motif_size", "max_motif_size", "min_repeats", "min_span",
        "words_per_thread", "tile_out_cap", "walk_limit_words", "result_cap", "flags")]


class SeqInfo(ctypes.Structure):
    _fields_ = [("n_records", ctypes.c_uint64), ("total_bases", ctypes.c_uint64), ("layout_bases", ctypes.c_uint64),
                ("packed_bytes", ctypes.c_uint64), ("n_exotic", ctypes.c_uint64), ("max_motif_cap", ctypes.c_uint32),
                ("reserved", ctypes.c_uint32), ("load_ms", ctypes.c_double)]


class ScanStats(ctypes.Structure):
    _fields_ = [("scan_ms", ctypes.c_double), ("kernel_ms", ctypes.c_double), ("n_results", ctypes.c_uint64),
                ("n_tiles", ctypes.c_uint64), ("n_spilled", ctypes.c_uint64), ("n_long", ctypes.c_uint64),
                ("n_candidates", ctypes.c_uint64), ("word_k_pairs", ctypes.c_uint64), ("reruns", ctypes.c_uint32),
                ("launches", ctypes.c_uint32), ("n_open", ctypes.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class XchgResult(ctypes.Structure):
    _fields_ = [("status", ctypes.c_uint32), ("worst_status", ctypes.c_uint32), ("steps_checked", ctypes.c_uint32),
                ("step", ctypes.c_uint32), ("any_open", ctypes.c_uint32), ("reserved", ctypes.c_uint32),
                ("total_rows", ctypes.c_uint64), ("base_rows", ctypes.c_uint64), ("total_open", ctypes.c_uint64),
                ("my_offset", ctypes.c_uint64), ("rows_of_rank", ctypes.c_uint64 * XCHG_MAX_WORLD)]


_lib = None


def lib():
    """Load libcrf.so once; raise (never fall back) if it is not there."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CrfError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           f"(nvcc, sm_100a). There is no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        vp, u32, u64, i = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int
        P = ctypes.POINTER
        L.crf_last_error.restype = ctypes.c_char_p
        L.crf_last_error.argtypes = []
        L.crf_abi_version.restype = i
        L.crf_ctx_create.argtypes = [i, P(vp)]
        L.crf_ctx_destroy.argtypes = [vp]
        L.crf_ctx_set_stream.argtypes = [vp, vp]
        L.crf_ctx_synchronize.argtypes = [vp]
        L.crf_seq_load_ascii.argtypes = [vp, vp, vp, u32, u32, i, P(vp)]
        L.crf_seq_load_ascii_ranges.argtypes = [vp, vp, vp, vp, vp, vp, u32, u32, i, P(vp)]
        L.crf_seq_load_packed.argtypes = [vp, vp, vp, vp, vp, u64, vp, u32, u32, i, P(vp)]
        L.crf_seq_load_packed_ranges.argtypes = [vp, vp, vp, vp, vp, u64, vp, vp, vp, vp, u32, u32, i, P(vp)]
        L.crf_pack_ascii.argtypes = [vp, u64, u32, vp, vp, vp, vp, u64, P(u64)]
        L.crf_seq_load_packed_runs.argtypes = [vp, vp, vp, vp, u64, vp, u64, vp, u32, u32, i, P(vp)]
        L.crf_seq_load_packed_runs_ranges.argtypes = [vp, vp, vp, vp, u64, vp, u64, vp, vp, vp, vp, u32, u32, i, P(vp)]
        L.crf_mask_runs.argtypes = [vp, u64, u32, vp, u64, P(u64)]
        L.crf_fasta_packed.argtypes = [vp, u32, P(vp), P(vp), P(vp), P(vp), P(u64)]
        L.crf_seq_load_2bit.argtypes = [vp, vp, vp, vp, u32, vp, u64, u32, i, P(vp)]
        L.crf_seq_load_nibbles.argtypes = [vp, vp, vp, vp, u32, vp, u64, u32, i, P(vp)]
        L.crf_seq_set_output_map.argtypes = [vp, vp, vp, vp]
        L.crf_seq_destroy.argtypes = [vp]
        L.crf_seq_info.argtypes = [vp, P(SeqInfo)]
        L.crf_scan.argtypes = [vp, P(ScanParams), P(u64)]
        L.crf_fetch.argtypes = [vp, vp, vp, vp, vp, u64, i]
        L.crf_scan_stats.argtypes = [vp, P(ScanStats)]
        L.crf_run_end.argtypes = [vp, u32, u32, u32, P(u32)]
        L.crf_interval_stop.argtypes = [vp, u32, u32, vp, vp, vp]
        L.crf_fetch_open.argtypes = [vp, vp, u32, P(u32)]
        L.crf_patch_end.argtypes = [vp, u64, u32]
        L.crf_write_rows.argtypes = [ctypes.c_char_p, i, i, vp, vp, vp, vp, vp, vp, vp, u64, P(u64)]
        L.crf_write_rows_at.argtypes = [ctypes.c_char_p, i, i, vp, vp, vp, vp, vp, vp, vp, vp, u64, P(u64)]
        L.crf_write_rows_twobit.argtypes = [ctypes.c_char_p, i, i, vp, vp, vp, vp, vp, vp, vp, u64, P(u64)]
        L.crf_write_rows_nibbles.argtypes = [ctypes.c_char_p, i, i, vp, vp, vp, vp, vp, vp, vp, u64, P(u64)]
        L.crf_mask_rows.argtypes = [vp, vp, vp, vp, u64, i, vp, u32, vp, u64, i]
        L.crf_write_fasta_masked.argtypes = [ctypes.c_char_p, vp, vp, vp, u64, vp, i, u32, P(u64)]
        L.crf_write_fastq_masked.argtypes = [ctypes.c_char_p, vp, vp, vp, vp, u64, vp, i, P(u64)]
        L.crf_fasta_open.argtypes = [ctypes.c_char_p, u32, i, P(vp)]
        L.crf_fasta_info.argtypes = [vp, P(u64), P(u64), P(i)]
        L.crf_fasta_data.argtypes = [vp, P(vp), P(vp), P(vp), P(u64)]
        L.crf_fasta_format.argtypes = [vp, P(i)]
        L.crf_fasta_quals.argtypes = [vp, P(vp)]
        L.crf_fasta_index.argtypes = [vp, P(vp), P(vp), P(u64)]
        L.crf_fasta_twobit.argtypes = [vp, P(vp), P(vp), P(vp), P(u64)]
        L.crf_fasta_nibbles.argtypes = [vp, P(vp), P(vp), P(vp), P(u64)]
        L.crf_fasta_close.argtypes = [vp]
        L.crf_gunzip.argtypes = [vp, ctypes.c_uint64, vp, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64), ctypes.c_int]
        L.crf_xchg_create.argtypes = [vp, u32, u32, u64, P(vp)]
        L.crf_xchg_destroy.argtypes = [vp]
        L.crf_xchg_export.argtypes = [vp, vp]
        L.crf_xchg_connect_ipc.argtypes = [vp, u32, vp]
        L.crf_xchg_connect_local.argtypes = [vp, u32, vp]
        L.crf_xchg_set_timeout.argtypes = [vp, ctypes.c_double]
        L.crf_xchg_set_compact.argtypes = [vp, i]
        L.crf_scan_gather.argtypes = [vp, P(ScanParams), vp, i]
        L.crf_xchg_push.argtypes = [vp, vp, i]
        L.crf_xchg_wait.argtypes = [vp, P(XchgResult)]
        L.crf_xchg_step_result.argtypes = [vp, u32, P(XchgResult)]
        L.crf_xchg_fetch.argtypes = [vp, vp, vp, vp, vp, u64, u64, i]
        L.crf_xchg_patch_end.argtypes = [vp, vp, vp, u32]
        L.crf_load_limit.argtypes = [u32]
        for name in EXPORTS:
            if name not in ("crf_last_error", "crf_load_limit"):
                getattr(L, name).restype = i
        L.crf_load_limit.restype = u64
        _lib = L
    return _lib


def _check(rc):
    if rc == CRF_OK:
        return
    msg = lib().crf_last_error().decode("utf-8", "replace")
    if rc == CRF_ERR_ARG:
        raise ValueError(msg)
    if rc == CRF_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == CRF_ERR_NOMEM:
        raise MemoryError(msg)
    if rc == CRF_ERR_IO:
        raise OSError(msg)
    raise CrfError(f"libcrf error {rc}: {msg}")


def _serialised(method):
    """Calls on one context (and on its sequences / exchange blocks) must not overlap (include/crf.h "Threading"):
    api.get_context() hands the same Context to every thread of the process, so the binding takes the context's lock."""
    @functools.wraps(method)
    def wrapper(self, *a, **kw):
        ctx = self if isinstance(self, Context) else (getattr(self, "ctx", None) or a[0])   # __init__(self, ctx, ...)
        with ctx._lock:
            return method(self, *a, **kw)
    return wrapper


def load_limit(max_motif_cap):
    """Layout positions (sum of record length + max_motif_cap) one load can hold (crf_load_limit)."""
    return int(lib().crf_load_limit(int(max_motif_cap)))


class Context:
    """One CUDA device (crf_ctx)."""

    def __init__(self, device=0):
        self._h = ctypes.c_void_p()
        self._lock = threading.RLock()
        self.device = device
        _check(lib().crf_ctx_create(device, ctypes.byref(self._h)))

    def set_stream(self, cuda_stream_ptr):
        _check(lib().crf_ctx_set_stream(self._h, ctypes.c_void_p(cuda_stream_ptr or 0)))

    def synchronize(self):
        _check(lib().crf_ctx_synchronize(self._h))

    def load(self, bases, offsets=None, max_motif_cap=50, on_device=False):
        """bases: bytes / uint8 ndarray (host) or an int device pointer (on_device=True).
        offsets: uint64 array of n_records+1 record boundaries (default: one record)."""
        return Sequence(self, bases, offsets, max_motif_cap, on_device)

    def load_ranges(self, bases, starts, lengths, own_lo=None, own_hi=None, max_motif_cap=50, on_device=False):
        """Records given as (start, length) ranges of `bases` (may overlap); optional owned
        sub-range per record (crf_seq_load_ascii_ranges)."""
        return Sequence(self, bases, None, max_motif_cap, on_device, ranges=(starts, lengths, own_lo, own_hi))

    def load_packed(self, planes, offsets=None, max_motif_cap=50, ranges=None):
        """planes: a PackedPlanes (host, from pack_ascii() / Fasta.packed()).  offsets: n_records + 1 record boundaries
        in the planes' position space (default: one record), or ranges=(starts, lengths, own_lo, own_hi)."""
        if offsets is None and ranges is None:
            offsets = np.array([0, planes.n_bases], dtype=np.uint64)
        return Sequence(self, None, offsets, max_motif_cap, False, ranges=ranges, packed=planes)

    def load_2bit(self, source, max_motif_cap=50, on_device=False):
        """crf_seq_load_2bit: the records of a .2bit file, loaded from its packed bytes.  source: a .2bit Fasta, or a
        TwoBitSource (Fasta.twobit(), .records(first, last) for some of them) whose dna may also be a CUDA uint8 tensor
        holding the file's bytes, or a device pointer (int) with on_device=True."""
        if isinstance(source, Fasta):
            source = source.twobit()
        return Sequence(self, None, None, max_motif_cap, on_device, twobit=source)

    def load_nibbles(self, source, max_motif_cap=50, on_device=False):
        """crf_seq_load_nibbles: the reads of a BAM file, loaded from their 4-bit codes.  source: a BAM Fasta, or a
        NibbleSource (Fasta.nibbles(), .records(first, last) for some of them) whose nib may also be a CUDA uint8 tensor
        holding the codes, or a device pointer (int) with on_device=True."""
        if isinstance(source, Fasta):
            source = source.nibbles()
        return Sequence(self, None, None, max_motif_cap, on_device, nibbles=source)

    @_serialised
    def mask_rows(self, record, start, end, dst_offset, mask_bits, n_rows=None, mask=None):
        """crf_mask_rows: the union of the rows [dst_offset[record] + start, dst_offset[record] + end) as a bit mask.
        record / start / end: host arrays, or device pointers (ints) with n_rows given.  dst_offset: host array, one
        uint64 per record.  mask: None returns a new host uint32 array of ceil(mask_bits / 32) words; an int is a device
        pointer to that many words, painted in place (returns None)."""
        on_device = isinstance(record, int)
        if on_device:
            ptrs = [ctypes.c_void_p(int(a)) for a in (record, start, end)]
        else:
            cols = [np.ascontiguousarray(a, dtype=np.uint32) for a in (record, start, end)]
            if not cols[0].shape == cols[1].shape == cols[2].shape or cols[0].ndim != 1:
                raise ValueError("record, start and end must be 1-d arrays of equal size")
            n_rows = cols[0].size
            ptrs = [ctypes.c_void_p(a.ctypes.data) for a in cols]
        dst = np.ascontiguousarray(dst_offset, dtype=np.uint64)
        out = np.zeros((int(mask_bits) + 31) // 32, np.uint32) if mask is None else None
        mptr = out.ctypes.data if out is not None else int(mask)
        _check(lib().crf_mask_rows(self._h, *ptrs, int(n_rows), int(on_device), ctypes.c_void_p(dst.ctypes.data), dst.size,
                                   ctypes.c_void_p(mptr), int(mask_bits), int(mask is not None)))
        return out

    def close(self):
        if self._h:
            lib().crf_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Sequence:
    """Records resident in HBM as packed planes (crf_seq)."""

    @_serialised
    def __init__(self, ctx, bases, offsets, max_motif_cap, on_device, ranges=None, packed=None, twobit=None,
                 nibbles=None):
        self.ctx = ctx
        self._h = ctypes.c_void_p()
        keep = None
        src = twobit if twobit is not None else nibbles
        if src is not None:                               # a .2bit or BAM source: bytes of codes, read from rec_byte[r]
            what, per_byte, kind, load = (("dna", 4, ".2bit", lib().crf_seq_load_2bit) if twobit is not None else
                                          ("nib", 2, "BAM", lib().crf_seq_load_nibbles))
            codes = getattr(src, what)
            ptr, on_device = _source_bytes(what, codes, on_device)
            offsets = np.ascontiguousarray(src.offsets, dtype=np.uint64)
            rec_byte = np.ascontiguousarray(src.rec_byte, dtype=np.uint64)
            lst = (np.ascontiguousarray(src.runs, dtype=np.uint64).reshape(-1, 2) if twobit is not None else
                   np.ascontiguousarray(src.exotic, dtype=np.uint64))
            if offsets.ndim != 1 or offsets.size < 2 or rec_byte.shape != (offsets.size - 1,):
                raise ValueError(f"a {kind} source needs n_records + 1 offsets and n_records rec_byte entries")
            _check_extent(what, codes, rec_byte, offsets, per_byte)
            self.offsets = offsets
            self.n_records = offsets.size - 1
            _check(load(ctx._h, ctypes.c_void_p(ptr), ctypes.c_void_p(rec_byte.ctypes.data),
                        ctypes.c_void_p(offsets.ctypes.data), self.n_records,
                        ctypes.c_void_p(lst.ctypes.data if lst.size else 0), lst.shape[0],
                        int(max_motif_cap), int(bool(on_device)), ctypes.byref(self._h)))
            return
        if packed is not None:
            pk = packed
            ex_ptr = pk.exotic.ctypes.data if pk.exotic.size else 0
            if pk.runs is not None:                       # the mask travels as runs: 0.25 B/bp over PCIe
                runs_ptr = pk.runs.ctypes.data if pk.runs.size else 0
                n_runs = pk.runs.shape[0]
                if ranges is not None:
                    starts, lengths, own_lo, own_hi = (None if a is None else np.ascontiguousarray(a, dtype=np.uint64)
                                                       for a in ranges)
                    self.n_records = starts.size
                    self.lengths = lengths
                    _check(lib().crf_seq_load_packed_runs_ranges(
                        ctx._h, pk.H_ptr, pk.L_ptr, ctypes.c_void_p(runs_ptr), n_runs, ctypes.c_void_p(ex_ptr), pk.exotic.size,
                        ctypes.c_void_p(starts.ctypes.data), ctypes.c_void_p(lengths.ctypes.data),
                        ctypes.c_void_p(own_lo.ctypes.data if own_lo is not None else 0),
                        ctypes.c_void_p(own_hi.ctypes.data if own_hi is not None else 0),
                        self.n_records, int(max_motif_cap), int(bool(pk.on_device)), ctypes.byref(self._h)))
                    return
                offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
                if offsets.ndim != 1 or offsets.size < 2:
                    raise ValueError("offsets must hold n_records + 1 entries")
                self.offsets = offsets
                self.n_records = offsets.size - 1
                _check(lib().crf_seq_load_packed_runs(ctx._h, pk.H_ptr, pk.L_ptr, ctypes.c_void_p(runs_ptr), n_runs,
                                                      ctypes.c_void_p(ex_ptr), pk.exotic.size,
                                                      ctypes.c_void_p(offsets.ctypes.data), self.n_records, int(max_motif_cap),
                                                      int(bool(pk.on_device)), ctypes.byref(self._h)))
                return
            if ranges is not None:
                starts, lengths, own_lo, own_hi = (None if a is None else np.ascontiguousarray(a, dtype=np.uint64)
                                                   for a in ranges)
                self.n_records = starts.size
                self.lengths = lengths
                _check(lib().crf_seq_load_packed_ranges(
                    ctx._h, pk.H_ptr, pk.L_ptr, pk.NM_ptr, ctypes.c_void_p(ex_ptr), pk.exotic.size,
                    ctypes.c_void_p(starts.ctypes.data), ctypes.c_void_p(lengths.ctypes.data),
                    ctypes.c_void_p(own_lo.ctypes.data if own_lo is not None else 0),
                    ctypes.c_void_p(own_hi.ctypes.data if own_hi is not None else 0),
                    self.n_records, int(max_motif_cap), int(bool(pk.on_device)), ctypes.byref(self._h)))
                return
            offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
            if offsets.ndim != 1 or offsets.size < 2:
                raise ValueError("offsets must hold n_records + 1 entries")
            self.offsets = offsets
            self.n_records = offsets.size - 1
            _check(lib().crf_seq_load_packed(ctx._h, pk.H_ptr, pk.L_ptr, pk.NM_ptr, ctypes.c_void_p(ex_ptr), pk.exotic.size,
                                             ctypes.c_void_p(offsets.ctypes.data), self.n_records, int(max_motif_cap),
                                             int(bool(pk.on_device)), ctypes.byref(self._h)))
            return
        if on_device:
            ptr = int(bases)
            if offsets is None and ranges is None:
                raise ValueError("offsets are required with a device pointer")
        else:
            if isinstance(bases, np.ndarray):
                if bases.dtype != np.uint8 or not bases.flags.c_contiguous:
                    raise ValueError("bases must be a C-contiguous uint8 array")
                keep = bases
                ptr = bases.ctypes.data
                nbytes = bases.size
            else:
                keep = bytes(bases) if not isinstance(bases, bytes) else bases
                ptr = ctypes.cast(ctypes.c_char_p(keep), ctypes.c_void_p).value or 0
                nbytes = len(keep)
            if offsets is None and ranges is None:
                offsets = np.array([0, nbytes], dtype=np.uint64)
        if ranges is not None:
            starts, lengths, own_lo, own_hi = (None if a is None else np.ascontiguousarray(a, dtype=np.uint64)
                                               for a in ranges)
            if starts.shape != lengths.shape or starts.ndim != 1:
                raise ValueError("starts and lengths must be 1-d arrays of equal size")
            self.n_records = starts.size
            self.lengths = lengths
            _check(lib().crf_seq_load_ascii_ranges(
                ctx._h, ctypes.c_void_p(ptr), ctypes.c_void_p(starts.ctypes.data), ctypes.c_void_p(lengths.ctypes.data),
                ctypes.c_void_p(own_lo.ctypes.data if own_lo is not None else 0),
                ctypes.c_void_p(own_hi.ctypes.data if own_hi is not None else 0),
                self.n_records, int(max_motif_cap), int(bool(on_device)), ctypes.byref(self._h)))
            return
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        if offsets.ndim != 1 or offsets.size < 2:
            raise ValueError("offsets must hold n_records + 1 entries")
        self.offsets = offsets
        self.n_records = offsets.size - 1
        _check(lib().crf_seq_load_ascii(ctx._h, ctypes.c_void_p(ptr), ctypes.c_void_p(offsets.ctypes.data),
                                        self.n_records, int(max_motif_cap), int(bool(on_device)),
                                        ctypes.byref(self._h)))
        del keep

    @_serialised
    def set_output_map(self, out_record=None, out_shift=None, open_ended=None):
        """Report results in the coordinates of the chromosomes the units were cut from (crf_seq_set_output_map)."""
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=dt)
                for a, dt in ((out_record, np.uint32), (out_shift, np.uint64), (open_ended, np.uint8))]
        for a in arrs:
            if a is not None and a.size != self.n_records:
                raise ValueError("output map arrays need one entry per record of the load")
        _check(lib().crf_seq_set_output_map(self._h, *(ctypes.c_void_p(a.ctypes.data if a is not None else 0)
                                                       for a in arrs)))

    def info(self):
        out = SeqInfo()
        _check(lib().crf_seq_info(self._h, ctypes.byref(out)))
        return out

    @staticmethod
    def _params(min_motif_size, max_motif_size, min_repeats, min_span, knobs):
        return ScanParams(int(min_motif_size), int(max_motif_size), int(min_repeats), int(min_span),
                          int(knobs.get("words_per_thread", 0)), int(knobs.get("tile_out_cap", 0)),
                          int(knobs.get("walk_limit_words", 0)), int(knobs.get("result_cap", 0)),
                          int(knobs.get("flags", 0)))

    @_serialised
    def scan(self, min_motif_size, max_motif_size, min_repeats, min_span, **knobs):
        pr = self._params(min_motif_size, max_motif_size, min_repeats, min_span, knobs)
        n = ctypes.c_uint64()
        _check(lib().crf_scan(self._h, ctypes.byref(pr), ctypes.byref(n)))
        return n.value

    @_serialised
    def scan_gather(self, xchg, min_motif_size, max_motif_size, min_repeats, min_span, append=False, **knobs):
        """crf_scan_gather: scan + push of the rows to rank 0, asynchronous (Xchg.wait() tells how it went).
        append: the rows go after those of the job's earlier phases."""
        pr = self._params(min_motif_size, max_motif_size, min_repeats, min_span, knobs)
        _check(lib().crf_scan_gather(self._h, ctypes.byref(pr), xchg._h, int(bool(append))))

    @_serialised
    def push(self, xchg, append=False):
        """crf_xchg_push: rows of the last completed scan() -> rank 0 (asynchronous)."""
        _check(lib().crf_xchg_push(self._h, xchg._h, int(bool(append))))

    @_serialised
    def fetch(self, n):
        rec, start, end, k = (np.empty(n, np.uint32) for _ in range(4))
        _check(lib().crf_fetch(self._h, rec.ctypes.data, start.ctypes.data, end.ctypes.data, k.ctypes.data, n, 0))
        return rec, start, end, k

    @_serialised
    def fetch_device(self, rec_ptr, start_ptr, end_ptr, k_ptr, capacity):
        _check(lib().crf_fetch(self._h, rec_ptr, start_ptr, end_ptr, k_ptr, capacity, 1))

    @_serialised
    def fetch_host(self, rec_ptr, start_ptr, end_ptr, k_ptr, capacity):
        """Fetch into caller-owned host buffers given by address (e.g. pinned memory)."""
        _check(lib().crf_fetch(self._h, rec_ptr, start_ptr, end_ptr, k_ptr, capacity, 0))

    @_serialised
    def stats(self):
        out = ScanStats()
        _check(lib().crf_scan_stats(self._h, ctypes.byref(out)))
        return out

    @_serialised
    def fetch_open(self, cap=256):
        """(n, 5) uint32 rows (row index, record, start, end, k) of the open-ended results, in result order."""
        rows = np.zeros((cap, 5), np.uint32)
        n = ctypes.c_uint32()
        _check(lib().crf_fetch_open(self._h, rows.ctypes.data, cap, ctypes.byref(n)))
        return rows[:min(n.value, cap)]

    @_serialised
    def patch_end(self, row, new_end):
        _check(lib().crf_patch_end(self._h, int(row), int(new_end)))

    @_serialised
    def run_end(self, record, pos, k):
        out = ctypes.c_uint32()
        _check(lib().crf_run_end(self._h, int(record), int(pos), int(k), ctypes.byref(out)))
        return out.value

    @_serialised
    def interval_stop(self, min_motif_size, max_motif_size, end_pos, full_len):
        """crf_interval_stop: per record, where the interval-mode loop that ends its interval at end_pos breaks, the
        record being the prefix of a sequence of full_len bases.  int64 array: a position, STOP_TO_END or STOP_UNDECIDED."""
        end_pos = np.ascontiguousarray(end_pos, dtype=np.uint64)
        full_len = np.ascontiguousarray(full_len, dtype=np.uint64)
        if end_pos.shape != (self.n_records,) or full_len.shape != (self.n_records,):
            raise ValueError("end_pos and full_len need one entry per record of the load")
        stop = np.empty(self.n_records, np.int64)
        _check(lib().crf_interval_stop(self._h, int(min_motif_size), int(max_motif_size), ctypes.c_void_p(end_pos.ctypes.data),
                                       ctypes.c_void_p(full_len.ctypes.data), ctypes.c_void_p(stop.ctypes.data)))
        return stop

    @_serialised
    def close(self):
        if self._h:
            lib().crf_seq_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PackedPlanes:
    """2-bit planes + not-ACGT mask of `n_bases` positions (what crf_seq_load_packed uploads): three uint32 arrays (or raw
    pointers) of ceil(n_bases / 32) words and the sorted exotic list (position << 8 | upper-cased byte)."""

    def __init__(self, n_bases, H, L, NM, exotic, keep=None, on_device=False, runs=None):
        self.n_bases = int(n_bases)
        self.H, self.L, self.NM = H, L, NM
        self.exotic = np.ascontiguousarray(exotic, dtype=np.uint64)
        #: the mask as sorted runs of masked positions, shape (n, 2) -- when set, loads send these instead of the NM plane
        self.runs = None if runs is None else np.ascontiguousarray(runs, dtype=np.uint64).reshape(-1, 2)
        self.on_device = on_device
        self._keep = keep

        def ptr(a):
            return ctypes.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else int(a))
        self.H_ptr, self.L_ptr, self.NM_ptr = ptr(H), ptr(L), ptr(NM)

    @property
    def n_words(self):
        return (self.n_bases + 31) // 32

    @property
    def nbytes(self):
        """Bytes a load of all of it sends to the device."""
        if self.runs is not None:
            return 8 * self.n_words + 8 * int(self.runs.size) + 8 * int(self.exotic.size)
        return 12 * self.n_words + 8 * int(self.exotic.size)

    def with_runs(self, n_threads=0):
        """The same planes with the mask as runs (crf_mask_runs; host only)."""
        self.runs = mask_runs(self.NM_ptr, self.n_bases, n_threads)
        return self


def mask_runs(nm, n_bases, n_threads=0):
    """(n, 2) uint64 array of the maximal runs [from, to) of masked positions of an NM plane (array or pointer)."""
    ptr = nm if isinstance(nm, ctypes.c_void_p) else ctypes.c_void_p(nm.ctypes.data if isinstance(nm, np.ndarray) else int(nm))
    cap = 4096
    while True:
        runs = np.empty((cap, 2), np.uint64)
        n = ctypes.c_uint64()
        rc = lib().crf_mask_runs(ptr, int(n_bases), int(n_threads), ctypes.c_void_p(runs.ctypes.data), cap, ctypes.byref(n))
        if rc == CRF_ERR_CAPACITY:
            cap = int(n.value) + 16
            continue
        _check(rc)
        return runs[:n.value].copy()


def gunzip(data, use_zlib=False):
    """Host-only: gzip bytes -> bytes through crf_gunzip: the FASTA reader's decoder with zlib behind it (use_zlib False / 0),
    zlib alone (True / 1), or the reader's decoder alone (2: NotImplementedError for what it declines)."""
    data = bytes(data)
    src = ctypes.cast(ctypes.c_char_p(data), ctypes.c_void_p)
    cap = max(4 * len(data), 1 << 12)
    while True:
        out = np.empty(cap, np.uint8)
        n = ctypes.c_uint64()
        rc = lib().crf_gunzip(src, len(data), ctypes.c_void_p(out.ctypes.data), cap, ctypes.byref(n), int(use_zlib))
        if rc == CRF_ERR_CAPACITY:
            cap = int(n.value)
            continue
        _check(rc)
        return out[:n.value].tobytes()


def pack_ascii(bases, n_threads=0, out=None):
    """Host-only: ASCII bases (bytes / uint8 array) -> PackedPlanes (crf_pack_ascii; threaded, AVX2 when available).
    out: optional (H, L, NM) uint32 arrays to fill (e.g. views of pinned memory)."""
    if isinstance(bases, np.ndarray):
        if bases.dtype != np.uint8 or not bases.flags.c_contiguous:
            raise ValueError("bases must be a C-contiguous uint8 array")
        arr = bases
    else:
        arr = np.frombuffer(bytes(bases), dtype=np.uint8)
    n = arr.size
    nw = (n + 31) // 32
    H, L, NM = out if out is not None else (np.empty(max(nw, 1), np.uint32) for _ in range(3))
    cap = 1024
    while True:
        exo = np.empty(cap, np.uint64)
        n_exo = ctypes.c_uint64()
        rc = lib().crf_pack_ascii(ctypes.c_void_p(arr.ctypes.data if n else 0), n, int(n_threads), ctypes.c_void_p(H.ctypes.data),
                                  ctypes.c_void_p(L.ctypes.data), ctypes.c_void_p(NM.ctypes.data),
                                  ctypes.c_void_p(exo.ctypes.data), cap, ctypes.byref(n_exo))
        if rc == CRF_ERR_CAPACITY:
            cap = int(n_exo.value) + 16
            continue
        _check(rc)
        break
    return PackedPlanes(n, H, L, NM, exo[:n_exo.value].copy(), keep=arr)


class Xchg:
    """One rank's exchange block for the multi-GPU gather (crf_xchg, csrc/crf_xchg.cuh)."""

    def __init__(self, ctx, rank, world, row_cap):
        self.ctx, self.rank, self.world, self.row_cap = ctx, int(rank), int(world), int(row_cap)
        self._h = ctypes.c_void_p()
        _check(lib().crf_xchg_create(ctx._h, self.rank, self.world, self.row_cap, ctypes.byref(self._h)))

    def export(self):
        buf = ctypes.create_string_buffer(IPC_HANDLE_BYTES)
        _check(lib().crf_xchg_export(self._h, buf))
        return buf.raw

    def connect_ipc(self, peer, handle):
        buf = ctypes.create_string_buffer(bytes(handle), IPC_HANDLE_BYTES)
        _check(lib().crf_xchg_connect_ipc(self._h, int(peer), buf))

    def connect_local(self, peer, other):
        _check(lib().crf_xchg_connect_local(self._h, int(peer), other._h))

    def set_timeout(self, seconds):
        _check(lib().crf_xchg_set_timeout(self._h, float(seconds)))

    def set_compact(self, on=True):
        _check(lib().crf_xchg_set_compact(self._h, int(bool(on))))

    def wait(self):
        res = XchgResult()
        _check(lib().crf_xchg_wait(self._h, ctypes.byref(res)))
        return res

    def step_result(self, step):
        """The result of one of the last 64 steps a wait() has covered."""
        res = XchgResult()
        _check(lib().crf_xchg_step_result(self._h, int(step), ctypes.byref(res)))
        return res

    def fetch(self, n, first=0):
        rec, start, end, k = (np.empty(n, np.uint32) for _ in range(4))
        _check(lib().crf_xchg_fetch(self._h, rec.ctypes.data, start.ctypes.data, end.ctypes.data, k.ctypes.data,
                                    int(first), int(n), 0))
        return rec, start, end, k

    def fetch_to(self, rec_ptr, start_ptr, end_ptr, k_ptr, n, first=0, on_device=False):
        _check(lib().crf_xchg_fetch(self._h, rec_ptr, start_ptr, end_ptr, k_ptr, int(first), int(n), int(bool(on_device))))

    def patch_end(self, rows, new_end):
        rows = np.ascontiguousarray(rows, dtype=np.uint64)
        new_end = np.ascontiguousarray(new_end, dtype=np.uint32)
        _check(lib().crf_xchg_patch_end(self._h, rows.ctypes.data, new_end.ctypes.data, rows.size))

    def close(self):
        if self._h:
            lib().crf_xchg_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TwoBitSource:
    """The packed form of a .2bit file's records, what crf_seq_load_2bit and crf_write_rows_twobit take: dna (the file's
    bytes: a host uint8 array, a CUDA torch.uint8 tensor, or a device pointer), rec_byte[r] (the byte where record r's
    packed bases start), offsets (n_records + 1, the records' position space) and runs ((n, 2) N blocks in that space)."""

    def __init__(self, dna, rec_byte, offsets, runs, keep=None):
        self.dna, self.rec_byte, self.offsets, self.runs = dna, rec_byte, offsets, runs
        self._keep = keep

    def records(self, first, last):
        """Records [first, last) (the run list stays whole: a load ignores runs outside its records)."""
        return TwoBitSource(self.dna, self.rec_byte[first:last], self.offsets[first:last + 1], self.runs, self._keep)


class NibbleSource:
    """The packed form of a BAM file's reads, what crf_seq_load_nibbles and crf_write_rows_nibbles take: nib (4-bit codes
    =ACMGRSVTWYHKDBN, high nibble first: a host uint8 array, a CUDA torch.uint8 tensor, or a device pointer), rec_byte[r]
    (the byte where record r's codes start), offsets (n_records + 1, the records' position space) and exotic (codes other
    than A, C, G, T, N as position << 8 | letter, ascending, in that space)."""

    def __init__(self, nib, rec_byte, offsets, exotic, keep=None):
        self.nib, self.rec_byte, self.offsets, self.exotic = nib, rec_byte, offsets, exotic
        self._keep = keep

    def records(self, first, last):
        """Records [first, last) (the exotic list stays whole: a load ignores entries outside its records)."""
        return NibbleSource(self.nib, self.rec_byte[first:last], self.offsets[first:last + 1], self.exotic, self._keep)


class Fasta:
    """A FASTA, FASTQ, .2bit or BAM file read by the native reader (crf_fasta_open): `bases` (uint8 view of all records
    back to back, owned by the library until close(); a .2bit or BAM file's text is decoded on first use), `offsets`
    (n_records+1, uint64), `names` (list of str), `names_blob` (NUL-separated, as crf_write_rows takes them), `format`
    ("fasta" / "fastq" / "2bit" / "bam") and `quals` (a FASTQ or BAM file's qualities as a uint8 view laid out like
    `bases`, or None)."""

    def __init__(self, path, n_threads=0, pinned=False, qualities=False):
        """pinned: False / True (page-locked base buffer and planes) / 2 (page-locked planes only: the text stays pageable).
        qualities: keep a FASTQ or BAM file's qualities (else they are dropped: no host memory for them)."""
        self._h = ctypes.c_void_p()
        _check(lib().crf_fasta_open(os.fsencode(path), n_threads, int(pinned) | (4 if qualities else 0),
                                    ctypes.byref(self._h)))
        n_rec, total, pin = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_int()
        _check(lib().crf_fasta_info(self._h, ctypes.byref(n_rec), ctypes.byref(total), ctypes.byref(pin)))
        offsets, names, nbytes = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_uint64()
        _check(lib().crf_fasta_index(self._h, ctypes.byref(offsets), ctypes.byref(names), ctypes.byref(nbytes)))
        self.n_records, self.total_bases, self.pinned = n_rec.value, total.value, bool(pin.value)
        self._bases = None
        self.offsets = np.ctypeslib.as_array(ctypes.cast(offsets, ctypes.POINTER(ctypes.c_uint64)),
                                             shape=(self.n_records + 1,)).copy()
        self.names_blob = ctypes.string_at(names, nbytes.value) if nbytes.value else b""
        self._names = None
        fmt, quals = ctypes.c_int(), ctypes.c_void_p()
        _check(lib().crf_fasta_format(self._h, ctypes.byref(fmt)))
        _check(lib().crf_fasta_quals(self._h, ctypes.byref(quals)))
        self.format = {1: "fastq", 2: "2bit", 3: "bam"}.get(fmt.value, "fasta")
        self.quals = np.ctypeslib.as_array(ctypes.cast(quals, ctypes.POINTER(ctypes.c_uint8)),
                                           shape=(max(self.total_bases, 1),))[:self.total_bases] if quals.value else None

    @property
    def bases(self):
        """uint8 view of all records back to back (crf_fasta_data; a .2bit or BAM file's text is decoded on the first
        call)."""
        if self._bases is None and self._h:
            bases = ctypes.c_void_p()
            _check(lib().crf_fasta_data(self._h, ctypes.byref(bases), None, None, None))
            self._bases = np.ctypeslib.as_array(ctypes.cast(bases, ctypes.POINTER(ctypes.c_uint8)),
                                                shape=(max(self.total_bases, 1),))[:self.total_bases]
        return self._bases

    def _codes(self, fn, per_byte):
        """(codes, rec_byte, list address, list length) from crf_fasta_twobit or crf_fasta_nibbles (ValueError for any other
        format).  codes is a view of the handle's bytes up to the end of the last record's, valid until close()."""
        codes, rec_byte, lst, n = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_uint64()
        _check(fn(self._h, ctypes.byref(codes), ctypes.byref(rec_byte), ctypes.byref(lst), ctypes.byref(n)))
        rb = _u64s(rec_byte, self.n_records)
        lengths = np.diff(self.offsets.astype(np.int64))
        size = int((rb.astype(np.int64) + (lengths + per_byte - 1) // per_byte).max()) if self.n_records else 0
        view = np.ctypeslib.as_array(ctypes.cast(codes, ctypes.POINTER(ctypes.c_uint8)), shape=(max(size, 1),))[:size] \
            if codes.value else np.zeros(0, np.uint8)
        return view, rb, lst, n.value

    def twobit(self):
        """TwoBitSource of a .2bit file (crf_fasta_twobit; ValueError for any other format).  dna is a view of the handle's
        bytes, valid until close()."""
        dna, rb, runs, n_runs = self._codes(lib().crf_fasta_twobit, 4)
        return TwoBitSource(dna, rb, self.offsets, _u64s(runs, 2 * n_runs).reshape(-1, 2), keep=self)

    def nibbles(self):
        """NibbleSource of a BAM file (crf_fasta_nibbles; ValueError for any other format).  nib is a view of the handle's
        codes, valid until close()."""
        nib, rb, ex, n_ex = self._codes(lib().crf_fasta_nibbles, 2)
        return NibbleSource(nib, rb, self.offsets, _u64s(ex, n_ex), keep=self)

    @property
    def names(self):
        """Record names as str (decoded on first use: a reads file has millions)."""
        if self._names is None:
            self._names = [x.decode("utf-8", "replace") for x in self.names_blob.split(b"\0")[:self.n_records]]
        return self._names

    def record(self, i):
        """uint8 view of record i."""
        return self.bases[int(self.offsets[i]):int(self.offsets[i + 1])]

    def packed(self, n_threads=0):
        """PackedPlanes of the whole file (crf_fasta_packed: made on first use, page-locked when the reader is)."""
        H, L, NM, ex = (ctypes.c_void_p() for _ in range(4))
        n_ex = ctypes.c_uint64()
        _check(lib().crf_fasta_packed(self._h, int(n_threads), ctypes.byref(H), ctypes.byref(L), ctypes.byref(NM),
                                      ctypes.byref(ex), ctypes.byref(n_ex)))
        return PackedPlanes(self.total_bases, H.value, L.value, NM.value, _u64s(ex, n_ex.value), keep=self).with_runs(n_threads)

    def close(self):
        if self._h:
            self._bases = self.quals = None
            lib().crf_fasta_close(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _u64s(ptr, n):
    """A copy of n uint64 at a library address (an empty array when n is 0)."""
    return np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(ctypes.c_uint64)), shape=(n,)).copy() \
        if n else np.zeros(0, np.uint64)


def _write_rows_with(fn, path, names, src, record, start, end, k, tsv, append):
    """One of the native rows writers: fn(path, append, tsv, names blob, *src, record, start, end, k, n_rows, &bytes), where
    src are the arguments that say where the motif is read.  names: list of str, or the NUL-separated blob."""
    if isinstance(names, (bytes, bytearray)):
        blob = bytes(names)
    else:
        blob = b"".join(n.encode("utf-8") + b"\0" for n in names) if names is not None else None
    arrs = [np.ascontiguousarray(a, dtype=np.uint32) for a in (record, start, end, k)]
    nbytes = ctypes.c_uint64()
    _check(fn(os.fsencode(path), int(append), int(tsv),
              ctypes.cast(ctypes.c_char_p(blob), ctypes.c_void_p) if blob is not None else None, *src,
              *(ctypes.c_void_p(a.ctypes.data) for a in arrs), len(arrs[0]), ctypes.byref(nbytes)))
    return nbytes.value


def write_rows(path, names, bases, offsets, record, start, end, k, tsv=False, append=False, origin=None):
    """Native BED / TSV writer (crf_write_rows).  bases: bytes or uint8 array with all records back to back;
    names: list of str, or the NUL-separated blob.  origin: per record, a uint64 added to the printed start and end
    (crf_write_rows_at; the rows of a record longer than 2^32 bases are written unit by unit, relative to each unit)."""
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    if isinstance(bases, np.ndarray):
        bptr = bases.ctypes.data
    else:
        bptr = ctypes.cast(ctypes.c_char_p(bases), ctypes.c_void_p).value or 0
    src = (ctypes.c_void_p(bptr), ctypes.c_void_p(offsets.ctypes.data))
    if origin is None:
        return _write_rows_with(lib().crf_write_rows, path, names, src, record, start, end, k, tsv, append)
    origin = np.ascontiguousarray(origin, dtype=np.uint64)
    return _write_rows_with(lib().crf_write_rows_at, path, names, (*src, ctypes.c_void_p(origin.ctypes.data)), record, start,
                            end, k, tsv, append)


def write_rows_twobit(path, names, dna, rec_byte, record, start, end, k, tsv=False, append=False):
    """crf_write_rows_twobit: write_rows for records of a .2bit file, the motif read from the packed bytes (dna: host uint8
    array of the file's bytes, rec_byte[r]: where record r's bases start, as TwoBitSource has them)."""
    rec_byte = np.ascontiguousarray(rec_byte, dtype=np.uint64)
    src = (ctypes.c_void_p(_host_bytes("dna", dna)[0]), ctypes.c_void_p(rec_byte.ctypes.data))
    return _write_rows_with(lib().crf_write_rows_twobit, path, names, src, record, start, end, k, tsv, append)


def write_rows_nibbles(path, names, nib, rec_byte, record, start, end, k, tsv=False, append=False):
    """crf_write_rows_nibbles: write_rows for reads of a BAM file, the motif read from the 4-bit codes (nib: host uint8
    array, rec_byte[r]: where record r's codes start, as NibbleSource has them)."""
    rec_byte = np.ascontiguousarray(rec_byte, dtype=np.uint64)
    src = (ctypes.c_void_p(_host_bytes("nib", nib)[0]), ctypes.c_void_p(rec_byte.ctypes.data))
    return _write_rows_with(lib().crf_write_rows_nibbles, path, names, src, record, start, end, k, tsv, append)


def _check_extent(what, buf, rec_byte, offsets, per_byte):
    """ValueError unless every non-empty record's packed bytes, rec_byte[r] .. rec_byte[r] + ceil(length / per_byte), lie
    inside buf (not checked for a device pointer given as an int: its size is unknown)."""
    if isinstance(buf, int):
        return
    size = buf.numel() if hasattr(buf, "numel") else len(buf)
    lengths = np.diff(offsets.astype(np.int64))
    if (lengths < 0).any():
        raise ValueError("offsets must be non-decreasing")
    full = lengths > 0
    if full.any():
        end = rec_byte.astype(np.int64)[full] + (lengths[full] + per_byte - 1) // per_byte
        if int(end.max()) > size:
            raise ValueError(f"a record's bytes run past the end of {what} ({int(end.max())} > {size} bytes)")


def _source_bytes(what, buf, on_device):
    """(address, on_device) of the bytes a .2bit or BAM load reads: a torch uint8 tensor (a CUDA one is read on the
    device), a device pointer (int, with on_device=True), or host bytes / a uint8 array."""
    if hasattr(buf, "data_ptr"):
        if str(buf.dtype) != "torch.uint8" or not buf.is_contiguous():
            raise ValueError(f"{what} must be a contiguous torch.uint8 tensor")
        if buf.is_cuda:
            import torch
            torch.cuda.current_stream(buf.device).synchronize()     # its bytes are written before the upload
            on_device = True
        return buf.data_ptr(), on_device
    if isinstance(buf, int):
        if not on_device:
            raise ValueError(f"a pointer as {what} needs on_device=True")
        return buf, on_device
    return _host_bytes(what, buf)[0], on_device


def _host_bytes(what, buf):
    """(address, size) of bytes or a 1-d C-contiguous uint8 array."""
    if isinstance(buf, np.ndarray):
        if buf.dtype != np.uint8 or buf.ndim != 1 or not buf.flags.c_contiguous:
            raise ValueError(f"{what} must be a 1-d C-contiguous uint8 array")
        return buf.ctypes.data, buf.size
    return ctypes.cast(ctypes.c_char_p(buf), ctypes.c_void_p).value or 0, len(buf)


def _masked_args(names, bases, offsets, mask, quals=None):
    """The checked arguments both masked writers take: names blob, bases address, offsets, mask (and quals address)."""
    blob = bytes(names) if isinstance(names, (bytes, bytearray)) else b"".join(n.encode("utf-8") + b"\0" for n in names)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    if offsets.ndim != 1 or offsets.size < 1:
        raise ValueError("offsets must hold n_records + 1 entries")
    mask = np.ascontiguousarray(mask, dtype=np.uint32)
    n = int(offsets[-1])
    bptr, size = _host_bytes("bases", bases)
    if n > size or 32 * mask.size < n:
        raise ValueError(f"offsets reach base {n}; bases hold {size} and the mask {32 * mask.size}")
    qptr = None
    if quals is not None:
        qptr, qsize = _host_bytes("quals", quals)
        if n > qsize:
            raise ValueError(f"offsets reach base {n}; quals hold {qsize}")
    return blob, bptr, offsets, mask, qptr


def write_fasta_masked(path, names, bases, offsets, mask, hard=False, line_width=60):
    """Native repeat-masked FASTA writer (crf_write_fasta_masked).  names: list of str or the NUL-separated blob; bases:
    bytes or uint8 array with all records back to back, record r = bases[offsets[r]:offsets[r+1]]; mask: uint32 words,
    bit p for bases[p] (Context.mask_rows).  hard: masked bases become N instead of lower case."""
    blob, bptr, offsets, mask, _ = _masked_args(names, bases, offsets, mask)
    nbytes = ctypes.c_uint64()
    _check(lib().crf_write_fasta_masked(os.fsencode(path), ctypes.cast(ctypes.c_char_p(blob), ctypes.c_void_p),
                                        ctypes.c_void_p(bptr), ctypes.c_void_p(offsets.ctypes.data), offsets.size - 1,
                                        ctypes.c_void_p(mask.ctypes.data), int(bool(hard)), int(line_width),
                                        ctypes.byref(nbytes)))
    return nbytes.value


def write_fastq_masked(path, names, bases, quals, offsets, mask, hard=False):
    """Native repeat-masked FASTQ writer (crf_write_fastq_masked): as write_fasta_masked, with quals (bytes or uint8 array
    laid out like bases, Fasta.quals) written unchanged on each record's quality line."""
    blob, bptr, offsets, mask, qptr = _masked_args(names, bases, offsets, mask, quals)
    nbytes = ctypes.c_uint64()
    _check(lib().crf_write_fastq_masked(os.fsencode(path), ctypes.cast(ctypes.c_char_p(blob), ctypes.c_void_p),
                                        ctypes.c_void_p(bptr), ctypes.c_void_p(qptr), ctypes.c_void_p(offsets.ctypes.data),
                                        offsets.size - 1, ctypes.c_void_p(mask.ctypes.data), int(bool(hard)),
                                        ctypes.byref(nbytes)))
    return nbytes.value
