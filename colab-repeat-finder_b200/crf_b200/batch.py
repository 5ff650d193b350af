"""detect_repeats_batch() and scan_batch(): many independent sequences (reads, contigs, exons) in one device load per group
of sequences instead of one load, scan, fetch and stream sync per sequence.

Sequence i gives exactly what api.detect_repeats(s_i, filter_settings) gives: the same rows, or the same exception
(DESIGN.md section 6, "Many sequences").  Full mode is scan_batch: the sequences become the records of multi-record
loads, grouped to fit crf_load_limit, one crf_scan each.  With interval attributes every sequence is one interval of the
packed concatenation and the batch goes through intervals.run_intervals.
"""
import sys

import numpy as np

from . import _cabi, api, intervals
from .cli import group_records

#: what the last detect_repeats_batch() / scan_batch() call did: device loads, and the sequences it left to api.detect_repeats
#: one call each (min_repeats == 1, a sequence longer than one load, the interval cases run_intervals does not batch)
last_stats = {}

#: layout positions one load holds (crf_load_limit); a name of its own so that tests can shrink it for this module alone
_load_limit = _cabi.load_limit

_USE_BATCH = "use detect_repeats_batch, which runs such input through detect_repeats"


def _has_interval(fs):
    return hasattr(fs, "interval_start_0based") or hasattr(fs, "interval_end")


def scan_batch(bases, offsets, filter_settings, device=None, **knobs):
    """Full mode for many records at once, as integer columns.

    bases: the records back to back -- bytes / bytearray / a C-contiguous numpy uint8 array on the host, or a 1-d contiguous
    CUDA torch.uint8 tensor.  offsets: n + 1 non-decreasing record boundaries into bases (host array-like or a torch tensor).
    Returns (record, start, end, k), uint32 columns sorted by (record, start, end): the rows api.detect_repeats gives
    record bases[offsets[r]:offsets[r+1]], start / end relative to the record.  Host input gives numpy arrays.

    A CUDA tensor gives CUDA torch.uint32 tensors on the same device, and neither the bases nor the rows cross PCIe (only
    the offsets): each group of records is loaded from the tensor (crf_seq_load_ascii with a device pointer) and its rows are
    fetched device to device into tensors allocated by torch.  device=None means the tensor's device.  Stream ordering: the
    caller's current torch stream is synchronised before the first load, so work still queued there that writes `bases`
    has finished; the library then runs on the context's own stream, and every fetch ends in a sync of that stream, so the
    returned tensors are complete when this returns.

    Interval attributes on filter_settings, min_repeats == 1 and a record longer than one device load raise
    NotImplementedError: detect_repeats_batch handles them."""
    api.validate_filter_settings(filter_settings)
    kmin, kmax = int(filter_settings.min_motif_size), int(filter_settings.max_motif_size)
    min_repeats, min_span = int(filter_settings.min_repeats), int(filter_settings.min_span)
    if _has_interval(filter_settings):
        raise NotImplementedError(f"scan_batch runs full mode only (no interval attributes); {_USE_BATCH}")
    if min_repeats == 1:
        raise NotImplementedError(f"scan_batch does not run min_repeats == 1; {_USE_BATCH}")
    torch = sys.modules.get("torch")
    on_device = torch is not None and isinstance(bases, torch.Tensor)
    if on_device:
        if not bases.is_cuda or bases.dtype != torch.uint8 or bases.dim() != 1 or not bases.is_contiguous():
            raise ValueError("bases must be a 1-d contiguous CUDA torch.uint8 tensor, or host bytes / a numpy uint8 array")
        device = bases.device.index if device is None else device
        if bases.device.index != device:
            raise ValueError(f"bases is on cuda:{bases.device.index}, the scan would run on device {device}")
        if isinstance(offsets, torch.Tensor):
            offsets = offsets.cpu().numpy()
        n_bases = bases.numel()
    else:
        if not isinstance(bases, np.ndarray):
            bases = np.frombuffer(bases, dtype=np.uint8)
        if bases.dtype != np.uint8 or bases.ndim != 1 or not bases.flags.c_contiguous:
            raise ValueError("bases must be a 1-d C-contiguous numpy uint8 array")
        n_bases = bases.size
    offsets = np.asarray(offsets)
    if offsets.ndim != 1 or offsets.size < 1 or offsets.dtype.kind not in "iu":
        raise ValueError("offsets must be a 1-d integer array of n_records + 1 boundaries")
    offsets = offsets.astype(np.int64)
    lengths = np.diff(offsets)
    if offsets[0] < 0 or offsets[-1] > n_bases or (lengths < 0).any():
        raise ValueError(f"offsets must be non-decreasing boundaries inside the {n_bases} bases")
    limit = _load_limit(kmax)
    too_long = np.flatnonzero(lengths + kmax > limit)
    if too_long.size:
        raise NotImplementedError(f"record {int(too_long[0])} ({int(lengths[too_long[0]])} bases) is longer than one device "
                                  f"load; {_USE_BATCH}")
    ctx = api.get_context(device)
    if on_device:
        torch.cuda.current_stream(bases.device).synchronize()
    else:
        planes = _cabi.pack_ascii(bases).with_runs()
    parts, loads = [], 0
    for first, last in group_records(lengths, kmax, limit):
        base0 = int(offsets[first])
        if int(offsets[last]) == base0:
            continue                                     # empty records only: no rows
        if on_device:
            seq = ctx.load(bases.data_ptr() + base0, offsets[first:last + 1] - base0, max_motif_cap=kmax, on_device=True)
        else:
            seq = ctx.load_packed(planes, offsets[first:last + 1], max_motif_cap=kmax)
        loads += 1
        with seq:
            if first:                                    # rows name the batch's record, not the load's
                seq.set_output_map(out_record=np.arange(first, last, dtype=np.uint32))
            nrow = seq.scan(kmin, kmax, min_repeats, min_span, **knobs)
            if on_device:
                cols = torch.empty((4, nrow), dtype=torch.int32, device=bases.device)      # uint32 bits
                seq.fetch_device(*(int(c.data_ptr()) for c in cols), nrow)
            else:
                cols = np.stack(seq.fetch(nrow))
        parts.append(cols)
    last_stats.clear()
    last_stats.update(loads=loads, fallback=0)
    if on_device:
        cols = torch.cat(parts, dim=1) if len(parts) > 1 else parts[0] if parts else \
            torch.empty((4, 0), dtype=torch.int32, device=bases.device)
        return tuple(cols.view(torch.uint32))
    cols = np.concatenate(parts, axis=1) if parts else np.zeros((4, 0), np.uint32)
    return tuple(cols)


def _rows_as_tuples(seqs, outcome, origin, rec, start, end, k):
    """Per sequence: outcome[i] if it is not None, else its rows (rec == i) as (start, end, motif) tuples, start / end shifted
    by origin[i] and the motif cut from the caller's own object, as api.detect_repeats builds them."""
    bounds = np.searchsorted(rec, np.arange(len(seqs) + 1)).tolist()
    start, end, k, origin = start.tolist(), end.tolist(), k.tolist(), origin.tolist()
    out = []
    for i, o in enumerate(outcome):
        if o is not None:
            out.append(o)
            continue
        s, a0 = seqs[i], origin[i]
        out.append([(start[j] + a0, end[j] + a0, api._upper_slice(s, start[j] + a0, k[j])) for j in range(bounds[i], bounds[i + 1])])
    return out


def detect_repeats_batch(sequences, filter_settings, device=None, **knobs):
    """[api.detect_repeats(s, filter_settings, device=device, **knobs) for s in sequences], computed with one device load per
    group of sequences.  sequences: any iterable of str / bytes.  If a sequence raises, raises what the first such sequence
    (in input order) raises.

    Full mode runs scan_batch over the packed concatenation; with interval attributes every sequence is the interval
    [interval_start_0based, interval_end) of itself (defaults 0 and its length) and the batch goes through
    intervals.run_intervals.  min_repeats == 1, a sequence longer than one load, and the intervals run_intervals does not
    batch go through api.detect_repeats one call each (last_stats["fallback"] counts them)."""
    seqs = list(sequences)
    if not seqs:
        return []                                        # (the per-sequence loop never reads the settings)
    api.validate_filter_settings(filter_settings)
    kmax = int(filter_settings.max_motif_size)
    raws, encode_error = [], None
    for s in seqs:
        try:
            raws.append(api._encode(s))
        except Exception as exc:                         # noqa: BLE001 (the loop stops here: later sequences never run)
            encode_error = exc
            break
    seqs = seqs[:len(raws)]

    def single(i):
        return api.detect_repeats(seqs[i], filter_settings, device=device, **knobs)

    last_stats.clear()
    last_stats.update(loads=0, fallback=0)
    out = []
    if int(filter_settings.min_repeats) == 1:
        last_stats["fallback"] = len(seqs)
        out = [single(i) for i in range(len(seqs))]
    elif seqs:
        lengths = np.fromiter(map(len, raws), dtype=np.int64, count=len(raws))
        if not _has_interval(filter_settings):
            fit = np.flatnonzero(lengths + kmax <= _load_limit(kmax))
            blob = b"".join(raws) if fit.size == len(raws) else b"".join(raws[i] for i in fit.tolist())
            rec, start, end, k = scan_batch(blob, np.concatenate([[0], np.cumsum(lengths[fit])]), filter_settings, device,
                                            **knobs)
            outcome = [None] * len(seqs)
            long_ones = np.setdiff1d(np.arange(len(seqs)), fit).tolist()
            for i in long_ones:
                outcome[i] = single(i)
            last_stats["fallback"] = len(long_ones)
            out = _rows_as_tuples(seqs, outcome, np.zeros(len(seqs), np.int64), fit[rec.astype(np.int64)], start, end, k)
        else:
            a = int(getattr(filter_settings, "interval_start_0based", 0))
            b = np.full(len(seqs), int(filter_settings.interval_end)) if hasattr(filter_settings, "interval_end") else lengths
            planes = _cabi.pack_ascii(b"".join(raws)).with_runs()
            outcome, origin, iv, start, end, k = intervals.run_intervals(
                planes, np.cumsum(lengths) - lengths, lengths, np.full(len(seqs), a), b, filter_settings, device, knobs, single,
                load_limit=_load_limit(kmax))
            last_stats.update(loads=intervals.last_stats["loads"], fallback=intervals.last_stats["fallback"])
            for o in outcome:
                if isinstance(o, BaseException):
                    raise o
            out = _rows_as_tuples(seqs, outcome, origin, iv, start, end, k)
    if encode_error is not None:
        raise encode_error
    return out
