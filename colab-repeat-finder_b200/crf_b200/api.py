"""detect_repeats(): host-side mirror of the reference's scan driver on top of libcrf.so.

Same signature, return value and exceptions as the reference's perfect_repeat_finder.py:10-81.
All per-base work (the tracker loop, prf:66-74 / utils/perfect_repeat_tracker.py:43-101) runs in
the CUDA kernels behind crf_b200._cabi; this module only validates arguments, slices the
interval, and turns (start, end, k) triples back into the reference's tuples.
"""
import os
import threading

import numpy as np

from . import _cabi

_ctx_lock = threading.Lock()
_ctx = {}


def default_device():
    """CRF_DEVICE, else LOCAL_RANK (one process per GPU under torchrun), else 0."""
    for var in ("CRF_DEVICE", "LOCAL_RANK"):
        if os.environ.get(var, "") != "":
            return int(os.environ[var])
    return 0


def get_context(device=None):
    """Process-wide context per device (created on first use)."""
    device = default_device() if device is None else device
    with _ctx_lock:
        if device not in _ctx:
            _ctx[device] = _cabi.Context(device)
        return _ctx[device]


def validate_filter_settings(fs):
    """The four checks of perfect_repeat_finder.py:23-30 (same messages; bare getattr raises
    AttributeError when an attribute is missing, like the reference)."""
    if not getattr(fs, "min_motif_size") or fs.min_motif_size < 1:
        raise ValueError(f"min_motif_size is set to {fs.min_motif_size}. It must be at least 1.")
    if not getattr(fs, "max_motif_size") or fs.max_motif_size < fs.min_motif_size:
        raise ValueError(f"max_motif_size is set to {fs.max_motif_size}. It must be at least min_motif_size.")
    if not getattr(fs, "min_repeats") or fs.min_repeats < 1:
        raise ValueError(f"min_repeats is set to {fs.min_repeats}. It must be at least 1.")
    if not getattr(fs, "min_span") or fs.min_span < 1:
        raise ValueError(f"min_span is set to {fs.min_span}. It must be at least 1.")


def _encode(seq):
    """str -> bytes with one byte per symbol.  ASCII is upper-cased on the device; other text is
    upper-cased here (str.upper, prf:33) and must stay within latin-1."""
    if isinstance(seq, (bytes, bytearray, memoryview)):
        return bytes(seq)
    if seq.isascii():
        return seq.encode("ascii")
    up = seq.upper()
    if len(up) != len(seq):
        raise NotImplementedError("input contains characters whose upper-case form has a different length")
    try:
        return up.encode("latin-1")
    except UnicodeEncodeError as exc:
        raise NotImplementedError("input contains characters outside latin-1; the GPU path stores one byte "
                                  "per symbol") from exc


def _upper_slice(seq, start, k):
    piece = seq[start:start + k]
    if isinstance(piece, (bytes, bytearray, memoryview)):
        return bytes(piece).decode("latin-1").upper()
    return piece.upper()


def scan_arrays(raw, kmin, kmax, min_repeats, min_span, device=None, **knobs):
    """One record (bytes / uint8 array) -> (start, end, k), sorted by (start, end).  uint32 arrays when the record fits
    one device load; a longer record is cut into units spread over several loads (multi.RankScan) and start / end come
    back as uint64."""
    ctx = get_context(device)
    if len(raw) + kmax <= _cabi.load_limit(kmax):
        with ctx.load(raw, max_motif_cap=kmax) as seq:
            n = seq.scan(kmin, kmax, min_repeats, min_span, **knobs)
            _, start, end, k = seq.fetch(n)
        return start, end, k
    from . import multi, partition
    if not isinstance(raw, np.ndarray):
        raw = np.frombuffer(raw, dtype=np.uint8)
    rs = multi.RankScan(ctx, multi.ThreadComm.split(1)[0], raw, [0], [len(raw)], kmin, kmax, min_repeats, min_span,
                        chunk=partition.DEFAULT_CHUNK, halo=partition.DEFAULT_HALO, knobs=knobs)
    try:
        rs.step_async()
        rs.finish()
        _, start, end, k = rs.fetch()
    finally:
        rs.close()
    return start, end, k


def _n_trim(raw, a, b):
    """prf:40-44 on bytes: returns (a, b, Ltrunc)."""
    n = len(raw)
    arr = np.frombuffer(raw, dtype=np.uint8)
    is_n = (arr == ord("N")) | (arr == ord("n"))
    ltrunc = n
    while a < b and is_n[a]:            # raises IndexError past the end, like the reference
        a += 1
    while b > a and is_n[b - 1]:
        b -= 1
        ltrunc -= 1
    return a, b, ltrunc


def _interval_stop_position(ctx, s, end_position, kmin, kmax, knobs):
    """Position T after which the reference's lock-step loop breaks (prf:73-74), or None if it
    runs to the end of `s`.  A tracker is mid-repeat (trk:63-65) at t iff >= k consecutive ones of
    M_k end at min(t, L-k-1); those are read off a probe scan that keeps every run of >= k ones
    (min_repeats=2, min_span=1, no primitivity filter) over a window just past the interval end."""
    L = len(s)
    E = end_position
    if E >= L - 1:
        return None
    window = 256
    while True:
        # tracker k at t has its last compare at j = min(t, L-k-1) and needs the k compares ending there: the window
        # starts k before that -- before E+1 for most, but up to 2k before the END for a tracker that has already
        # stopped (L-k-1 < E+1, i.e. the interval ends within kmax of the end of the sequence)
        ws = max(0, min(E + 1 - kmax, L - 2 * kmax))
        hi_t = min(L - 1, E + window)                   # last t examined
        we = min(L, hi_t + 1 + kmax)
        with ctx.load(s[ws:we], max_motif_cap=kmax) as seq:
            n = seq.scan(kmin, kmax, 2, 1, **{**knobs, "flags": int(knobs.get("flags", 0)) | _cabi.SCAN_NO_PRIMITIVITY})
            _, st, en, kk = seq.fetch(n)
        st = st.astype(np.int64) + ws
        i0 = en.astype(np.int64) + ws - kk
        kk = kk.astype(np.int64)
        lo = st + kk - 1                                # first t at which the tracker is mid-repeat
        hi = i0 - 1                                     # last such t ...
        if we == L:                                     # ... forever once the tracker has stopped
            hi = np.where(i0 == L - kk, np.int64(L), hi)
        diff = np.zeros(hi_t - E + 2, dtype=np.int64)   # coverage of t in [E+1, hi_t]
        lo_c = np.clip(lo, E + 1, hi_t + 1) - (E + 1)
        hi_c = np.clip(hi + 1, E + 1, hi_t + 1) - (E + 1)
        keep = hi_c > lo_c
        np.add.at(diff, lo_c[keep], 1)
        np.add.at(diff, hi_c[keep], -1)
        covered = np.cumsum(diff)[:hi_t - E] > 0        # one entry per t in [E+1, hi_t]
        free = np.flatnonzero(~covered)
        if free.size:
            return E + 1 + int(free[0])
        if hi_t >= L - 1:
            return None
        window *= 4


def _is_primitive(motif):
    """not consists_of_perfect_repeats(motif) (trk:108-142): no proper divisor of len(motif) is a period."""
    n = len(motif)
    return not any(n % d == 0 and motif == motif[:d] * (n // d) for d in range(1, n // 2 + 1))


def _position0_candidates(s, kmin, kmax, min_span, stop):
    """min_repeats == 1: what the trackers emit for the run that starts at position 0 when it has fewer than k-1
    matches -- the one place where trk:87 (`seq[i+1] == seq[i+1-period]`) reads negative indices, i.e. the END of
    the sequence.  At most one candidate per motif size, each a walk of < 2k symbol compares; everything else
    the reference reports comes from the GPU scan (a run with st > 0 and r < k-1 can never pass trk:91, see
    DESIGN.md section 6).  Yields (end, motif_length); raises IndexError where trk:87 does."""
    L = len(s)
    N = ord("N")
    for k in range(kmin, kmax + 1):
        reach = max(L - k, 0)                            # where tracker k stands when the loop ends (trk:50) ...
        if stop is not None:
            reach = min(reach, stop + 1)                 # ... or where the early break left it (prf:73-74)
        r = 0
        while r < min(reach, k - 1) and s[r] == s[r + k] and s[r] != N:
            r += 1
        if r >= k - 1:
            continue                                     # an ordinary run: reported by the scan
        motif = s[0:k]
        if N in motif:                                   # trk:83
            continue
        run, i = r + 1, r
        if run + k - 1 >= min_span:                      # trk:86 (min_repeats * period == k always holds)
            while i < L - 1:
                j = i + 1 - k
                if j < -L:
                    raise IndexError("string index out of range")
                if s[i + 1] != s[j]:
                    break
                i += 1
                run += 1
        if run >= min_span and run >= k and _is_primitive(motif):      # trk:91,98
            yield i + 1, len(motif)


def _detect_single_copy(input_sequence, raw, filter_settings, kmin, kmax, min_span, ctx, device, knobs):
    """detect_repeats for min_repeats == 1 (SURVEY Appendix A.4; derivation in DESIGN.md section 6)."""
    if kmin == 1 and min_span <= 1:
        raise NotImplementedError(
            "min_repeats == 1 with min_motif_size == 1 and min_span == 1 reports every single base as a repeat "
            "(perfect_repeat_tracker.py:86-91); this degenerate setting is not implemented on the GPU path")
    n = len(raw)
    a = int(getattr(filter_settings, "interval_start_0based", 0))
    b = int(getattr(filter_settings, "interval_end", n))
    if a < 0 or b < 0:
        raise NotImplementedError("negative interval coordinates are not supported")
    a, b, ltrunc = _n_trim(raw, a, b)                    # the wrap-around reads the trimmed string's end: trim for real
    s = raw[a:ltrunc].upper()                            # the symbol compares below are on the upper-cased string (prf:33)
    L = len(s)
    stop = _interval_stop_position(ctx, s, b - a, kmin, kmax, knobs)
    if stop is not None and b == L and stop + 1 < L - kmin:
        raise AssertionError(f"{kmin}bp motif RepeatTracker did not reach end of the sequence")      # prf:77-78
    rows = {}
    if L:
        start, end, k = scan_arrays(s, kmin, kmax, 1, min_span, device=device, **knobs)
        start, end, k = start.astype(np.int64), end.astype(np.int64), k.astype(np.int64)
        if stop is not None:
            # processed mismatch positions, plus what done() (prf:79) makes of a tracker the break left with exactly
            # k-1 matches behind it: its pre-filter (trk:86) sees 2k-1 bases, then trk:87 follows the run to its end
            keep = (end - k <= stop) | ((start == stop + 2 - k) & (2 * k - 1 >= min_span))
            start, end, k = start[keep], end[keep], k[keep]
        rows = {(s0, e0): k0 for s0, e0, k0 in zip(start.tolist(), end.tolist(), k.tolist())}
    for e0, k0 in _position0_candidates(s, kmin, kmax, min_span, stop):
        if k0 < rows.get((0, e0), k0 + 1):               # same interval: the shorter motif stays (trk:94-96)
            rows[(0, e0)] = k0
    return [(s0 + a, e0 + a, _upper_slice(input_sequence, s0 + a, k0)) for (s0, e0), k0 in sorted(rows.items())]


def detect_repeats(input_sequence, filter_settings, verbose=False, show_progress_bar=False, debug=False,
                   device=None, **knobs):
    """Detect perfect tandem repeats.  Drop-in for the reference's detect_repeats (prf:10-81).

    Returns a list of (start_0based, end, motif) tuples sorted by (start, end).
    """
    validate_filter_settings(filter_settings)
    kmin, kmax = int(filter_settings.min_motif_size), int(filter_settings.max_motif_size)
    min_repeats, min_span = int(filter_settings.min_repeats), int(filter_settings.min_span)
    raw = _encode(input_sequence)
    n = len(raw)
    if min_repeats == 1:
        return _detect_single_copy(input_sequence, raw, filter_settings, kmin, kmax, min_span, get_context(device),
                                   device, knobs)
    has_interval = hasattr(filter_settings, "interval_start_0based") or hasattr(filter_settings, "interval_end")
    ctx = get_context(device)

    if not has_interval:
        # full mode: N-trimming (prf:40-46) only moves the origin, which the masks make moot
        start, end, k = scan_arrays(raw, kmin, kmax, min_repeats, min_span, device=device, **knobs)
        offset = 0
    else:
        a = int(getattr(filter_settings, "interval_start_0based", 0))
        b = int(getattr(filter_settings, "interval_end", n))
        if a < 0 or b < 0:
            raise NotImplementedError("negative interval coordinates are not supported")
        a, b, ltrunc = _n_trim(raw, a, b)
        s = raw[a:ltrunc]                               # prf:46 (not clipped to b)
        L = len(s)
        stop = _interval_stop_position(ctx, s, b - a, kmin, kmax, knobs)
        if stop is not None and b == L and stop + 1 < L - kmin:
            raise AssertionError(f"{kmin}bp motif RepeatTracker did not reach end of the sequence")  # prf:77-78
        if stop is None:
            start, end, k = scan_arrays(s, kmin, kmax, min_repeats, min_span, device=device, **knobs)
        else:
            cut = min(L, stop + 1 + kmax)
            start, end, k = scan_arrays(s[:cut], kmin, kmax, min_repeats, min_span, device=device, **knobs)
            keep = (end.astype(np.int64) - k) <= stop   # the run's mismatch position was processed
            start, end, k = start[keep], end[keep], k[keep]
        offset = a

    out = []
    for s0, e0, k0 in zip(start.tolist(), end.tolist(), k.tolist()):
        out.append((s0 + offset, e0 + offset, _upper_slice(input_sequence, s0 + offset, k0)))
    return out
