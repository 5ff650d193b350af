"""detect_repeats_intervals(): interval mode for many intervals of one sequence, one device load per group of intervals.

Interval i gives exactly what api.detect_repeats(S, fs + {interval_start_0based: a_i, interval_end: b_i}) gives: the same
rows, or the same exception.  Instead of a probe load + probe scan + second load per interval, every interval's sequence
prefix goes into one ranged load of the packed source, crf_interval_stop decides where the reference's loop breaks for
all of them at once, and one scan of the same load gives the rows (DESIGN.md section 6, "Many intervals").
"""
import copy
import time

import numpy as np

from . import _cabi, api

#: t examined past the interval end by the first round (the probe window of api._interval_stop_position); each further
#: round for the intervals the loaded prefix could not decide multiplies it by 4
FIRST_WINDOW = 256

#: what the last scan_intervals() call did: rounds, loads, seconds spent in load / stop / scan / fetch (host clock around
#: calls that each end in a stream sync), and the intervals left to the single-interval path (CLI and API)
last_stats = {}


def n_runs(planes):
    """Maximal runs [start, end) of N / n in the planes' position space: the mask runs with the exotic symbols (IUPAC
    letters and the like, which the mask covers too but api._n_trim does not skip) cut out.  int64 arrays."""
    runs = planes.runs if planes.runs is not None else _cabi.mask_runs(planes.NM_ptr, planes.n_bases)
    runs = runs.astype(np.int64).reshape(-1, 2)
    ex = (planes.exotic >> np.uint64(8)).astype(np.int64)
    # every exotic position lies inside a mask run and splits it: pairing the sorted starts with the sorted ends
    starts = np.sort(np.concatenate([runs[:, 0], ex + 1]))
    ends = np.sort(np.concatenate([ex, runs[:, 1]]))
    keep = ends > starts
    return starts[keep], ends[keep]


def n_trim(nstarts, nends, base, a, b, n):
    """api._n_trim (prf:40-44) for many intervals 0 <= a < b <= n of records of n bases at source position base, given
    the N runs of the source: a moves forward over N / n up to b, b moves back over N / n down to the new a, and Ltrunc
    shrinks with b.  Returns (a', b', Ltrunc), int64 arrays."""
    base, a, b, n = (np.asarray(x, dtype=np.int64) for x in (base, a, b, n))
    ga, gb = base + a, base + b
    if nstarts.size == 0:
        return a.copy(), b.copy(), n.copy()
    last = nstarts.size - 1
    i = np.searchsorted(nends, ga, side="right")                 # first run that ends after ga ...
    ic = np.minimum(i, last)
    a2 = np.where((i <= last) & (nstarts[ic] <= ga), np.minimum(nends[ic], gb), ga)    # ... holds it: skip to its end
    j = np.searchsorted(nends, gb - 1, side="right")             # the run holding gb - 1, if any
    jc = np.minimum(j, last)
    b2 = np.where((j <= last) & (nstarts[jc] <= gb - 1), np.maximum(nstarts[jc], a2), gb)
    return a2 - base, b2 - base, n - (gb - b2)


def _groups(need, limit):
    """Consecutive groups of items whose `need` sums stay within `limit` (each need <= limit): [(first, last)), ...]."""
    csum = np.cumsum(need)
    out, first = [], 0
    while first < need.size:
        before = int(csum[first - 1]) if first else 0
        last = int(np.searchsorted(csum, before + limit, side="right"))
        out.append((first, last))
        first = last
    return out


def scan_intervals(ctx, planes, src, full_len, end_pos, kmin, kmax, min_repeats, min_span, knobs=None, load_limit=None):
    """The batched half of interval mode (min_repeats >= 2).  Interval i's sequence is s_i = planes[src_i : src_i +
    full_len_i] (already N-trimmed), its interval ends at end_pos_i.  Loads the prefixes s_i[0 : min(L_i, E_i + 1 + window
    + kmax)], asks crf_interval_stop where each loop breaks, scans the same load and keeps the rows whose mismatch position
    was processed (end - k <= T); intervals the prefix could not decide go round again with 4x the window.
    Returns (stop, iv, start, end, k, too_long): stop per interval (a position or STOP_TO_END), the rows as flat int64
    columns (iv = interval index; start / end relative to s_i; sorted by (iv, start, end)), and the mask of intervals whose
    prefix alone outgrew one load (not done here)."""
    knobs = knobs or {}
    src, full_len, end_pos = (np.asarray(x, dtype=np.int64) for x in (src, full_len, end_pos))
    n = src.size
    limit = _cabi.load_limit(kmax) if load_limit is None else load_limit
    stop = np.full(n, _cabi.STOP_TO_END, dtype=np.int64)
    too_long = np.zeros(n, dtype=bool)
    parts = []
    stats = {"rounds": 0, "loads": 0, "load_s": 0.0, "stop_s": 0.0, "scan_s": 0.0, "fetch_s": 0.0}
    todo = np.flatnonzero(full_len > 0)                  # (an empty s_i has no rows)
    window = FIRST_WINDOW + kmax
    while todo.size:
        stats["rounds"] += 1
        P = np.minimum(full_len[todo], end_pos[todo] + 1 + window + kmax)
        big = P + kmax > limit
        too_long[todo[big]] = True
        todo, P = todo[~big], P[~big]
        undecided = []
        for first, last in _groups(P + kmax, limit):
            idx, plen = todo[first:last], P[first:last]
            t0 = time.perf_counter()
            with ctx.load_packed(planes, max_motif_cap=kmax, ranges=(src[idx], plen, None, None)) as seq:
                t1 = time.perf_counter()
                st = seq.interval_stop(kmin, kmax, end_pos[idx], full_len[idx])
                t2 = time.perf_counter()
                nrow = seq.scan(kmin, kmax, min_repeats, min_span, **knobs)
                t3 = time.perf_counter()
                rec, s0, e0, kk = (np.asarray(c).astype(np.int64) for c in seq.fetch(nrow))
                t4 = time.perf_counter()
            stats["loads"] += 1
            for key, dt in (("load_s", t1 - t0), ("stop_s", t2 - t1), ("scan_s", t3 - t2), ("fetch_s", t4 - t3)):
                stats[key] += dt
            done = st != _cabi.STOP_UNDECIDED
            stop[idx[done]] = st[done]
            undecided.append(idx[~done])
            t_row = st[rec]
            keep = (t_row == _cabi.STOP_TO_END) | ((t_row >= 0) & (e0 - kk <= t_row))
            parts.append((idx[rec[keep]], s0[keep], e0[keep], kk[keep]))
        todo = np.concatenate(undecided) if undecided else np.zeros(0, np.int64)
        window *= 4
    cols = [np.concatenate([p[j] for p in parts]) if parts else np.zeros(0, np.int64) for j in range(4)]
    order = np.argsort(cols[0], kind="stable")          # groups are in interval order, rows of an interval in (start, end)
    last_stats.clear()
    last_stats.update(stats, intervals=int(n), too_long=int(too_long.sum()))
    return (stop, *(c[order] for c in cols), too_long)


def _settings_for(filter_settings, a, b):
    fs = copy.copy(filter_settings)
    fs.interval_start_0based, fs.interval_end = a, b
    return fs


def run_intervals(planes, base, n, a, b, filter_settings, device=None, knobs=None, single=None, load_limit=None):
    """Interval mode for intervals [a_i, b_i) of records of n_i bases that start at source position base_i of `planes`.
    single(i) runs interval i through api.detect_repeats and returns its rows as (start, end, motif) tuples; it is used
    for min_repeats == 1, more motif sizes than crf_interval_stop takes, a >= b, negative coordinates, b > n, and intervals
    whose prefix alone outgrows one load.
    Returns (outcome, a', iv, start, end, k): outcome[i] = None (rows in the columns; start / end relative to a'_i),
    a list of tuples (from single), or the exception interval i raises."""
    kmin, kmax = int(filter_settings.min_motif_size), int(filter_settings.max_motif_size)
    min_repeats, min_span = int(filter_settings.min_repeats), int(filter_settings.min_span)
    a, b = (np.asarray(x, dtype=np.int64).reshape(-1) for x in (a, b))
    base, n = (np.broadcast_to(np.asarray(x, dtype=np.int64), a.shape) for x in (base, n))
    m = a.size
    outcome = [None] * m
    batched = (a >= 0) & (b >= 0) & (a < b) & (b <= n)
    if min_repeats == 1 or kmax - kmin + 1 > _cabi.STOP_MAX_MOTIF_SIZES:
        batched[:] = False
    bi = np.flatnonzero(batched)
    a2, b2, lt = n_trim(*n_runs(planes), base[bi], a[bi], b[bi], n[bi]) if bi.size else (np.zeros(0, np.int64),) * 3
    L, E = lt - a2, b2 - a2
    stop, iv, start, end, k, too_long = scan_intervals(api.get_context(device), planes, base[bi] + a2, L, E, kmin, kmax,
                                                       min_repeats, min_span, knobs, load_limit)
    iv = bi[iv]
    bad = (stop >= 0) & (b2 == L) & (stop + 1 < L - kmin)                  # prf:77-78, as api.detect_repeats
    for i in bi[bad].tolist():
        outcome[i] = AssertionError(f"{kmin}bp motif RepeatTracker did not reach end of the sequence")
    origin = np.zeros(m, dtype=np.int64)
    origin[bi] = a2
    fallback = np.flatnonzero(~batched).tolist() + bi[too_long].tolist()
    last_stats["fallback"] = len(fallback)
    first_raise = min([i for i, o in enumerate(outcome) if o is not None], default=m)
    for i in sorted(fallback):
        if i > first_raise:                                                 # an earlier interval raises already
            break
        try:
            outcome[i] = single(i)
        except Exception as exc:                                            # noqa: BLE001 (re-raised by the caller)
            outcome[i] = exc
            first_raise = min(first_raise, i)
    keep = ~np.isin(iv, bi[too_long | bad])
    return outcome, origin, iv[keep], start[keep], end[keep], k[keep]


def detect_repeats_intervals(input_sequence, intervals, filter_settings, device=None, **knobs):
    """Interval mode for many intervals of one sequence: [detect_repeats(input_sequence, filter_settings + {
    interval_start_0based: a, interval_end: b}) for (a, b) in intervals], computed with one device load per group of
    intervals.  If an interval raises, raises what the first such interval (in input order) raises."""
    api.validate_filter_settings(filter_settings)
    raw = api._encode(input_sequence)
    ab = np.asarray([(int(x), int(y)) for x, y in intervals], dtype=np.int64).reshape(-1, 2)
    if not ab.shape[0]:
        return []
    planes = _cabi.pack_ascii(raw).with_runs()

    def single(i):
        return api.detect_repeats(input_sequence, _settings_for(filter_settings, int(ab[i, 0]), int(ab[i, 1])),
                                  device=device, **knobs)

    outcome, origin, iv, start, end, k = run_intervals(planes, 0, len(raw), ab[:, 0], ab[:, 1], filter_settings, device,
                                                       knobs, single)
    for o in outcome:
        if isinstance(o, BaseException):
            raise o
    bounds = np.searchsorted(iv, np.arange(len(outcome) + 1))
    out = []
    for i, o in enumerate(outcome):
        if o is not None:
            out.append(o)
            continue
        lo, hi, a0 = int(bounds[i]), int(bounds[i + 1]), int(origin[i])
        out.append([(s0 + a0, e0 + a0, api._upper_slice(input_sequence, s0 + a0, k0))
                    for s0, e0, k0 in zip(start[lo:hi].tolist(), end[lo:hi].tolist(), k[lo:hi].tolist())])
    return out
