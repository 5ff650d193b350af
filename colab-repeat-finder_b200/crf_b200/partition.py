"""Partitioning a genome over 1/2/4/8 GPUs and stitching the runs that leave a partition.

The B200-native analogue of the reference's scale-out (hail_batch_pipeline/run_hail_batch_pipeline.py:
76-77, 115-123, 153: 500 kb intervals, one CPU job each, `sort | uniq` + merge afterwards).  Here the
result is exact by construction, so no uniq/merge pass exists:

  * a record is cut into fixed-size chunks ("units"); unit = owned range [u0, u1) plus one base of
    left context and `halo` bases on the right, data range [d0, d1);
  * contiguous runs of units go to ranks, balanced by base pairs;
  * a rank scans all its units in one launch; a repeat is reported by the unit that owns its
    START (the kernel drops other starts) and followed to its end inside the unit's data;
  * only a repeat that reaches the end of its unit's data (i.e. longer than the halo) is
    "right-open"; its true end is found by asking the unit that owns the position where
    knowledge stopped (crf_run_end), hopping unit to unit if it is longer still.

M_k[j] depends on S[j] and S[j+k] only, so the match masks inside a unit are exact wherever both
bases are present; the halo only has to cover one qualifying repeat (max(min_span, min_repeats*kmax)).
"""
from collections import namedtuple

import numpy as np

Unit = namedtuple("Unit", "index record u0 u1 d0 d1 rec_len")

DEFAULT_CHUNK = 1 << 25     # 33.5 Mbp owned per unit
DEFAULT_HALO = 1 << 20      # 1 Mbp (3 % of a unit): only a perfect repeat longer than this needs the stitch exchange;
                            # the halo is never scanned for starts, it is only read when a run is followed into it


MIN_SPLIT = 1 << 20        # a share boundary closer than this to a chunk boundary moves onto it


def halo_needed(kmax, min_repeats, min_span):
    """The shortest halo that holds one qualifying repeat of the largest motif (and the base that ends it)."""
    return max(min_span, min_repeats * kmax) + kmax + 2


class Plan:
    """Records -> units (owned chunk + 1 base of left context + halo) -> contiguous shares, one per rank.

    The shares are balanced by cost: `density` = [(lo, hi, cost_per_bp), ...] over the concatenated records (global base
    pairs; default: uniform, i.e. balanced by base pairs).  A share boundary may fall anywhere, not only between chunks:
    the chunk it falls into is cut in two units there, so a measured imbalance of a few percent can be corrected
    (RankScan.rebalance) without making every unit -- and with it the share of halo that is scanned twice -- smaller."""

    def __init__(self, lengths, n_ranks, chunk=DEFAULT_CHUNK, halo=DEFAULT_HALO, kmax=50, min_repeats=3, min_span=9,
                 density=None):
        need = halo_needed(kmax, min_repeats, min_span)
        if halo < need:
            raise ValueError(f"halo {halo} is shorter than one qualifying repeat of the largest motif ({need})")
        if chunk < 1:
            raise ValueError("chunk must be positive")
        self.lengths = [int(x) for x in lengths]
        self.n_ranks = n_ranks
        self.chunk, self.halo = chunk, halo
        rec_base = np.concatenate([[0], np.cumsum(np.asarray(self.lengths, dtype=np.int64))])
        total = int(rec_base[-1])
        self.total = total
        # where the shares end, in global base pairs
        cuts = self._cuts(total, n_ranks, density)
        self.cuts = cuts
        min_split = min(MIN_SPLIT, max(1, chunk // 8))
        units, bounds, ci = [], [0], 1
        for r, length in enumerate(self.lengths):
            if length == 0:
                continue
            g0 = int(rec_base[r])
            edges = set(range(0, length, chunk)) | {length}
            for c in cuts[1:-1]:                        # share boundaries inside this record
                pos = c - g0
                if 0 < pos < length:
                    near = min(edges, key=lambda e: abs(e - pos))
                    if abs(near - pos) >= min_split:
                        edges.add(pos)
            edges = sorted(edges)
            for u0, u1 in zip(edges[:-1], edges[1:]):
                units.append(Unit(len(units), r, u0, u1, max(0, u0 - 1), min(length, u1 + halo), length))
        self.units = units
        # share i = the units whose owned range starts before cut i (and at or after cut i - 1)
        starts = np.array([int(rec_base[u.record]) + u.u0 for u in units], dtype=np.int64)
        ends = np.array([int(rec_base[u.record]) + u.u1 for u in units], dtype=np.int64)
        mids = (starts + ends) // 2
        for i in range(1, n_ranks):
            j = int(np.searchsorted(mids, cuts[i], side="left"))
            bounds.append(min(max(j, bounds[-1]), len(units)))
        bounds.append(len(units))
        self.bounds = bounds
        self._rec_units = {}
        for u in units:
            self._rec_units.setdefault(u.record, ([], []))
            self._rec_units[u.record][0].append(u.u0)
            self._rec_units[u.record][1].append(u.index)
        del ci

    @staticmethod
    def _cuts(total, n_ranks, density):
        if not density:
            return [total * i // n_ranks for i in range(n_ranks + 1)]
        segs = sorted((int(lo), int(hi), float(c)) for lo, hi, c in density if hi > lo)
        # fill gaps / clip so that the segments tile [0, total)
        tiled, pos = [], 0
        mean = sum((hi - lo) * c for lo, hi, c in segs) / max(1, sum(hi - lo for lo, hi, c in segs))
        for lo, hi, c in segs:
            lo, hi = max(lo, pos), min(hi, total)
            if lo > pos:
                tiled.append((pos, lo, mean))
            if hi > lo:
                tiled.append((lo, hi, max(c, 1e-12)))
                pos = hi
        if pos < total:
            tiled.append((pos, total, mean))
        whole = sum((hi - lo) * c for lo, hi, c in tiled)
        cuts, acc, k = [0], 0.0, 1
        for lo, hi, c in tiled:
            w = (hi - lo) * c
            while k < n_ranks and acc + w >= whole * k / n_ranks:
                cuts.append(int(lo + (whole * k / n_ranks - acc) / c))
                k += 1
            acc += w
        while len(cuts) < n_ranks:
            cuts.append(total)
        cuts.append(total)
        return cuts

    def units_of(self, rank):
        return self.units[self.bounds[rank]:self.bounds[rank + 1]]

    def rank_of_unit(self, index):
        return int(np.searchsorted(np.array(self.bounds[1:]), index, side="right"))

    def unit_owning(self, record, pos):
        import bisect
        u0s, idx = self._rec_units[record]
        return self.units[idx[bisect.bisect_right(u0s, pos) - 1]]

    def share_range(self, rank):
        """[lo, hi) in global base pairs (records concatenated) of the bases `rank` owns."""
        us = self.units_of(rank)
        if not us:
            return 0, 0
        rec_base = np.concatenate([[0], np.cumsum(np.asarray(self.lengths, dtype=np.int64))])
        return int(rec_base[us[0].record]) + us[0].u0, int(rec_base[us[-1].record]) + us[-1].u1

    def load_args(self, rank, record_starts):
        """(starts, lengths, own_lo, own_hi) for Context.load_ranges; record_starts[r] = offset of
        record r inside the caller's base buffer."""
        mine = self.units_of(rank)
        starts = np.array([int(record_starts[u.record]) + u.d0 for u in mine], dtype=np.uint64)
        lens = np.array([u.d1 - u.d0 for u in mine], dtype=np.uint64)
        own_lo = np.array([u.u0 - u.d0 for u in mine], dtype=np.uint64)
        own_hi = np.array([u.u1 - u.d0 for u in mine], dtype=np.uint64)
        return starts, lens, own_lo, own_hi


def load_positions(plan, share, kmax):
    """Layout positions the load of `share` takes (crf_load_limit: every unit's data plus a gap of kmax)."""
    return sum(u.d1 - u.d0 + kmax for u in plan.units_of(share))


def plan_loads(lengths, world, phases, limit, density=None, **plan_args):
    """The Plan of phases x world shares with the fewest phases (at least `phases`) whose every share fits one load of
    `limit` layout positions -- a record longer than one load ends up spread over several loads of the same rank.
    Returns (plan, phases).  A single unit above the limit (a chunk as long as a load) stays as it is: its load refuses it."""
    kmax = plan_args.get("kmax", 50)
    while True:
        plan = Plan(lengths, phases * world, density=density, **plan_args)
        worst = max(load_positions(plan, v, kmax) for v in range(phases * world))
        if worst <= limit or max(u.d1 - u.d0 + kmax for u in plan.units) > limit:
            return plan, phases
        phases = max(phases + 1, -(-phases * worst // limit))


def localize(plan, rank, unit_local, start, end, k):
    """Per-unit results of one rank -> record coordinates + the right-open subset.

    Returns (record, start, end, k, open_mask): open_mask marks runs that reached the end of their
    unit's data although the record continues (their `end` is a lower bound)."""
    mine = plan.units_of(rank)
    if len(mine) == 0:
        z = np.zeros(0, dtype=np.int64)
        return z, z, z, z, np.zeros(0, dtype=bool)
    d0 = np.array([u.d0 for u in mine], dtype=np.int64)
    d1 = np.array([u.d1 for u in mine], dtype=np.int64)
    rec = np.array([u.record for u in mine], dtype=np.int64)
    rlen = np.array([u.rec_len for u in mine], dtype=np.int64)
    ul = np.asarray(unit_local, dtype=np.int64)
    g_start = np.asarray(start, dtype=np.int64) + d0[ul]
    g_end = np.asarray(end, dtype=np.int64) + d0[ul]
    open_mask = (g_end == d1[ul]) & (d1[ul] < rlen[ul])
    return rec[ul], g_start, g_end, np.asarray(k, dtype=np.int64), open_mask


def stitch(plan, open_runs, run_end_fn, exchange_fn=None, rank=0, owner=None):
    """Finish right-open runs.

    owner: maps the plan's share number (plan.rank_of_unit) to the rank that holds it (default: identity; a phased
    multi-GPU job has phases x N shares, share v on rank v % N).

    open_runs : list of (record, start, end_lower_bound, k) -- the same list on every rank.
    run_end_fn(unit, local_pos, k) -> local run end, callable for units of *this* rank only.
    exchange_fn(dict) -> merged dict over ranks (None on a single rank).
    Returns the list of (record, start, end, k) with true ends, in input order."""
    pending = {i: (rec, end - k, k) for i, (rec, _s, end, k) in enumerate(open_runs)}   # position p: M_k[p] unknown
    final_i0 = {}
    while pending:
        answers = {}
        for i, (rec, p, k) in pending.items():
            unit = plan.unit_owning(rec, p)
            holder = plan.rank_of_unit(unit.index)
            if (owner(holder) if owner else holder) == rank:
                answers[i] = int(run_end_fn(unit, p - unit.d0, k)) + unit.d0
        if exchange_fn is not None:
            answers = exchange_fn(answers)
        nxt = {}
        for i, (rec, p, k) in pending.items():
            e = answers[i]
            unit = plan.unit_owning(rec, p)
            if e + k == unit.d1 and unit.d1 < unit.rec_len and e > p:
                nxt[i] = (rec, e, k)       # still inside a run at the end of this unit's data: hop on
            else:
                final_i0[i] = e
        pending = nxt
    return [(rec, s, final_i0[i] + k, k) for i, (rec, s, _e, k) in enumerate(open_runs)]


def stitch_collective(plan, open_mine, run_end_fn, rank, world, dist, device):
    """stitch() for world > 1 with tensor collectives (a count all-gather, a row all-gather sized by the largest count, one
    all-reduce per hop) instead of pickled objects.  open_mine: this rank's (record, start, end_lower_bound, k) rows --
    any number of them.  Returns the stitched rows of ALL ranks, identical on every rank."""
    import torch
    counts = torch.empty(world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(counts, torch.tensor([len(open_mine)], dtype=torch.int64, device=device))
    slots = max(int(counts.max().item()), 1)
    mine = torch.full((slots + 1, 4), -1, dtype=torch.int64)
    mine[0, 0] = len(open_mine)
    if open_mine:
        mine[1:1 + len(open_mine)] = torch.tensor(open_mine, dtype=torch.int64)
    mine = mine.to(device)
    allrows = torch.empty((world * mine.shape[0], 4), dtype=torch.int64, device=device)   # concatenated along dim 0
    dist.all_gather_into_tensor(allrows, mine)
    allrows = allrows.cpu().numpy().reshape(world, mine.shape[0], 4)
    open_all = [tuple(int(x) for x in allrows[r, 1 + i]) for r in range(world) for i in range(int(allrows[r, 0, 0]))]

    def exchange(answers):
        t = torch.full((max(len(open_all), 1),), -1, dtype=torch.int64)
        for i, v in answers.items():
            t[i] = v
        t = t.to(device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.cpu().tolist()
        return {i: v for i, v in enumerate(t) if v >= 0}

    return stitch(plan, open_all, run_end_fn, exchange, rank)


def scan_partitioned(ctx, bases, record_starts, lengths, kmin, kmax, min_repeats, min_span, rank=0, world=1,
                     chunk=DEFAULT_CHUNK, halo=DEFAULT_HALO, on_device=False, dist=None, tensor_device=None, **knobs):
    """Scan `lengths` records split over `world` ranks; every rank returns the full, stitched,
    (record, start, end)-sorted result as numpy arrays (record, start, end, k).

    dist: torch.distributed (initialised) when world > 1; results travel with all_gather_object
    (bench.py uses a device-side gather instead).  tensor_device: stitch with fixed-size tensor collectives
    on that device (stitch_collective) instead of pickled objects."""
    plan = Plan(lengths, world, chunk, halo, kmax, min_repeats, min_span)
    starts, lens, own_lo, own_hi = plan.load_args(rank, record_starts)
    mine = plan.units_of(rank)
    if len(mine):
        seq = ctx.load_ranges(bases, starts, lens, own_lo, own_hi, max_motif_cap=kmax, on_device=on_device)
        n = seq.scan(kmin, kmax, min_repeats, min_span, **knobs)
        ul, st, en, kk = seq.fetch(n)
    else:
        seq = None
        ul = st = en = kk = np.zeros(0, dtype=np.uint32)
    rec, g_st, g_en, g_k, open_mask = localize(plan, rank, ul, st, en, kk)
    open_mine = [(int(a), int(b), int(c), int(d)) for a, b, c, d in
                 zip(rec[open_mask], g_st[open_mask], g_en[open_mask], g_k[open_mask])]
    closed = np.stack([rec[~open_mask], g_st[~open_mask], g_en[~open_mask], g_k[~open_mask]]) if len(rec) else \
        np.zeros((4, 0), dtype=np.int64)

    def gather_obj(obj):
        if world == 1:
            return [obj]
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    open_all = [x for part in gather_obj(open_mine) for x in part]

    def run_end_fn(unit, local_pos, k):
        return seq.run_end(unit.index - plan.bounds[rank], local_pos, k)

    def exchange(answers):
        merged = {}
        for part in gather_obj(answers):
            merged.update(part)
        return merged

    if world > 1 and tensor_device is not None:
        stitched = stitch_collective(plan, open_mine, run_end_fn, rank, world, dist, tensor_device)
    else:
        stitched = stitch(plan, open_all, run_end_fn, exchange if world > 1 else None, rank)
    parts = gather_obj(closed)
    rows = np.concatenate(parts, axis=1) if parts else closed
    if stitched:
        rows = np.concatenate([rows, np.array(stitched, dtype=np.int64).T], axis=1)
        order = np.lexsort((rows[2], rows[1], rows[0]))
        rows = rows[:, order]
    if seq is not None:
        seq.close()
    return rows[0], rows[1], rows[2], rows[3]
