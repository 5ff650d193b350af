"""Multi-GPU scan: every rank scans its share of the (record, chunk) units and the GPUs concatenate their sorted
rows on rank 0 over NVLink peer memory (crf_xchg, csrc/crf_xchg.cuh) -- no host round trip inside a step.

The B200-native counterpart of the reference's scale-out (hail_batch_pipeline/run_hail_batch_pipeline.py:76-77,
96-123, 153: one CPU job per 500 kb interval, BED files concatenated, `sort | uniq`).  Two ways to run N ranks:

  * one process per GPU (torchrun): `DistComm(torch.distributed)`; exchange blocks are shared through CUDA IPC;
  * one process, one thread per GPU (the CLI's --devices): `ThreadComm`; plain peer access.

Either way the step is `RankScan.step_async()` on every rank (kernel launches only) and `RankScan.finish()` (one
stream synchronisation; the rare cases -- a buffer outgrown, a repeat longer than the halo -- are settled there).
"""
import threading

import numpy as np

from . import _cabi, partition


class DistComm:
    """Ranks are processes of a torch.distributed group (any backend).  Used at set-up (IPC handles) and for the
    rare stitch of runs longer than the halo; never inside a step."""
    same_process = False

    def __init__(self, dist, rank, world):
        self.dist, self.rank, self.world = dist, rank, world

    def allgather_obj(self, obj):
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out


class ThreadComm:
    """Ranks are threads of this process, one per device (ThreadComm.split(world) gives one endpoint per rank)."""
    same_process = True

    class _Shared:
        def __init__(self, world):
            self.world = world
            self.barrier = threading.Barrier(world)
            self.slots = [None] * world

    def __init__(self, shared, rank):
        self._s, self.rank, self.world = shared, rank, shared.world

    @classmethod
    def split(cls, world):
        shared = cls._Shared(world)
        return [cls(shared, r) for r in range(world)]

    def allgather_obj(self, obj):
        s = self._s
        s.slots[self.rank] = obj
        s.barrier.wait()
        out = list(s.slots)
        s.barrier.wait()
        return out


def default_row_cap(total_bp):
    """Rows rank 0's buffer holds: 1 per 32 bp of the whole job (a human genome has ~2 per kbp), 16 bytes each."""
    return int(min(0xFFFFFFF0, max(1 << 20, total_bp // 32)))


def global_rows(rows_of_rank, rank, local_rows):
    """Row numbers inside rank 0's buffer of `rank`'s local result rows (rank order = genome order)."""
    offsets = np.concatenate([[0], np.cumsum(np.asarray(rows_of_rank, dtype=np.int64))])
    return np.asarray(local_rows, dtype=np.int64) + int(offsets[rank])


def unit_rows_to_records(units, unit, start, end, k):
    """Unit-relative rows (unit index, start, end, k) -> (record uint32, start uint64, end uint64, k): each unit's
    origin d0 is added in 64 bits (partition.localize does the same arithmetic in int64)."""
    rec = np.array([u.record for u in units], dtype=np.uint32)
    d0 = np.array([u.d0 for u in units], dtype=np.uint64)
    unit = np.asarray(unit, dtype=np.int64)
    return rec[unit], np.asarray(start).astype(np.uint64) + d0[unit], np.asarray(end).astype(np.uint64) + d0[unit], k


class RankScan:
    """One rank (one GPU) of a partitioned scan.

    bases / record_starts / lengths describe ALL records (every rank sees the same description; `bases` is this
    rank's view of the bytes: a host array, _cabi.PackedPlanes or, with on_device, a device pointer).  reads=True
    splits the records by count instead of cutting them into chunks (config C5: many short independent sequences).

    phases > 1: the genome-ordered unit list is cut into phases x N contiguous shares and rank r takes share p * N + r in
    phase p -- one sequence per phase.  A step scans the phases one after the other while the rows of the phase before
    travel to rank 0 on the exchange's own stream: the gather, which is bound by rank 0's NVLink ingress, hides behind
    the next phase's scan.  Genome order = phase-major, rank-minor, so rank 0's buffer still holds the sorted result.
    The phase count is raised above `phases` when a share would not fit one load (crf_load_limit): that is how a record
    longer than one load is scanned, on one GPU (N = 1: several loads, scanned one after the other) or on several.

    Records longer than one load ("long" mode): every unit is reported as a record of its own (output map: out_record =
    global unit index, no shift), so the rows stay unit-relative and 32-bit on the device; fetch() adds each unit's
    origin on the host in 64 bits (start / end come back as uint64), fetch_units() hands the unit-relative rows out."""

    def __init__(self, ctx, comm, bases, record_starts, lengths, kmin, kmax, min_repeats, min_span, on_device=False,
                 chunk=partition.DEFAULT_CHUNK, halo=partition.DEFAULT_HALO, reads=False, row_cap=None, knobs=None,
                 timeout_s=None, base_offset=0, phases=1):
        self.ctx, self.comm = ctx, comm
        self.rank, self.world = comm.rank, comm.world
        self.filters = (int(kmin), int(kmax), int(min_repeats), int(min_span))
        self.knobs = dict(knobs or {})
        lengths = [int(x) for x in lengths]
        self.total_bp = int(sum(lengths))
        self.reads = reads
        self.limit = _cabi.load_limit(kmax)
        self.long = not reads and any(n + kmax > self.limit for n in lengths)
        if self.long:                                  # any filter a single load accepts works with units of a long record
            halo = max(halo, partition.halo_needed(kmax, min_repeats, min_span))
        self.phases = max(1, int(phases))
        self._lengths, self._record_starts = lengths, record_starts
        self._plan_args = dict(chunk=chunk, halo=halo, kmax=kmax, min_repeats=min_repeats, min_span=min_span)
        self._source = (bases, on_device, base_offset)
        self.seqs = [None] * self.phases
        self._make_shares(None)
        self.reload(bases, on_device=on_device, base_offset=base_offset)
        self.xchg = None
        if self.world > 1:
            self.xchg = _cabi.Xchg(ctx, self.rank, self.world, row_cap or default_row_cap(self.total_bp))
            if timeout_s:
                self.xchg.set_timeout(timeout_s)
            n_out = len(self.plan.units) if self.long else len(lengths)     # record numbers the rows carry
            if n_out < 65536 and kmax < 65536:         # 12-byte rows over NVLink (record and motif size share a word)
                self.xchg.set_compact(True)
            if comm.same_process:
                peers = comm.allgather_obj(self.xchg)
                for r, other in enumerate(peers):
                    if r != self.rank:
                        self.xchg.connect_local(r, other)
                comm.allgather_obj(None)               # every rank is connected before anyone pushes
            else:
                handles = comm.allgather_obj(self.xchg.export())
                for r, h in enumerate(handles):
                    if r != self.rank:
                        self.xchg.connect_ipc(r, h)
                comm.allgather_obj(None)
        self.last = None
        self.steps_repeated = 0

    def _make_shares(self, density):
        """Units and load arguments of this rank (all phases) for a cost density over the genome (None: by base pairs)."""
        lengths, record_starts, reads = self._lengths, self._record_starts, self.reads
        P = self.phases
        shares = P * self.world                       # "virtual ranks": share v = phase v // N of rank v % N
        self.load_args, self.units = [], []
        if reads:
            n_rec = len(lengths)
            self.plan = None
            self.first_record = []
            for p in range(P):
                v = p * self.world + self.rank
                lo, hi = n_rec * v // shares, n_rec * (v + 1) // shares
                self.first_record.append(lo)
                self.load_args.append((np.asarray(record_starts[lo:hi], dtype=np.uint64),
                                       np.asarray(lengths[lo:hi], dtype=np.uint64), None, None))
                self.units.append([])
            self.my_bp = int(sum(int(a[1].sum()) for a in self.load_args))
            self.n_units = n_rec
        else:
            whole = self.world == 1 and self._plan_args["chunk"] >= max(lengths + [1])
            self.plan, P = partition.plan_loads(lengths, self.world, P, self.limit, density=density, **self._plan_args)
            if P != self.phases:
                self.phases = P
                self.seqs = [None] * P
            for p in range(P):
                v = p * self.world + self.rank
                starts, lens, own_lo, own_hi = self.plan.load_args(v, record_starts)
                if whole:
                    own_lo = own_hi = None
                self.load_args.append((starts, lens, own_lo, own_hi))
                self.units.append(self.plan.units_of(v))
            self.my_bp = int(sum(u.u1 - u.u0 for us in self.units for u in us))
            self.n_units = len(self.plan.units)

    def rebalance(self, min_gain=0.02):
        """Re-cut the shares by MEASURED cost: every rank reports the scan time of its last step and its range of the genome;
        the new share boundaries equalise the time (cost per base pair taken as constant inside each old share) and this
        rank's sequences are loaded again.  All ranks must call it together; returns the expected relative gain (0.0 when
        the shares were left alone because less than `min_gain` was to be had)."""
        if self.world == 1 or self.reads or self.phases != 1 or self.plan is None:
            return 0.0
        t = float(self.stats().get("scan_ms", 0.0))
        lo, hi = self.plan.share_range(self.rank)
        info = self.comm.allgather_obj((t, lo, hi))
        times = [x[0] for x in info]
        if min(times) <= 0 or any(x[2] <= x[1] for x in info):
            return 0.0
        gain = 1.0 - (sum(times) / len(times)) / max(times)
        if gain < min_gain:
            return 0.0
        density = [(l, h, tt / (h - l)) for tt, l, h in info]
        self._make_shares(density)
        bases, on_device, base_offset = self._source
        self.reload(bases, on_device=on_device, base_offset=base_offset)
        return gain

    @property
    def seq(self):
        """The sequence of the first phase (single-phase callers)."""
        return self.seqs[0]

    def span(self):
        """[lo, hi) of the caller's base buffer this rank reads (its units plus their halos, all phases)."""
        lo, hi = None, 0
        for starts, lens, _, _ in self.load_args:
            if len(starts):
                a, b = int(starts.min()), int((starts + lens).max())
                lo = a if lo is None else min(lo, a)
                hi = max(hi, b)
        return (0, 0) if lo is None else (lo, hi)

    def reload(self, bases, on_device=False, base_offset=0):
        """(Re-)upload this rank's share.  `bases` starts at position `base_offset` of the buffer the record_starts refer
        to (a rank that keeps only its own span() on the host passes span()[0])."""
        kmax = self.filters[1]
        for p, (starts, lens, own_lo, own_hi) in enumerate(self.load_args):
            if self.seqs[p] is not None:
                self.seqs[p].close()
                self.seqs[p] = None
            if len(starts):
                if base_offset:                                      # (a reads share has millions of starts: no copy without need)
                    starts = starts - np.uint64(base_offset)
                if isinstance(bases, _cabi.PackedPlanes):          # planes packed on the host: 0.375 B/bp over PCIe
                    if base_offset % 32:
                        raise ValueError("packed planes must start at a multiple of 32 positions")
                    seq = self.ctx.load_packed(bases, max_motif_cap=kmax,
                                               ranges=(starts, lens, own_lo, own_hi))
                else:
                    seq = self.ctx.load_ranges(bases, starts, lens, own_lo, own_hi,
                                               max_motif_cap=kmax, on_device=on_device)
                if self.reads:
                    if self.world > 1:
                        seq.set_output_map(out_record=np.arange(self.first_record[p], self.first_record[p] + len(starts),
                                                                dtype=np.uint32))
                elif self.long:
                    us = self.units[p]
                    seq.set_output_map(out_record=[u.index for u in us],
                                       open_ended=[int(u.d1 < u.rec_len) for u in us])
                elif self.world > 1 or own_lo is not None:
                    us = self.units[p]
                    seq.set_output_map(out_record=[u.record for u in us], out_shift=[u.d0 for u in us],
                                       open_ended=[int(u.d1 < u.rec_len) for u in us])
            elif self.world > 1:
                # a share without units still takes part in the exchange: it pushes zero rows (an empty record to scan)
                seq = self.ctx.load_ranges(np.zeros(0, np.uint8), np.zeros(1, np.uint64), np.zeros(1, np.uint64),
                                           max_motif_cap=kmax)
            else:
                seq = None
            self.seqs[p] = seq

    # ---- the step -------------------------------------------------------------------------------------------
    def step_async(self):
        """Queue one whole step on this rank's streams (per phase: scan, assembly, push to rank 0); returns at once."""
        kmin, kmax, mr, ms = self.filters
        if self.world == 1:
            self._n = [0 if seq is None else seq.scan(kmin, kmax, mr, ms, **self.knobs) for seq in self.seqs]
        else:
            for p, seq in enumerate(self.seqs):
                seq.scan_gather(self.xchg, kmin, kmax, mr, ms, append=p > 0, **self.knobs)

    def finish(self):
        """Wait for the queued steps; settle the rare cases.  Returns the whole-job row count (the rows are on rank 0)."""
        self.steps_repeated = 0
        if self.world == 1:
            self.last = None
            if self.plan is not None and self.load_args[0][2] is not None and \
                    any(seq is not None and seq.stats().n_open for seq in self.seqs):
                self._stitch_local()
            return sum(self._n)
        kmin, kmax, mr, ms = self.filters
        res = self.xchg.wait()
        if res.worst_status == _cabi.XCHG_VOID_STEP:
            # some rank outgrew a buffer (first step of a new workload, usually): every rank repeats the job the slow
            # way -- crf_scan sizes everything -- and pushes again; the status is the same on all ranks, so all agree
            for p, seq in enumerate(self.seqs):
                seq.scan(kmin, kmax, mr, ms, **self.knobs)
                seq.push(self.xchg, append=p > 0)
            res = self.xchg.wait()
            self.steps_repeated = 1
        if res.worst_status == _cabi.XCHG_ROOT_FULL:
            raise _cabi.CrfError(f"{res.total_rows} rows do not fit rank 0's gather buffer ({self.xchg.row_cap} rows): "
                                 f"pass a larger row_cap")
        if res.worst_status != _cabi.XCHG_OK:
            raise _cabi.CrfError(f"multi-GPU gather failed with status {res.worst_status}")
        self.last = res
        # the last job's phases: steps res.step - P + 1 .. res.step
        self.phase_results = [res if p == self.phases - 1 else self.xchg.step_result(res.step - (self.phases - 1 - p))
                              for p in range(self.phases)]
        if self.plan is not None and any(r.any_open for r in self.phase_results):
            self._stitch()
        return int(res.total_rows)

    def _stitch(self):
        """A repeat longer than the halo reached the end of its unit's data: follow it on whoever holds the next bases
        (crf_run_end), hop by hop, then patch the ends inside rank 0's buffer.  Rare; host-driven."""
        N = self.world
        mine = []                                      # (phase, local row, record, start, end, k)
        for p, seq in enumerate(self.seqs):
            n_open = int(seq.stats().n_open)
            if n_open:
                mine += [(p,) + tuple(int(x) for x in row) for row in seq.fetch_open(cap=n_open)]
        per_rank = self.comm.allgather_obj(mine)
        open_all = [self._in_records(row[2:]) for part in per_rank for row in part]   # (record, start, end_lower_bound, k)

        def exchange(answers):
            merged = {}
            for part in self.comm.allgather_obj(answers):
                merged.update(part)
            return merged

        fixed = partition.stitch(self.plan, open_all, self._run_end, exchange, self.rank, owner=lambda v: v % N)
        if self.rank == 0:
            rows, ends, i = [], [], 0
            for r, part in enumerate(per_rank):
                for (p, local_row, record, *_rest) in part:
                    pr = self.phase_results[p]
                    g = global_rows(pr.rows_of_rank[:N], r, [local_row])
                    rows.append(int(pr.base_rows) + int(g[0]))
                    ends.append(self._as_reported(record, fixed[i][2]))
                    i += 1
            self.xchg.patch_end(rows, ends)

    def _stitch_local(self):
        """One rank, records cut into chunks: finish the open-ended rows in place (every phase's sequence)."""
        opened = []                                    # (phase, row, record, start, end, k)
        for p, seq in enumerate(self.seqs):
            n_open = 0 if seq is None else int(seq.stats().n_open)
            if n_open:
                opened += [(p,) + tuple(int(x) for x in r) for r in seq.fetch_open(cap=n_open)]
        fixed = partition.stitch(self.plan, [self._in_records(r[2:]) for r in opened], self._run_end, owner=lambda v: 0)
        for (p, row, record, *_rest), (_r, _s, e, _k) in zip(opened, fixed):
            self.seqs[p].patch_end(row, self._as_reported(record, e))

    def _run_end(self, unit, local_pos, k):
        """crf_run_end on the sequence that holds `unit` (one of this rank's shares)."""
        v = self.plan.rank_of_unit(unit.index)
        return self.seqs[v // self.world].run_end(unit.index - self.plan.bounds[v], local_pos, k)

    def _in_records(self, row):
        """An open row as the device reports it -> (record, start, end, k) in record coordinates (Python ints)."""
        record, start, end, k = row
        if not self.long:
            return record, start, end, k
        u = self.plan.units[record]
        return u.record, start + u.d0, end + u.d0, k

    def _as_reported(self, record, end):
        """A stitched end (record coordinates) -> the value patched into the device row (unit-relative in long mode)."""
        if not self.long:
            return end
        end -= self.plan.units[record].d0
        if end > 0xFFFFFFFF:
            raise _cabi.CrfError(f"a perfect repeat of unit {record} ends {end} bases after the unit's origin: runs longer "
                                 f"than 2^32 bases are not supported")
        return end

    def stats(self):
        """Scan statistics of the last step, summed over this rank's phases (kernel_ms, scan_ms, launches, ...)."""
        out = {}
        for seq in self.seqs:
            if seq is None:
                continue
            for name, value in seq.stats().as_dict().items():
                out[name] = out.get(name, 0) + value
        return out

    def fetch(self):
        """Rank 0: the whole job's rows (record, start, end, k), sorted by (record, start, end).  uint32 columns; in long
        mode start and end are uint64 (record coordinates may pass 2^32)."""
        rows = self._fetch_reported()
        return unit_rows_to_records(self.plan.units, *rows) if self.long else rows

    def fetch_units(self):
        """Rank 0, long mode: the rows as the device holds them, (unit index, start, end, k) uint32 with start / end
        relative to the unit's origin plan.units[unit].d0 -- what crf_write_rows_at takes."""
        if not self.long:
            raise _cabi.CrfError("fetch_units(): the rows are unit-relative only when a record is longer than one load")
        return self._fetch_reported()

    def _fetch_reported(self):
        if self.world == 1:
            parts = []
            for p, seq in enumerate(self.seqs):
                if seq is None:
                    continue
                rec, st, en, k = seq.fetch(self._n[p])
                if self.plan is not None and self.load_args[p][2] is None:
                    rec = np.array([u.record for u in self.units[p]], dtype=np.uint32)[rec] if len(rec) else rec
                parts.append((rec, st, en, k))
            if len(parts) == 1:
                return parts[0]
            if not parts:
                return tuple(np.zeros(0, np.uint32) for _ in range(4))
            return tuple(np.concatenate(col) for col in zip(*parts))
        if self.rank != 0:
            raise _cabi.CrfError("the gathered rows live on rank 0")
        return self.xchg.fetch(int(self.last.total_rows))

    def close(self):
        for p, seq in enumerate(self.seqs):
            if seq is not None:
                seq.close()
                self.seqs[p] = None
        if self.xchg is not None:
            self.comm.allgather_obj(None)              # nobody still pushes into a block that is about to go away
            self.xchg.close()
            self.xchg = None


def scan_on_devices(devices, bases, record_starts, lengths, kmin, kmax, min_repeats, min_span, chunk=partition.DEFAULT_CHUNK,
                    halo=partition.DEFAULT_HALO, reads=False, contexts=None, knobs=None, timeout_s=None, phases=1,
                    by_unit=False):
    """One process, one thread per device: scan host `bases` (a uint8 array, or _cabi.PackedPlanes) on all `devices`;
    returns (record, start, end, k) of the whole job.  `contexts`: reuse these _cabi.Context objects (one per device) instead of creating new ones.
    by_unit (a record longer than one load among them): return (RankScan.fetch_units() rows, the plan's units) instead."""
    world = len(devices)
    comms = ThreadComm.split(world)
    ctxs = list(contexts) if contexts else [_cabi.Context(d) for d in devices]
    for i in range(world):                     # ranks never share a context (= a stream): a rank waits for its peers
        if any(ctxs[i] is c for c in ctxs[:i]):
            ctxs[i] = _cabi.Context(devices[i])
    out, errors = {}, []

    def work(rank):
        rs = None
        try:
            rs = RankScan(ctxs[rank], comms[rank], bases, record_starts, lengths, kmin, kmax, min_repeats, min_span,
                          chunk=chunk, halo=halo, reads=reads, knobs=knobs, timeout_s=timeout_s, phases=phases)
            rs.step_async()
            rs.finish()
            if rank == 0:
                out["rows"] = (rs.fetch_units(), rs.plan.units) if by_unit else rs.fetch()
        except BaseException as exc:          # noqa: BLE001 -- re-raised in the caller's thread
            errors.append(exc)
            comms[rank]._s.barrier.abort()
        finally:
            try:
                if rs is not None:
                    rs.close()
            except threading.BrokenBarrierError:
                pass

    if world == 1:
        work(0)
    else:
        threads = [threading.Thread(target=work, args=(r,), name=f"crf-rank{r}") for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
    if errors:
        real = [e for e in errors if not isinstance(e, threading.BrokenBarrierError)]
        raise (real or errors)[0]
    return out["rows"]
