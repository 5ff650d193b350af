"""Command line of the drop-in.

Same flags, defaults, stdout lines and output files as the reference's main()
(the reference's perfect_repeat_finder.py:83-179), re-organised around two code paths:

  FASTA file  -> <basename(prefix)>.bed in the working directory (chrom, start_0based, end, motif); a FASTQ file is
                 read the same way, its read names as chrom; a .2bit file too, loaded from its packed bytes, and an
                 unaligned BAM file, loaded from its 4-bit codes
  raw string  -> <prefix>.tsv with a header line (start_0based, end, motif)

Deliberate deviations (SURVEY.md section 8b):
  * a FASTA file WITHOUT --interval works (the reference raises AttributeError at :139): all records go to the GPU
    in one load and one scan (a record longer than one load: in several), rows are written by the native writer
    (crf_write_rows);
  * --plot is accepted but plotting is out of scope here (matplotlib is not a dependency).
"""
import argparse
import os
import re
import sys

import numpy as np

from . import _cabi, api, fasta

# (flags, keyword arguments) -- the reference's options, prf:86-98
_FILTER_OPTIONS = [
    (("-min", "--min-motif-size"), dict(default=1, type=int, help="Smallest motif size (bp) to look for.")),
    (("-max", "--max-motif-size"), dict(default=50, type=int, help="Largest motif size (bp) to look for.")),
    (("--min-repeats",), dict(default=3, type=int, help="Report a locus only if the motif occurs at least this many "
                                                         "times in a row.")),
    (("--min-span",), dict(default=9, type=int, help="Report a locus only if it covers at least this many bases.")),
]
_OTHER_OPTIONS = [
    (("-i", "--interval"), dict(help="Restrict the scan to chrom:start_0based-end (FASTA input only).")),
    # not in the reference: its Hail pipeline runs --interval once per 500 kb tile and concatenates the BED files
    (("--intervals",), dict(metavar="BED", help="Run --interval for every line (chrom start_0based end ...) of a BED file "
                                                "in one pass (FASTA input only): the output is the concatenation, in file "
                                                "order, of what --interval writes for each line.  With --devices, the "
                                                "intervals run on the first GPU.")),
    (("-p", "--plot"), dict(help="Plot file name (accepted for compatibility; plotting is not part of this build).")),
    (("-o", "--output-prefix"), dict(help="Prefix of the output file: <prefix>.tsv for a sequence given on the command "
                                          "line, <basename(prefix)>.bed for a FASTA file.")),
    (("--verbose",), dict(action="store_true", help="Accepted for compatibility.")),
    (("--debug",), dict(action="store_true", help="Accepted for compatibility.")),
    (("--show-progress-bar",), dict(action="store_true", help="Accepted for compatibility.")),
    # not in the reference: its scale-out is a separate Hail Batch pipeline (run_hail_batch_pipeline.py:96-123)
    (("--devices",), dict(default=os.environ.get("CRF_DEVICES"),
                          help="GPUs for whole-FASTA runs, e.g. 0-7 or 0,2,3 (default: $CRF_DEVICES, else one GPU). "
                               "The records are cut into chunks, every GPU scans its share and the rows are gathered on "
                               "the first one over NVLink; the BED file is identical to a single-GPU run.")),
    (("--mask",), dict(choices=("soft", "hard"), help="Also write <basename(prefix)>.masked.fa (FASTA input only, not with "
                                                      "--interval / --intervals): the records with every base inside a "
                                                      "reported repeat lower-cased (soft) or replaced by N (hard).  For "
                                                      "FASTQ or BAM input: <basename(prefix)>.masked.fq, qualities "
                                                      "unchanged.")),
]


def build_parser():
    parser = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter,
                                     description="Find perfect tandem repeats (B200 build).")
    filters = parser.add_argument_group("Repeat Filters")
    for flags, kw in _FILTER_OPTIONS:
        filters.add_argument(*flags, **kw)
    for flags, kw in _OTHER_OPTIONS:
        parser.add_argument(*flags, **kw)
    parser.add_argument("input_sequence", help="A nucleotide string, or the path of a FASTA or FASTQ file (plain or .gz), "
                                               "of a UCSC .2bit file or of an unaligned BAM file (read as `samtools "
                                               "fastq -n` writes it)")
    return parser


def _check_filters(parser, args):
    """prf:102-109 -- same messages, exit status 2."""
    for value, flag, floor in ((args.min_motif_size, "--min-motif-size", "1"),):
        if value < 1:
            parser.error(f"{flag} is set to {value}. It must be at least {floor}.")
    if args.max_motif_size < args.min_motif_size:
        parser.error(f"--max-motif-size is set to {args.max_motif_size}. It must be at least --min-motif-size.")
    if args.min_repeats < 1:
        parser.error(f"--min-repeats is set to {args.min_repeats}. It must be at least 1.")
    if args.min_span < 1:
        parser.error(f"--min-span is set to {args.min_span}. It must be at least 1.")


def parse_devices(text):
    """"0-3" / "0,2,5" / "1" -> list of device indices (None or "" -> one device: api.default_device())."""
    if text is None or str(text).strip() == "":
        return [api.default_device()]
    out = []
    for part in str(text).split(","):
        part = part.strip()
        if "-" in part:
            lo, hi = part.split("-", 1)
            out.extend(range(int(lo), int(hi) + 1))
        else:
            out.append(int(part))
    if not out or min(out) < 0:
        raise ValueError(f"invalid device list {text!r}")
    return out


def group_records(lengths, max_motif_size, limit=None):
    """Cut the record list into consecutive groups that each fit one device load: a load lays every record out
    as length + max_motif_size positions and holds at most crf_load_limit() of them (32-bit positions on the
    device).  A single record above the limit is its own group (its units are spread over several
    loads, see _whole_fasta_to_bed).  Returns [(first, last)), ...].  One search per group, not a Python step per
    record: a reads file has millions of them."""
    limit = _cabi.load_limit(max_motif_size) if limit is None else limit
    csum = np.cumsum(np.asarray(lengths, dtype=np.int64) + max_motif_size)
    groups, first, n = [], 0, csum.size
    while first < n:
        before = int(csum[first - 1]) if first else 0
        last = max(int(np.searchsorted(csum, before + limit, side="right")), first + 1)
        groups.append((first, last))
        first = last
    return groups


def _whole_fasta_to_bed(fa, args, bed_path, mask_rows=None):
    """Every record of the file: as few loads as the position limit allows (one for a human genome), one scan per
    load (on one GPU, or split over --devices), native row writer.  The groups are slices of the reader's buffer (no
    copies on the Python side).  Returns the row count per record.  mask_rows: a list that gets the rows of every write
    (see _paint_mask)."""
    devices = parse_devices(getattr(args, "devices", None))
    lengths = np.diff(fa.offsets.astype(np.int64))
    counts = np.zeros(fa.n_records, dtype=np.int64)
    open(bed_path, "wb").close()
    limit = _cabi.load_limit(args.max_motif_size)
    groups = group_records(lengths, args.max_motif_size)
    # a .2bit file on one GPU: each group is loaded from the file's packed bytes (0.25 B/bp, packed into the layout on the
    # device) and its motifs are read from them; the text is never decoded
    # (a BAM file the same way, from its 4-bit codes at 0.5 B/bp)
    packed_src = None
    if len(devices) == 1 and fa.format == "2bit":
        packed_src, load, write = fa.twobit(), "load_2bit", _cabi.write_rows_twobit
    elif len(devices) == 1 and fa.format == "bam":
        packed_src, load, write = fa.nibbles(), "load_nibbles", _cabi.write_rows_nibbles
    if packed_src is not None and all(not lengths[f:l].size or int(lengths[f:l].max()) + args.max_motif_size <= limit
                                      for f, l in groups):
        data = packed_src.dna if fa.format == "2bit" else packed_src.nib
        for first, last in groups:
            if not int(lengths[first:last].sum()):
                continue
            with getattr(api.get_context(devices[0]), load)(packed_src.records(first, last),
                                                            max_motif_cap=args.max_motif_size) as seq:
                n = seq.scan(args.min_motif_size, args.max_motif_size, args.min_repeats, args.min_span)
                rec, start, end, k = seq.fetch(n)
            whole_file = first == 0 and last == fa.n_records
            write(bed_path, fa.names_blob if whole_file else fa.names[first:last], data, packed_src.rec_byte[first:last],
                  rec, start, end, k, append=True)
            if mask_rows is not None:
                mask_rows.append((rec, start, end, fa.offsets[first:last]))
            counts[first:last] += np.bincount(rec.astype(np.int64, copy=False), minlength=last - first)
        return counts
    # the text is packed to 2-bit planes + mask on the host (threaded, at ingest) and uploaded at 0.375 B/bp; the ASCII
    # buffer stays on the host for the motif column
    planes = fa.packed() if fa.total_bases else None
    for first, last in groups:
        total = int(lengths[first:last].sum())
        base0 = int(fa.offsets[first])
        blob = fa.bases[base0:base0 + total]
        offsets = fa.offsets[first:last + 1] - np.uint64(base0)
        if total and int(lengths[first:last].max()) + args.max_motif_size > limit:
            # a record longer than one load (its group holds only it): its units go to several loads, on one GPU or over
            # --devices; rows come back relative to their unit and the writer adds the unit's 64-bit origin
            from . import multi, partition
            (unit, start, end, k), units = multi.scan_on_devices(
                devices, planes, fa.offsets[first:last], lengths[first:last], args.min_motif_size, args.max_motif_size,
                args.min_repeats, args.min_span, chunk=partition.DEFAULT_CHUNK, halo=partition.DEFAULT_HALO,
                contexts=[api.get_context(d) for d in devices], by_unit=True)
            rec_of = np.array([u.record for u in units], dtype=np.int64)
            origin = np.array([u.d0 for u in units], dtype=np.uint64)
            names = [fa.names[first + r] for r in rec_of.tolist()]
            _cabi.write_rows(bed_path, names, blob, offsets[rec_of] + origin, unit, start, end, k, append=True, origin=origin)
            if mask_rows is not None:                              # unit-relative rows: the unit's origin goes to dst
                mask_rows.append((unit, start, end, fa.offsets[first + rec_of] + origin))
            counts[first:last] += np.bincount(rec_of[unit.astype(np.int64)], minlength=last - first)
            continue
        if total:
            if len(devices) > 1:
                from . import multi
                many_short = (last - first) > 4096 and int(lengths[first:last].max()) < (1 << 20)
                rec, start, end, k = multi.scan_on_devices(
                    devices, planes, fa.offsets[first:last], lengths[first:last], args.min_motif_size, args.max_motif_size,
                    args.min_repeats, args.min_span, reads=many_short, contexts=[api.get_context(d) for d in devices])
            else:
                with api.get_context(devices[0]).load_packed(planes, fa.offsets[first:last + 1],
                                                             max_motif_cap=args.max_motif_size) as seq:
                    n = seq.scan(args.min_motif_size, args.max_motif_size, args.min_repeats, args.min_span)
                    rec, start, end, k = seq.fetch(n)
            whole_file = first == 0 and last == fa.n_records          # the usual case: hand the name table over as it is
            _cabi.write_rows(bed_path, fa.names_blob if whole_file else fa.names[first:last], blob, offsets, rec, start,
                             end, k, append=True)
            if mask_rows is not None:
                mask_rows.append((rec, start, end, fa.offsets[first:last]))
            counts[first:last] += np.bincount(rec.astype(np.int64, copy=False), minlength=last - first)
    return counts


def _paint_mask(ctx, mask_rows, n_bases):
    """One crf_mask_rows call for the rows of a whole file.  mask_rows: (record, start, end, dst) parts, each numbering its
    own records, dst[r] = where record r of the part starts in the file's bases.  Returns the mask words."""
    parts = [(np.zeros(0, np.uint32),) * 3 + (np.zeros(0, np.uint64),)] + mask_rows
    rec, n_dst = [], 0
    for r, _, _, d in parts:
        rec.append(np.asarray(r, dtype=np.int64) + n_dst)
        n_dst += len(d)
    start, end, dst = (np.concatenate([p[j] for p in parts]) for j in (1, 2, 3))
    return ctx.mask_rows(np.concatenate(rec), start, end, dst.astype(np.uint64), n_bases)


def read_bed_intervals(parser, path):
    """(chrom, start, end) of every interval line of a BED file; '#', 'track' and 'browser' lines and blank lines are
    skipped, columns after the third are ignored.  A malformed line is a parser error naming it."""
    out = []
    with open(path, "rt") as f:
        for lineno, line in enumerate(f, 1):
            fields = line.split()
            if not fields or fields[0].startswith("#") or fields[0] in ("track", "browser"):
                continue
            try:
                out.append((fields[0], int(fields[1]), int(fields[2])))
            except (IndexError, ValueError):
                parser.error(f"--intervals {path}, line {lineno}: expected 'chrom start_0based end', got {line.rstrip()!r}")
    return out


def _intervals_to_bed(parser, fa, args, bed_path):
    """--intervals: every line as --interval would run it (same rows, same exceptions), batched by
    intervals.run_intervals on the first of --devices; one BED file, the lines' outputs concatenated in file order."""
    from . import intervals
    lines = read_bed_intervals(parser, args.intervals)
    first_index = {}
    for i, name in enumerate(fa.names):                                   # duplicate names: the first one (names.index)
        first_index.setdefault(name, i)
    for chrom, _, _ in lines:                                             # every line is checked before any scan
        if chrom not in first_index:
            parser.error(f"Chromosome {chrom} not found in the input FASTA file")
    m = len(lines)
    rec = np.array([first_index[c] for c, _, _ in lines], dtype=np.int64)
    lengths = np.diff(fa.offsets.astype(np.int64))
    a = np.array([s for _, s, _ in lines], dtype=np.int64)
    b = np.minimum(np.array([e for _, _, e in lines], dtype=np.int64), lengths[rec])        # prf:139-140
    device = parse_devices(getattr(args, "devices", None))[0]

    def single(i):
        return api.detect_repeats(fa.record(int(rec[i])).tobytes(), intervals._settings_for(args, int(a[i]), int(b[i])),
                                  device=device)

    planes = fa.packed() if fa.total_bases else _cabi.pack_ascii(b"").with_runs()
    outcome, origin, iv, start, end, k = intervals.run_intervals(planes, fa.offsets.astype(np.int64)[rec], lengths[rec], a, b,
                                                                 args, device, None, single)
    for o in outcome:
        if isinstance(o, BaseException):
            raise o
    counts = np.bincount(iv, minlength=m)
    start, end = start + origin[iv], end + origin[iv]                     # record coordinates, 64-bit
    extra = [(i, o) for i, o in enumerate(outcome) if o]                 # rows of the intervals done one by one
    if extra:
        for i, rows in extra:
            origin[i] = rows[0][0]
            counts[i] = len(rows)
        iv = np.concatenate([iv] + [np.full(len(rows), i, np.int64) for i, rows in extra])
        start = np.concatenate([start] + [np.array([r[0] for r in rows], np.int64) for _, rows in extra])
        end = np.concatenate([end] + [np.array([r[1] for r in rows], np.int64) for _, rows in extra])
        k = np.concatenate([k] + [np.array([len(r[2]) for r in rows], np.int64) for _, rows in extra])
        order = np.argsort(iv, kind="stable")
        iv, start, end, k = iv[order], start[order], end[order], k[order]
    # The writer takes 32-bit start / end relative to a 64-bit origin per writer record.  A row of a batched interval lies
    # in a prefix that fits one load, but an interval of the single-interval path may cover a whole record longer than
    # 2^32 bases: an interval's rows are cut into writer records at every 2^31 bases past its origin (in row order, so
    # the file order is unchanged), which keeps start and end below 2^32 for every run shorter than 2^31 bases.
    if (end - start >= 1 << 31).any():
        raise NotImplementedError("--intervals: a repeat of 2^31 bases or more cannot be written")
    chunk = (start - origin[iv]) >> 31
    new = np.ones(iv.size, dtype=bool)
    new[1:] = (iv[1:] != iv[:-1]) | (chunk[1:] != chunk[:-1])
    wrec = np.cumsum(new) - 1
    first = np.flatnonzero(new)
    w_iv = iv[first]
    w_origin = origin[w_iv] + (chunk[first] << 31)
    _cabi.write_rows(bed_path, [lines[i][0] for i in w_iv.tolist()], fa.bases, fa.offsets.astype(np.int64)[rec[w_iv]] + w_origin,
                     wrec, start - w_origin[wrec], end - w_origin[wrec], k, origin=w_origin.astype(np.uint64))
    for lo in range(0, m, 65536):                                         # the two lines of --interval, per line, batched
        sys.stdout.write("".join(f"Processing {c_} ({e_ - s_:,d} bp)\nFound {n_:,d} repeats\n"
                                 for (c_, s_, _), e_, n_ in zip(lines[lo:lo + 65536], b[lo:lo + 65536].tolist(),
                                                                 counts[lo:lo + 65536].tolist())))


def default_prefix(path, fmt):
    """The output prefix when -o is not given.  FASTA: the (unanchored) regex of prf:114, as the reference has it.  FASTQ:
    the path without a trailing .fastq / .fq, optionally followed by .gz / .bgz (reads.fq.gz -> reads).  .2bit: the path
    without a trailing .2bit.  BAM: the path without a trailing .bam."""
    if fmt == "2bit":
        return re.sub(r"\.2bit$", "", path)
    if fmt == "bam":
        return re.sub(r"\.bam$", "", path)
    if fmt == "fastq":
        return re.sub(r"\.(fastq|fq)(\.(gz|bgz))?$", "", path)
    return re.sub(".fa(sta)?(.gz)?", "", path)


def _run_fasta(parser, args):
    if args.intervals and args.interval:
        parser.error("--intervals and --interval cannot be used together")
    if args.mask and (args.interval or args.intervals):
        parser.error("--mask writes whole records: it cannot be used with --interval or --intervals")
    mask_rows = [] if args.mask else None
    # (page-locked planes only: the planes are what is uploaded, the text stays on the host for the motif column; a FASTQ
    # or BAM file's qualities are kept only for the masked FASTQ)
    with fasta.open_fasta(args.input_sequence, pinned=2, qualities=bool(args.mask)) as fa:
        if not args.output_prefix:                                                 # FASTA or FASTQ: known once it is read
            args.output_prefix = default_prefix(args.input_sequence, fa.format)
        bed_path = f"{os.path.basename(args.output_prefix)}.bed"                   # always in the working directory
        mask_path = f"{os.path.basename(args.output_prefix)}.masked.{'fq' if fa.format in ('fastq', 'bam') else 'fa'}" \
            if args.mask else None
        if args.intervals:
            _intervals_to_bed(parser, fa, args, bed_path)
        elif args.interval:
            fields = re.split("[:-]", args.interval)
            if len(fields) != 3:
                parser.error("Invalid --interval format. Must be chrom:start_0based-end")
            args.interval_chrom = fields[0]
            args.interval_start_0based, args.interval_end = int(fields[1]), int(fields[2])
            if args.interval_chrom not in fa.names:
                parser.error(f"Chromosome {args.interval_chrom} not found in the input FASTA file")
            chosen = fa.record(fa.names.index(args.interval_chrom))
            args.interval_end = min(args.interval_end, len(chosen))                    # prf:139-140
            print(f"Processing {args.interval_chrom} ({args.interval_end - args.interval_start_0based:,d} bp)")
            rows = api.detect_repeats(chosen.tobytes(), args)
            print(f"Found {len(rows):,d} repeats")
            with open(bed_path, "wt") as bed_file:
                bed_file.write("".join(f"{args.interval_chrom}\t{s}\t{e}\t{m}\n" for s, e, m in rows))
        elif args.min_repeats == 1:
            # the reference's single-copy quirks are per record (wrap-around at each record's position 0): one call each
            with open(bed_path, "wt") as bed_file:
                for i, name in enumerate(fa.names):
                    print(f"Processing {name} ({len(fa.record(i)):,d} bp)")
                    rows = api.detect_repeats(fa.record(i).tobytes(), args)
                    print(f"Found {len(rows):,d} repeats")
                    bed_file.write("".join(f"{name}\t{s}\t{e}\t{m}\n" for s, e, m in rows))
                    if mask_rows is not None and rows:             # one mask record per row: 64-bit starts go to dst
                        s = np.array([r[0] for r in rows], dtype=np.uint64)
                        e = np.array([r[1] for r in rows], dtype=np.uint64)
                        mask_rows.append((np.arange(len(rows)), np.zeros(len(rows), np.uint32), e - s, fa.offsets[i] + s))
        else:
            counts = _whole_fasta_to_bed(fa, args, bed_path, mask_rows)
            lengths = np.diff(fa.offsets.astype(np.int64))
            names, lengths, counts = fa.names, lengths.tolist(), counts.tolist()
            for lo in range(0, len(names), 65536):            # the reference's two lines per record; batched, a reads
                sys.stdout.write("".join(                     # file has millions of records
                    f"Processing {n_} ({l_:,d} bp)\nFound {c_:,d} repeats\n"
                    for n_, l_, c_ in zip(names[lo:lo + 65536], lengths[lo:lo + 65536], counts[lo:lo + 65536])))
        if mask_rows is not None:                                  # every record has been scanned: paint once, write
            words = _paint_mask(api.get_context(parse_devices(getattr(args, "devices", None))[0]), mask_rows, fa.total_bases)
            if fa.format in ("fastq", "bam"):
                _cabi.write_fastq_masked(mask_path, fa.names_blob, fa.bases, fa.quals, fa.offsets, words,
                                         hard=args.mask == "hard")
            else:
                _cabi.write_fasta_masked(mask_path, fa.names_blob, fa.bases, fa.offsets, words, hard=args.mask == "hard")
    print(f"Wrote results to {bed_path}")
    if mask_path:
        print(f"Wrote masked sequence to {mask_path}")


def _run_raw(parser, args):
    if args.interval:
        parser.error("The --interval option is only supported for FASTA files.")
    if args.intervals:
        parser.error("The --intervals option is only supported for FASTA files.")
    if args.mask:
        parser.error("The --mask option is only supported for FASTA files.")
    if not args.output_prefix:
        args.output_prefix = "repeats"
    tsv_path = f"{args.output_prefix}.tsv"
    rows = api.detect_repeats(args.input_sequence, args)
    print(f"Found {len(rows):,d} repeats")
    with open(tsv_path, "wt") as tsv_file:
        tsv_file.write("start_0based\tend\tmotif\n")
        tsv_file.writelines(f"{s}\t{e}\t{m}\n" for s, e, m in rows)
    print(f"Wrote results to {tsv_path}")
    if args.plot:
        if len(args.input_sequence) > 5_000:
            print(f"Warning: The input sequence is too long ({len(args.input_sequence):,d} bp). Skipping plot...")
        else:
            print("Warning: plotting is not part of this build (matplotlib is not a dependency). Skipping plot...")


def main(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    _check_filters(parser, args)
    if os.path.isfile(args.input_sequence):
        _run_fasta(parser, args)
    elif set(args.input_sequence.upper()) <= set("ACGTN"):
        _run_raw(parser, args)
    else:
        parser.error(f"Invalid input: {args.input_sequence}. This should be a FASTA file path or a string of nucleotides.")
    return 0


if __name__ == "__main__":
    sys.exit(main())
