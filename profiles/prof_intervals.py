#!/usr/bin/env python3
"""--intervals on a genome, against one -i run per interval.  Two workloads on S38 (the synthetic hg38-sized genome)
written as a 60-column FASTA:
  (a) a 500 kb tiling of every record (the Hail pipeline's fan-out, run_hail_batch_pipeline.py), k 1-6 (its setting);
  (b) 10^6 intervals of 1 kbp at seeded positions, k 1-50.
For each: the --intervals wall time (FASTA on disk -> BED on disk), the time spent in load / crf_interval_stop / scan /
fetch (host clock around calls that each end in a stream sync), the window rounds, the intervals left to the
single-interval path, and the -i loop timed on a seeded sample of intervals, extrapolated to all of them.
   python profiles/prof_intervals.py [--scale 1.0] [--sample 300]"""
import argparse
import contextlib
import io
import os
import random
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from crf_b200 import api, cli, intervals, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--scale", type=float, default=1.0)
ap.add_argument("--sample", type=int, default=300)
args = ap.parse_args()
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)

# What one warp's walk across a satellite costs: crf_interval_stop on a load holding ONE interval whose end lies 1 kbp
# into a 500 kb satellite (the warp walks ~499 kb to the satellite's end), against the same call with the interval
# ending in random sequence (a walk of a few words: launch, copies and sync).  Median of 30 calls after 5 warm-up calls.
from crf_b200 import _cabi  # noqa: E402
gen0 = np.random.default_rng(1)
flank = [np.frombuffer(b"ACGT", np.uint8)[gen0.integers(0, 4, 20_000)].tobytes() for _ in range(2)]
sat_seq = flank[0] + b"ACGGTTCAGT" * 50_000 + flank[1]
sat_planes = _cabi.pack_ascii(sat_seq).with_runs()
for kmax in (6, 50):
    with api.get_context(0).load_packed(sat_planes, max_motif_cap=kmax, ranges=([0], [len(sat_seq)], None, None)) as sq:
        med = {}
        for label, e in (("random", 5_000), ("satellite", 21_000)):
            ts = []
            for rep in range(35):
                t0 = time.perf_counter()
                T = int(sq.interval_stop(1, kmax, [e], [len(sat_seq)])[0])
                ts.append(time.perf_counter() - t0)
            med[label] = float(np.median(ts[5:]))
            print(f"walk k 1-{kmax}: interval end {e} ({label}): stop at {T}, {med[label] * 1e6:.1f} us per call "
                  f"(median of 30)", flush=True)
        walk = T - 21_000
        dt = med["satellite"] - med["random"]
        print(f"walk k 1-{kmax}: {walk} bases across the satellite cost {dt * 1e6:.1f} us more "
              f"= {walk / max(dt, 1e-9) / 1e9:.2f} Gbp/s for one warp", flush=True)
bases, offsets, meta = synth.s38(device="cuda:0", scale=args.scale)
seq = bases.cpu().numpy()
del bases
torch.cuda.synchronize()
work = tempfile.mkdtemp(prefix="crf_iv_")
fa = os.path.join(work, "genome.fa")
with open(fa, "wb") as f:
    for r, name in enumerate(meta["names"]):
        rec = seq[int(offsets[r]):int(offsets[r + 1])]
        f.write(b">" + name.encode() + b"\n")
        n_full = rec.size // 60
        lines = np.empty((n_full, 61), dtype=np.uint8)
        lines[:, :60] = rec[:n_full * 60].reshape(n_full, 60)
        lines[:, 60] = 10
        lines.tofile(f)
        del lines
        if rec.size % 60:
            f.write(rec[n_full * 60:].tobytes() + b"\n")
print(f"{meta['workload']}: {seq.size} bp written as FASTA", flush=True)
os.chdir(work)
names = meta["names"]
lengths = np.diff(offsets.astype(np.int64))
rng = random.Random(2026)

tiling = [(names[r], a, min(a + 500_000, int(lengths[r]))) for r in range(len(names)) for a in range(0, int(lengths[r]), 500_000)]
gen = np.random.default_rng(7)
rec_of = gen.choice(len(names), size=1_000_000, p=lengths / lengths.sum())
starts = (gen.random(1_000_000) * np.maximum(lengths[rec_of] - 1000, 1)).astype(np.int64)
kbp = [(names[r], int(a), int(a) + 1000) for r, a in zip(rec_of.tolist(), starts.tolist())]

for label, lines, flags in (("(a) 500 kb tiling, k 1-6", tiling, ["-min", "1", "-max", "6"]),
                            ("(b) 10^6 x 1 kbp, k 1-50", kbp, ["-min", "1", "-max", "50"])):
    with open("iv.bed", "w") as f:
        f.write("".join(f"{c}\t{a}\t{b}\n" for c, a, b in lines))
    base = [fa, "--min-repeats", "3", "--min-span", "9"] + flags
    for rep in range(2):
        out = io.StringIO()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(out):
            cli.main(base + ["--intervals", "iv.bed", "-o", "many"])
        wall = time.perf_counter() - t0
        st = dict(intervals.last_stats)
        rows = sum(1 for _ in open("many.bed", "rb"))
        print(f"{label}: {len(lines)} intervals, run {rep}: --intervals {wall:.2f} s wall, {rows} rows; "
              f"load {st['load_s'] * 1e3:.1f} ms, stop {st['stop_s'] * 1e3:.1f} ms, scan {st['scan_s'] * 1e3:.1f} ms, "
              f"fetch {st['fetch_s'] * 1e3:.1f} ms over {st['loads']} loads; window rounds {st['rounds']}; "
              f"fallback {st['fallback']} (too long {st['too_long']})", flush=True)
    # the -i loop without its FASTA read: what `-i` does with a line once the file is in memory (record bytes cached, so
    # this favours the loop: a real -i process reads the whole FASTA again every time)
    sample = rng.sample(lines, min(args.sample, len(lines)))
    fs = cli.build_parser().parse_args(base)
    recs = {c: seq[int(offsets[names.index(c)]):int(offsets[names.index(c) + 1])].tobytes() for c, _, _ in sample}
    t0 = time.perf_counter()
    for c, a, b in sample:
        api.detect_repeats(recs[c], intervals._settings_for(fs, a, min(b, len(recs[c]))))
    dt = time.perf_counter() - t0
    print(f"{label}: -i path (api.detect_repeats per interval, FASTA read excluded) on a seeded sample of {len(sample)} "
          f"intervals: {dt:.2f} s, {dt / len(sample) * 1e3:.2f} ms per interval -> EXTRAPOLATED to {len(lines)} intervals: "
          f"{dt / len(sample) * len(lines):.1f} s", flush=True)
os.chdir(ROOT)
shutil.rmtree(work, ignore_errors=True)
