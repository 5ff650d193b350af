#!/usr/bin/env python3
"""Many reads from Python: one api.detect_repeats call per read against detect_repeats_batch and scan_batch (host bytes and
a CUDA tensor).  Workload: synth.sr reads of 150 bp (config C5's shape), motif sizes 1-20, --min-repeats 3 --min-span 9.
For every size: the wall time of each call (host clock around a call that ends in a stream sync), twice in one process;
the per-read loop only on a seeded sample of reads (after 50 warm-up calls), extrapolated to all of them and labelled so.
   python profiles/prof_batch.py [--sizes 10000,1000000,10000000] [--sample 1000]"""
import argparse
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from crf_b200 import api, batch, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="10000,1000000,10000000")
ap.add_argument("--sample", type=int, default=1000)
args = ap.parse_args()
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
fs = argparse.Namespace(min_motif_size=1, max_motif_size=20, min_repeats=3, min_span=9)


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


for n in [int(x) for x in args.sizes.split(",")]:
    bases, offsets, meta = synth.sr(n, device="cuda:0")
    blob = bases.cpu().numpy().tobytes()
    reads = [blob[i:i + 150].decode() for i in range(0, len(blob), 150)]
    print(f"{meta['workload']}: {len(blob)} bp", flush=True)
    for rep in range(2):
        rows, dt = timed(lambda: batch.detect_repeats_batch(reads, fs, device=0))
        print(f"n={n} run {rep}: detect_repeats_batch (str in, tuples out) {dt:.3f} s, {sum(map(len, rows))} rows, "
              f"loads {batch.last_stats['loads']}", flush=True)
        del rows
        cols, dt = timed(lambda: batch.scan_batch(blob, offsets, fs, device=0))
        print(f"n={n} run {rep}: scan_batch host bytes -> numpy {dt * 1e3:.1f} ms, {cols[0].size} rows", flush=True)
        torch.cuda.synchronize()
        tcols, dt = timed(lambda: batch.scan_batch(bases, offsets, fs, device=0))
        same = all(np.array_equal(t.cpu().numpy(), h) for t, h in zip(tcols, cols))
        print(f"n={n} run {rep}: scan_batch CUDA tensor -> CUDA tensors {dt * 1e3:.1f} ms, {tcols[0].numel()} rows, "
              f"bit-identical to host input: {same}", flush=True)
        del cols, tcols
    sample = random.Random(n).sample(range(n), min(args.sample, n))
    for i in sample[:50]:
        api.detect_repeats(reads[i], fs, device=0)
    _, dt = timed(lambda: [api.detect_repeats(reads[i], fs, device=0) for i in sample])
    print(f"n={n}: api.detect_repeats per read on a seeded sample of {len(sample)} reads: {dt / len(sample) * 1e6:.1f} us "
          f"per read -> EXTRAPOLATED to {n} reads: {dt / len(sample) * n:.1f} s", flush=True)
    del bases, blob, reads
    torch.cuda.empty_cache()
