#!/usr/bin/env python3
"""Repeat masks (crf_mask_rows, the masked FASTA writer, repeat_mask), three measurements in one process:
  1. the command line on S38 (the hg38-sized synthetic genome written as a 60-column FASTA): FASTA on disk -> BED on disk,
     against FASTA on disk -> BED + soft-masked FASTA on disk (--mask soft); host clock around cli.main, twice each;
  2. crf_mask_rows on the S38 rows of that run (motif 1-50): wall time of the call (it ends in a stream sync) with rows and
     mask on the device and with both on the host (what the CLI does), five times each; then, in a separate
     torch.profiler run, the device time of its two kernels;
  3. repeat_mask on config C5 (10^7 reads of 150 bp, motif 1-20) from host bytes and from a CUDA tensor, twice each, with
     scan_batch alone beside it.
   python profiles/prof_mask.py [--scale 1.0] [--reads 10000000]"""
import argparse
import contextlib
import io
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from crf_b200 import api, batch, cli, mask, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--scale", type=float, default=1.0)
ap.add_argument("--reads", type=int, default=10_000_000)
args = ap.parse_args()
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)

# ---- 1. the command line on S38 ----------------------------------------------------------------------------------------
bases, offsets, meta = synth.s38(device="cuda:0", scale=args.scale)
seq = bases.cpu().numpy()
del bases
torch.cuda.synchronize()
work = tempfile.mkdtemp(prefix="crf_mask_")
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
print(f"{meta['workload']}: {seq.size} bp in {len(meta['names'])} records, {os.path.getsize(fa) / 1e6:.1f} MB FASTA", flush=True)
os.chdir(work)
for rep in range(2):
    for extra in ([], ["--mask", "soft"]):
        out = io.StringIO()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(out):
            rc = cli.main([fa, "-o", "out"] + extra)
        dt = time.perf_counter() - t0
        size = os.path.getsize("out.masked.fa") / 1e6 if extra else 0.0
        print(f"cli {' '.join(extra) or '(BED only)'}: run {rep}: {dt * 1e3:8.1f} ms wall, rc {rc}, "
              f"BED {os.path.getsize('out.bed') / 1e6:.1f} MB" + (f", masked FASTA {size:.1f} MB" if extra else ""), flush=True)
        if extra:
            os.remove("out.masked.fa")

# ---- 2. crf_mask_rows on the S38 rows ------------------------------------------------------------------------------------
fs = argparse.Namespace(min_motif_size=1, max_motif_size=50, min_repeats=3, min_span=9)
dev = torch.from_numpy(seq).to("cuda:0")
rec, st, en, _ = batch.scan_batch(dev, offsets, fs, device=0)
n_rows, n_bases = rec.numel(), seq.size
dst = np.asarray(offsets, np.uint64)[:-1]
ctx = api.get_context(0)
words = torch.empty((n_bases + 31) // 32, dtype=torch.int32, device="cuda:0")
torch.cuda.synchronize()
host_cols = [c.cpu().numpy() for c in (rec, st, en)]
covered = None
for label, call in (("rows + mask in HBM", lambda: ctx.mask_rows(rec.data_ptr(), st.data_ptr(), en.data_ptr(), dst, n_bases,
                                                                   n_rows=n_rows, mask=words.data_ptr())),
                    ("rows + mask on the host", lambda: ctx.mask_rows(*host_cols, dst, n_bases))):
    times = []
    for _ in range(6):
        t0 = time.perf_counter()
        got = call()
        times.append(time.perf_counter() - t0)
    if got is not None:
        covered = int(np.unpackbits(got.view(np.uint8)).sum())
    print(f"crf_mask_rows, {label}: {n_rows} rows over {n_bases} bases: wall "
          f"{', '.join(f'{t * 1e3:.2f}' for t in times[1:])} ms (first call {times[0] * 1e3:.2f} ms)", flush=True)
same = np.array_equal(words.cpu().numpy().view(np.uint32), ctx.mask_rows(*host_cols, dst, n_bases))
print(f"masked bases {covered} ({covered / n_bases:.2%}); device and host masks identical: {same}", flush=True)
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(5):
        ctx.mask_rows(rec.data_ptr(), st.data_ptr(), en.data_ptr(), dst, n_bases, n_rows=n_rows, mask=words.data_ptr())
for e in prof.key_averages():
    if "mask" in e.key or "Memset" in e.key:
        print(f"profiler (5 calls, rows + mask in HBM): {e.key}: {e.count} launches, "
              f"{e.device_time_total / e.count / 1e3:.3f} ms each", flush=True)
del dev, rec, st, en, words, host_cols, seq
os.chdir(ROOT)
shutil.rmtree(work, ignore_errors=True)
torch.cuda.empty_cache()

# ---- 3. repeat_mask on config C5 -----------------------------------------------------------------------------------------
fs = argparse.Namespace(min_motif_size=1, max_motif_size=20, min_repeats=3, min_span=9)
bases, offsets, meta = synth.sr(args.reads, device="cuda:0")
blob = bases.cpu().numpy().tobytes()
torch.cuda.synchronize()
print(f"{meta['workload']}: {len(blob)} bp", flush=True)
for rep in range(2):
    t0 = time.perf_counter()
    cols = batch.scan_batch(blob, offsets, fs, device=0)
    t_scan = time.perf_counter() - t0
    t0 = time.perf_counter()
    host = mask.repeat_mask(blob, offsets, fs, device=0)
    t_host = time.perf_counter() - t0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tmask = mask.repeat_mask(bases, offsets, fs, device=0)
    torch.cuda.synchronize()
    t_dev = time.perf_counter() - t0
    same = np.array_equal(tmask.cpu().numpy(), host)
    print(f"reads run {rep}: scan_batch host bytes {t_scan * 1e3:.1f} ms ({cols[0].size} rows); repeat_mask host bytes -> "
          f"numpy {t_host * 1e3:.1f} ms; CUDA tensor -> CUDA tensor {t_dev * 1e3:.1f} ms; {int(host.sum())} masked bases; "
          f"bit-identical: {same}", flush=True)
    del cols, host, tmask
