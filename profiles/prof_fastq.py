#!/usr/bin/env python3
"""FASTQ input, in one process: config C5 (10^7 reads of 150 bp, synth.sr, motif 1-20) written as FASTQ (seeded qualities)
and as FASTA (one line per read) in three containers each: plain, gzip -1 and BGZF (level 1).
  1. the reader alone (crf_fasta_open) on every file, with its stage times (CRF_FASTA_TRACE=1, on stderr), twice each;
  2. the command line, file on disk -> BED on disk (stdout to /dev/null), host clock around cli.main, twice each;
  3. the same with --mask soft on the plain files (BED + masked FASTQ / FASTA).
   python profiles/prof_fastq.py [--reads 10000000]"""
import argparse
import contextlib
import os
import shutil
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from crf_b200 import cli, fasta, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=10_000_000)
args = ap.parse_args()
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)


def gzip1(raw):
    comp = zlib.compressobj(1, zlib.DEFLATED, 31)
    return b"".join([comp.compress(raw[i:i + (64 << 20)]) for i in range(0, len(raw), 64 << 20)] + [comp.flush()])


def bgzf(raw, block=65280):
    def member(chunk):
        comp = zlib.compressobj(1, zlib.DEFLATED, -15)
        data = comp.compress(chunk) + comp.flush()
        return (b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\0\xff" + struct.pack("<H", 6) + b"BC" +
                struct.pack("<HH", 2, 12 + 6 + len(data) + 8 - 1) + data + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    with ThreadPoolExecutor(16) as ex:
        return b"".join(ex.map(member, (raw[i:i + block] for i in range(0, len(raw), block)))) + member(b"")


n, rl = args.reads, 150
bases, offsets, meta = synth.sr(n, device="cuda:0")
reads = bases.cpu().numpy().reshape(n, rl)
del bases
torch.cuda.synchronize()
rng = np.random.default_rng(150)
quals = rng.integers(33, 127, (n, rl), dtype=np.uint8)
quals[:, 0] = np.frombuffer(b"@+>I", np.uint8)[rng.integers(0, 4, n)]
idx = np.arange(n, dtype=np.int64)
name = np.empty((n, 9), np.uint8)
name[:, 0] = ord("r")
for d in range(8):
    name[:, 8 - d] = ord("0") + (idx // 10 ** d) % 10
fa = np.empty((n, 11 + rl + 1), np.uint8)
fa[:, 0], fa[:, 1:10], fa[:, 10], fa[:, 11:11 + rl], fa[:, -1] = ord(">"), name, 10, reads, 10
fq = np.empty((n, 11 + rl + 3 + rl + 1), np.uint8)
fq[:, 0], fq[:, 1:10], fq[:, 10], fq[:, 11:11 + rl] = ord("@"), name, 10, reads
fq[:, 11 + rl:14 + rl] = np.frombuffer(b"\n+\n", np.uint8)
fq[:, 14 + rl:14 + 2 * rl], fq[:, -1] = quals, 10
del reads, quals, name
work = tempfile.mkdtemp(prefix="crf_fastq_")
files = []
for kind, arr in (("fa", fa), ("fq", fq)):
    raw = arr.tobytes()
    for suffix, make in (("", None), (".gz", gzip1), (".bgz", bgzf)):
        path = os.path.join(work, f"reads.{kind}{suffix}")
        t0 = time.perf_counter()
        with open(path, "wb") as f:
            f.write(make(raw) if make else raw)
        files.append(path)
        print(f"wrote {os.path.basename(path)}: {os.path.getsize(path) / 1e6:.1f} MB ({len(raw) / 1e6:.1f} MB of text) in "
              f"{time.perf_counter() - t0:.1f} s", flush=True)
    del raw
del fa, fq
print(f"{meta['workload']}", flush=True)

# ---- 1. the reader ---------------------------------------------------------------------------------------------------
os.environ["CRF_FASTA_TRACE"] = "1"
for path in files:
    for rep in range(2):
        print(f"reader {os.path.basename(path)} run {rep}:", flush=True)
        t0 = time.perf_counter()
        with fasta.open_fasta(path, pinned=2) as h:
            dt = time.perf_counter() - t0
            print(f"  {h.format}, {h.n_records} records, {h.total_bases} bases: {dt * 1e3:.1f} ms wall", flush=True)
        sys.stderr.flush()
del os.environ["CRF_FASTA_TRACE"]

# ---- 2. / 3. the command line ----------------------------------------------------------------------------------------
os.chdir(work)
for extra in ([], ["--mask", "soft"]):
    for path in files:
        if extra and not path.endswith((".fa", ".fq")):
            continue
        for rep in range(2):
            with open(os.devnull, "w") as null, contextlib.redirect_stdout(null):
                t0 = time.perf_counter()
                rc = cli.main([path, "-min", "1", "-max", "20", "-o", "out"] + extra)
                dt = time.perf_counter() - t0
            masked = [f for f in os.listdir(work) if f.startswith("out.masked")]
            msg = f", {masked[0]} {os.path.getsize(masked[0]) / 1e6:.1f} MB" if masked else ""
            print(f"cli {os.path.basename(path)} {' '.join(extra) or '(BED only)'}: run {rep}: {dt * 1e3:8.1f} ms wall, rc {rc}, "
                  f"BED {os.path.getsize('out.bed') / 1e6:.1f} MB{msg}", flush=True)
            for f in masked:
                os.remove(f)
os.chdir(ROOT)
shutil.rmtree(work, ignore_errors=True)
