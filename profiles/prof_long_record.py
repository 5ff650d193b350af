#!/usr/bin/env python3
"""A record longer than one device load (synth.long_record, 2^32 + 150 Mbp, motif sizes 1-50): the scan rate over all of
its loads on one GPU (multi.RankScan, one rank, as api.scan_arrays runs it) and the command line's wall time, FASTA file
on disk -> BED file on disk.  Prints one JSON line; the GPU's name and power limit are part of it.
   python profiles/prof_long_record.py [--length N] [--repeats R]"""
import argparse
import contextlib
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))
import torch  # noqa: E402
from crf_b200 import api, cli, multi, partition, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--length", type=int, default=(1 << 32) + 150_000_000)
ap.add_argument("--repeats", type=int, default=3)
args = ap.parse_args()

bases, _, _ = synth.long_record(args.length, device="cuda:0")
host = bases.cpu().numpy()
del bases
torch.cuda.synchronize()
ctx = api.get_context(0)
t0 = time.perf_counter()
rs = multi.RankScan(ctx, multi.ThreadComm.split(1)[0], host, [0], [args.length], 1, 50, 3, 9)
load_s = time.perf_counter() - t0
steps = []
for _ in range(args.repeats):
    t0 = time.perf_counter()
    rs.step_async()
    n = rs.finish()
    wall = time.perf_counter() - t0
    st = rs.stats()
    steps.append({"wall_s": round(wall, 4), "scan_ms": round(st["scan_ms"], 2), "kernel_ms": round(st["kernel_ms"], 2),
                  "rows": int(n)})
phases = rs.phases
rs.close()
best = min(steps, key=lambda s: s["scan_ms"])

work = tempfile.mkdtemp(prefix="crf_long_")
try:
    fa = os.path.join(work, "long.fa")
    with open(fa, "wb") as f:
        f.write(b">long\n")
        f.write(memoryview(host))
        f.write(b"\n")
    del host
    cwd = os.getcwd()
    os.chdir(work)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        cli.main([fa, "-o", "long"])
    cli_s = time.perf_counter() - t0
    bed_bytes = os.path.getsize(os.path.join(work, "long.bed"))
    os.chdir(cwd)
finally:
    shutil.rmtree(work, ignore_errors=True)

try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
except OSError:
    gpu = torch.cuda.get_device_name(0)
print(json.dumps({"workload": f"synth.long_record({args.length}), k 1-50, min_repeats 3, min_span 9", "gpu": gpu,
                  "loads": phases, "chunk": partition.DEFAULT_CHUNK, "halo": partition.DEFAULT_HALO,
                  "load_s": round(load_s, 3), "steps": steps,
                  "scan_gbp_per_s": round(args.length / (best["scan_ms"] * 1e6), 1),
                  "kernel_gbp_per_s": round(args.length / (best["kernel_ms"] * 1e6), 1),
                  "cli_fasta_to_bed_s": round(cli_s, 2), "bed_bytes": bed_bytes}))
