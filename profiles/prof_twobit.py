#!/usr/bin/env python3
""".2bit input, in one process: S38 (synth.s38, 24 records, 3.09 Gbp) written as FASTA (one line per record), as gzip -1
FASTA and as .2bit (tests/test_twobit.py:s38_twobit).
  1. the reader alone (crf_fasta_open) on every file, stage times on stderr (CRF_FASTA_TRACE=1), twice each;
  2. the command line, file on disk -> BED on disk (stdout to /dev/null), host clock around cli.main, twice each, after a
     warm-up run on a small file;
  3. the loads of the whole genome: crf_seq_load_2bit from the .2bit handle and crf_seq_load_packed_runs from the FASTA
     handle's planes (load_ms of crf_seq_info, device events), 3 times each, then once each under torch.profiler for the
     kernel times of twobit_pack_kernel, repack_kernel and mask_runs_kernel.
   python profiles/prof_twobit.py"""
import contextlib
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))
import torch  # noqa: E402
from crf_b200 import api, cli, fasta  # noqa: E402
from tests.test_twobit import s38_twobit  # noqa: E402

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)

work = tempfile.mkdtemp(prefix="crf_twobit_")
tb_path, fa_path, gz_path = (os.path.join(work, f) for f in ("S38.2bit", "S38.fa", "S38.fa.gz"))
t0 = time.perf_counter()
bases, offsets, meta = s38_twobit(tb_path)
host = bases.cpu().numpy()
del bases
torch.cuda.empty_cache()
comp = zlib.compressobj(1, zlib.DEFLATED, 31)
with open(fa_path, "wb") as f, open(gz_path, "wb") as g:
    for r, name in enumerate(meta["names"]):
        rec = b">" + name.encode() + b"\n" + host[int(offsets[r]):int(offsets[r + 1])].tobytes() + b"\n"
        f.write(rec)
        for i in range(0, len(rec), 64 << 20):
            g.write(comp.compress(rec[i:i + (64 << 20)]))
    g.write(comp.flush())
del host
print(f"{meta['workload']}; files written in {time.perf_counter() - t0:.1f} s: " +
      ", ".join(f"{os.path.basename(p)} {os.path.getsize(p) / 1e6:.1f} MB" for p in (fa_path, gz_path, tb_path)), flush=True)
files = [fa_path, gz_path, tb_path]

# ---- 1. the reader ----------------------------------------------------------------------------------------------------
os.environ["CRF_FASTA_TRACE"] = "1"
for path in files:
    for rep in range(2):
        t0 = time.perf_counter()
        with fasta.open_fasta(path, pinned=2) as h:
            dt = time.perf_counter() - t0
            print(f"reader {os.path.basename(path)} run {rep}: {h.format}, {h.n_records} records, {h.total_bases} bases: "
                  f"{dt * 1e3:.1f} ms wall", flush=True)
        sys.stderr.flush()
del os.environ["CRF_FASTA_TRACE"]

# ---- 2. the command line ----------------------------------------------------------------------------------------------
os.chdir(work)
with open("warm.fa", "w") as f:
    f.write(">w\n" + "ACGT" * 1000 + "\n")
with open(os.devnull, "w") as null, contextlib.redirect_stdout(null):
    cli.main(["warm.fa", "-o", "warm"])
for path in files:
    for rep in range(2):
        with open(os.devnull, "w") as null, contextlib.redirect_stdout(null):
            t0 = time.perf_counter()
            rc = cli.main([path, "-o", "out"])
            dt = time.perf_counter() - t0
        print(f"cli {os.path.basename(path)}: run {rep}: {dt * 1e3:8.1f} ms wall, rc {rc}, BED "
              f"{os.path.getsize('out.bed') / 1e6:.1f} MB", flush=True)
os.chdir(ROOT)

# ---- 3. the loads -----------------------------------------------------------------------------------------------------
ctx = api.get_context()
with fasta.open_fasta(tb_path, pinned=2) as tb, fasta.open_fasta(fa_path, pinned=2) as fa:
    planes = fa.packed()

    def load_2bit():
        return ctx.load_2bit(tb, max_motif_cap=50)

    def load_runs():
        return ctx.load_packed(planes, fa.offsets, max_motif_cap=50)
    for name, fn in (("crf_seq_load_2bit", load_2bit), ("crf_seq_load_packed_runs", load_runs)) * 2:
        ms = []
        for _ in range(3):
            t0 = time.perf_counter()
            with fn() as seq:
                wall = (time.perf_counter() - t0) * 1e3
                ms.append(f"{seq.info().load_ms:.1f} ms device events / {wall:.1f} ms host clock")
        print(f"{name}: " + ", ".join(ms), flush=True)
    from torch.profiler import ProfilerActivity, profile
    for name, fn in (("crf_seq_load_2bit", load_2bit), ("crf_seq_load_packed_runs", load_runs)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with fn():
                torch.cuda.synchronize()
        kernels = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA" and "kernel" in ev.name:
                kernels.setdefault(ev.name, []).append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
        for k, v in sorted(kernels.items()):
            print(f"  {name}: {k}: {len(v)} launches, {sum(v) / 1e3:.3f} ms", flush=True)
shutil.rmtree(work, ignore_errors=True)
