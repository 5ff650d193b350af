#!/usr/bin/env python3
"""BAM input, in one process (the card's name and power limit first):
  C5   10^7 reads of 150 bp (synth.sr), as a level-1 unaligned BAM and as the same reads in .fq.bgz (tests/test_fastq.py
       c5_files), and
  HIFI 2 x 10^5 reads of 15 kbp with qualities, half of them reverse (flag 0x14), generated from seed 9, as a level-1 BAM.
For each:
  1. the reader alone (crf_fasta_open, pinned=2 as the command line opens it) in a process of its own: wall time and peak
     RSS (VmHWM, which a new process starts afresh), twice each;
  2. the loads of all reads: crf_seq_load_nibbles from the BAM handle and crf_seq_load_packed_runs from the planes of the
     same reads (load_ms of crf_seq_info, device events), 3 times each, then once each under torch.profiler for the
     kernel times of nibble_pack_kernel and repack_kernel;
  3. the command line, file on disk -> BED on disk (stdout to /dev/null), host clock around the process, twice each.
   python profiles/prof_bam.py"""
import os
import resource
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))
import torch  # noqa: E402
from crf_b200 import api, fasta  # noqa: E402
from tests.test_fastq import bgzf, c5_files  # noqa: E402

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
work = tempfile.mkdtemp(prefix="crf_bam_")
CODES = np.zeros(256, np.uint8)
for i, c in enumerate(b"=ACMGRSVTWYHKDBN"):
    CODES[c] = i


def bam_bytes(names, reads, quals, flags):
    """An unaligned BAM stream of equal-length reads (names: (n, w) bytes without NUL; reads / quals: (n, L) letters and
    Phred values; flags: (n,)), built with numpy."""
    n, L = reads.shape
    w = names.shape[1] + 1
    fixed = np.zeros((n, 36), np.uint8)
    fixed32 = fixed.view("<i4")
    fixed32[:, 0] = 32 + w + (L + 1) // 2 + L                         # block_size
    fixed32[:, 1] = fixed32[:, 2] = -1                                 # refID, pos
    fixed[:, 12] = w                                                   # l_read_name
    fixed[:, 13] = 255
    fixed[:, 14:16] = np.frombuffer(np.uint16(4680).tobytes(), np.uint8)
    fixed[:, 18:20] = flags.astype("<u2").view(np.uint8).reshape(n, 2)
    fixed32[:, 5] = L
    fixed32[:, 6] = fixed32[:, 7] = -1
    c = CODES[reads]
    if L & 1:
        c = np.concatenate([c, np.zeros((n, 1), np.uint8)], 1)
    seq = (c[:, 0::2] << 4) | c[:, 1::2]
    rec = np.concatenate([fixed, names, np.zeros((n, 1), np.uint8), seq, quals], 1)
    text = b"@HD\tVN:1.6\tSO:unknown\n"
    head = b"BAM\1" + np.int32(len(text)).tobytes() + text + np.int32(0).tobytes()
    return head + rec.tobytes()


def c5_workload():
    host, offsets, quals, paths = c5_files(__import__("pathlib").Path(work), 10_000_000, ("fq.bgz",))
    n, rl = 10_000_000, 150
    idx = np.arange(n, dtype=np.int64)
    names = np.empty((n, 9), np.uint8)
    names[:, 0] = ord("r")
    for d in range(8):
        names[:, 8 - d] = ord("0") + (idx // 10 ** d) % 10
    blob = bam_bytes(names, host.reshape(n, rl), quals.reshape(n, rl) - 33, np.full(n, 4))
    path = os.path.join(work, "reads.bam")
    with open(path, "wb") as f:
        f.write(bgzf(blob, level=1))
    os.remove(paths["fa"])
    return {"C5 uBAM": path, "C5 fq.bgz": str(paths["fq.bgz"])}


def hifi_workload():
    rng = np.random.default_rng(9)
    n, rl = 200_000, 15_000
    path = os.path.join(work, "hifi.bam")
    with open(path, "wb") as f:
        for lo in range(0, n, 20_000):                                 # 20 000 reads (300 Mbp) at a time
            m = 20_000
            unit = rng.integers(0, 4, (m, 6))
            codes = np.where(rng.random((m, rl)) < 0.3, np.tile(unit, rl // 6), rng.integers(0, 4, (m, rl)))
            reads = np.frombuffer(b"ACGT", np.uint8)[codes]
            quals = rng.integers(0, 60, (m, rl), dtype=np.uint8)
            names = np.frombuffer(b"".join(b"m84_%08d/ccs" % (lo + i) for i in range(m)), np.uint8).reshape(m, -1)
            blob = bam_bytes(names, reads, quals, np.where(np.arange(m) % 2, 0x14, 0x4))
            if lo:
                blob = blob[len(b"BAM\1") + 4 + 22 + 4:]                  # the header once
            f.write(bgzf(blob, level=1)[:-28])                        # (one end-of-file block, at the end)
        f.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return {"HIFI uBAM": path}


READER = ("import sys, time\n"
          f"sys.path.insert(0, {os.path.join(ROOT, 'colab-repeat-finder_b200')!r})\n"
          "from crf_b200 import _cabi\n"
          "_cabi.lib()\n"
          "t0 = time.perf_counter()\n"
          "with _cabi.Fasta(sys.argv[1], pinned=2) as fa:\n"
          "    dt = time.perf_counter() - t0\n"
          "    hwm = [l for l in open('/proc/self/status') if l.startswith('VmHWM')][0].split()[1]\n"
          "    print(f'{fa.format}, {fa.n_records} records, {fa.total_bases} bases: {dt * 1e3:.0f} ms wall, peak RSS '\n"
          "          f'{int(hwm) / 1024:.0f} MiB')\n")

t0 = time.perf_counter()
files = {**c5_workload(), **hifi_workload()}
print(f"files written in {time.perf_counter() - t0:.1f} s: " +
      ", ".join(f"{k} {os.path.getsize(p) / 1e6:.0f} MB" for k, p in files.items()), flush=True)

# ---- 1. the reader ----------------------------------------------------------------------------------------------------
for name, path in files.items():
    for rep in range(2):
        out = subprocess.run([sys.executable, "-c", READER, path], capture_output=True, text=True, check=True).stdout
        print(f"reader {name} run {rep}: {out.strip()}", flush=True)

# ---- 2. the loads -----------------------------------------------------------------------------------------------------
ctx = api.get_context()
for name in ("C5 uBAM", "HIFI uBAM"):
    with fasta.open_fasta(files[name], pinned=2) as fa:
        t0 = time.perf_counter()
        planes = fa.packed()
        print(f"{name}: decode + host planes {time.perf_counter() - t0:.2f} s", flush=True)

        def load_nibbles():
            return ctx.load_nibbles(fa, max_motif_cap=50)

        def load_runs():
            return ctx.load_packed(planes, fa.offsets, max_motif_cap=50)
        rows = {}
        for lname, fn in (("crf_seq_load_nibbles", load_nibbles), ("crf_seq_load_packed_runs", load_runs)) * 2:
            ms = []
            for _ in range(3):
                t0 = time.perf_counter()
                with fn() as seq:
                    wall = (time.perf_counter() - t0) * 1e3
                    ms.append(f"{seq.info().load_ms:.1f} ms device events / {wall:.1f} ms host clock")
                    if lname not in rows:
                        rows[lname] = [a.copy() for a in seq.fetch(seq.scan(1, 50, 3, 9))]
            print(f"{name}: {lname}: " + ", ".join(ms), flush=True)
        assert all(np.array_equal(a, b) for a, b in zip(*rows.values())), "the two loads give different rows"
        print(f"{name}: both loads give the same {len(rows['crf_seq_load_nibbles'][0])} rows", flush=True)
        del rows
        from torch.profiler import ProfilerActivity, profile
        for lname, fn in (("crf_seq_load_nibbles", load_nibbles), ("crf_seq_load_packed_runs", load_runs)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                with fn():
                    torch.cuda.synchronize()
            kernels = {}
            for ev in prof.events():
                if ev.device_type.name == "CUDA" and "kernel" in ev.name:
                    kernels.setdefault(ev.name, []).append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
            for k, v in sorted(kernels.items()):
                print(f"  {name}: {lname}: {k}: {len(v)} launches, {sum(v) / 1e3:.3f} ms", flush=True)
        del planes

# ---- 3. the command line ----------------------------------------------------------------------------------------------
for name, path in files.items():
    for rep in range(2):
        with open(os.devnull, "w") as null:
            t0 = time.perf_counter()
            rc = subprocess.run([sys.executable, os.path.join(ROOT, "perfect_repeat_finder.py"), path, "-o", "out"],
                                stdout=null, cwd=work).returncode
            dt = time.perf_counter() - t0
        print(f"cli {name}: run {rep}: {dt:.2f} s wall (process), rc {rc}, BED "
              f"{os.path.getsize(os.path.join(work, 'out.bed')) / 1e6:.1f} MB", flush=True)
print(f"peak RSS of this process {resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024:.0f} MiB")
shutil.rmtree(work, ignore_errors=True)
