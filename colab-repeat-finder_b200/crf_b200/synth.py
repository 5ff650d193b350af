"""Deterministic synthetic workloads for the BASELINE.json configs (SURVEY.md section 8d).

Bench / test infrastructure, not part of the scan path.  Every base is a pure function of
(seed, record, position) built from 32-bit integer hashes, so the same bytes come out of numpy
(CPU tests) and torch (generated directly in HBM on the GPU box -- a 3.1 Gbp genome is not
shipped through the repo snapshot).

  S22  chr22-shaped single record (config C1/C2 stand-in; benchmark/chr22.fa.gz is not in the
       reference checkout, .MISSING_LARGE_BLOBS:1)
  S38  24 records with the hg38 primary-assembly lengths, ~3.1 Gbp (config C3)
  SX   one record with very long repeats placed around chunk boundaries (config C4)
  SR   n reads x 150 bp (config C5)
"""
import numpy as np

M32 = 0xFFFFFFFF

HG38_LENGTHS = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636,
                138394717, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345,
                83257441, 80373285, 58617616, 64444167, 46709983, 50818468, 156040895, 57227415]
HG38_NAMES = [f"chr{i}" for i in range(1, 23)] + ["chrX", "chrY"]

CELL = 512  # one planted repeat per 512-base cell  (~1.95 per kbp)


ASCII = np.frombuffer(b"ACGT", dtype=np.uint8).astype(np.int64)


class _Backend:
    """The handful of array ops the generators need, on numpy or torch (int64 everywhere)."""

    def __init__(self, device=None):
        self.torch = None
        if device is not None:
            import torch
            self.torch = torch
            self.device = torch.device(device)
        self.ascii_lut = self.from_numpy(ASCII)

    def arange(self, lo, hi):
        if self.torch:
            return self.torch.arange(lo, hi, dtype=self.torch.int64, device=self.device)
        return np.arange(lo, hi, dtype=np.int64)

    def where(self, c, a, b):
        return self.torch.where(c, a, b) if self.torch else np.where(c, a, b)

    def minimum(self, a, b):
        if self.torch:
            return self.torch.clamp(a, max=b)
        return np.minimum(a, b)

    def to_u8(self, x):
        return x.to(self.torch.uint8) if self.torch else x.astype(np.uint8)

    def from_numpy(self, a):
        return self.torch.from_numpy(a).to(self.device) if self.torch else a

    def empty_u8(self, n):
        if self.torch:
            return self.torch.empty(n, dtype=self.torch.uint8, device=self.device)
        return np.empty(n, dtype=np.uint8)

    def sync(self):
        """The generators run on torch's stream, the library on its own: the bytes must be complete before a device
        pointer is handed to crf_seq_load_ascii."""
        if self.torch and self.device.type == "cuda":
            self.torch.cuda.synchronize(self.device)


def hash32(x):
    """lowbias32 on int64 arrays holding values in [0, 2^32) (wrap-around products are masked)."""
    x = ((x ^ (x >> 16)) * 0x7feb352d) & M32
    x = ((x ^ (x >> 15)) * 0x846ca68b) & M32
    return x ^ (x >> 16)


def _k_table(kmax):
    """1024-entry lookup: index uniform -> motif size with P(k) ~ 1/k on [1, kmax]."""
    u = (np.arange(1024) + 0.5) / 1024.0
    return np.minimum(kmax, np.floor((kmax + 1.0) ** u)).astype(np.int64)


def _fill_chunk(be, out, rec_salt, lo, hi, kmax, ktab, lower_case):
    """Bases of record positions [lo, hi) -> out[lo:hi] (ASCII).  Background i.i.d. ACGT, one
    planted perfect repeat per CELL (motif size ~1/k, span 3k + geometric(mean ~20))."""
    p = be.arange(lo, hi)
    cell = p // CELL
    h = hash32((cell * 0x9E3779B1 + rec_salt) & M32)
    h2 = hash32(h ^ 0x5bd1e995)
    k = ktab[(h & 1023)]
    start = cell * CELL + ((h >> 10) & 127)
    extra = (h2 & 15) + ((h2 >> 4) & 15) + ((h2 >> 8) & 7)          # mean ~18.5, max 37
    span = be.minimum(3 * k + extra, CELL - 128 - 4)
    rel = p - start
    in_rep = (rel >= 0) & (rel < span)
    j = be.where(in_rep, rel % k, rel * 0)
    planted = hash32((h2 + j * 0x632BE5AB) & M32) & 3
    background = hash32(((p * 0x85EBCA6B) ^ rec_salt) & M32) & 3
    code = be.where(in_rep, planted, background)
    asc = be.ascii_lut[code]
    if lower_case:
        low = (hash32(((p >> 10) * 0xC2B2AE35 + rec_salt + 7) & M32) & 1) << 5   # 1 kb soft-masked blocks
        asc = asc | low
    out[lo:hi] = be.to_u8(asc)


def _n_runs(rng, length, telomere, centromere_frac, n_gaps, gap_len):
    runs = []
    if length > 4 * telomere:
        runs += [(0, telomere), (length - telomere, length)]
    c = int(length * centromere_frac)
    if c:
        s = int(length * 0.40)
        runs.append((s, min(length, s + c)))
    for _ in range(n_gaps):
        if length > 4 * gap_len:
            s = int(rng.integers(telomere, length - telomere - gap_len))
            runs.append((s, s + gap_len))
    return runs


def generate_records(lengths, seed, device=None, kmax=50, lower_case=True, telomere=10_000,
                     centromere_frac=0.03, n_gaps=20, gap_len=50_000, n_satellites=0, satellite_range=(10_000, 500_000),
                     chunk=1 << 26):
    """Concatenated ASCII records + uint64 offsets.  Returns (bases, offsets, meta)."""
    be = _Backend(device)
    rng = np.random.Generator(np.random.PCG64(seed))
    ktab = be.from_numpy(_k_table(kmax))
    total = int(sum(lengths))
    out = be.empty_u8(total)
    offsets = np.zeros(len(lengths) + 1, dtype=np.uint64)
    meta = {"n_runs": [], "satellites": []}
    base = 0
    for r, length in enumerate(lengths):
        offsets[r] = base
        view = out[base:base + length]
        salt = int(hash32(np.array([(seed * 1000003 + r) & M32], dtype=np.int64))[0])
        for lo in range(0, length, chunk):
            _fill_chunk(be, view, salt, lo, min(length, lo + chunk), kmax, ktab, lower_case)
        for s, e in _n_runs(rng, length, telomere, centromere_frac, n_gaps, gap_len):
            view[s:e] = ord("N")
            meta["n_runs"].append((r, s, e))
        base += length
    offsets[len(lengths)] = base
    # satellites: long perfect arrays (10-500 kbp), placed anywhere in the genome
    for _ in range(n_satellites):
        r = int(rng.integers(0, len(lengths)))
        length = lengths[r]
        ln = int(rng.integers(*satellite_range))
        if length < 4 * ln:
            continue
        s = int(rng.integers(telomere, length - ln - telomere))
        k = int(rng.integers(1, kmax + 1))
        unit = rng.integers(0, 4, size=k)
        if k > 1 and len(set(unit.tolist())) == 1:
            unit[0] = (unit[0] + 1) % 4
        reps = be.from_numpy(np.frombuffer(b"ACGT", dtype=np.uint8)[unit])
        idx = be.arange(0, ln) % k
        out[int(offsets[r]) + s:int(offsets[r]) + s + ln] = reps[idx]
        meta["satellites"].append((r, s, s + ln, k))
    be.sync()
    return out, offsets, meta


def long_record(length, seed=64, device=None, kmax=50, chunk=1 << 26):
    """One record of `length` bases, which may pass 2^32 (the test workload of records longer than one device load).
    The background of _fill_chunk repeats with period 2^32 (32-bit hashes of the position), so every 2^32-block of
    positions gets a salt of its own: the bases at p and p - 2^32 differ, and a position read 2^32 off is caught.
    Returns (bases, offsets, meta) like generate_records."""
    be = _Backend(device)
    ktab = be.from_numpy(_k_table(kmax))
    out = be.empty_u8(length)
    block = 1 << 32
    assert block % chunk == 0
    for lo in range(0, length, chunk):
        salt = int(hash32(np.array([(seed * 1000003 + (lo // block) * 0x9E3779B1) & M32], dtype=np.int64))[0])
        _fill_chunk(be, out, salt, lo, min(length, lo + chunk), kmax, ktab, True)
    be.sync()
    meta = {"workload": f"one record of {length} bp, seed {seed}"}
    return out, np.array([0, length], dtype=np.uint64), meta


def s38(device=None, scale=1.0, seed=38):
    """hg38-sized genome (config C3).  scale < 1 shrinks every record (CPU tests)."""
    lengths = [max(1000, int(n * scale)) for n in HG38_LENGTHS]
    tel = max(10, int(10_000 * min(1.0, scale * 10)))
    bases, offsets, meta = generate_records(
        lengths, seed, device=device, telomere=tel, gap_len=max(50, int(50_000 * min(1.0, scale * 10))),
        n_satellites=100, satellite_range=(max(100, int(10_000 * min(1.0, scale * 10))),
                                           max(1000, int(500_000 * min(1.0, scale * 10)))))
    meta["names"] = HG38_NAMES
    meta["workload"] = f"S38 synthetic hg38-sized genome, 24 records, {int(offsets[-1])} bp, seed {seed}"
    return bases, offsets, meta


def s22(device=None, scale=1.0, seed=22):
    """chr22-shaped single record (configs C1/C2): leading 10.51 Mbp of N, acrocentric gaps."""
    length = max(1000, int(50_818_468 * scale))
    bases, offsets, meta = generate_records([length], seed, device=device, telomere=0, centromere_frac=0.0, n_gaps=0)
    def sc(x):
        return int(x * scale)
    for s, e in [(0, 10_510_000), (12_904_726, 15_168_968), (18_238_733, 18_339_255), (50_808_468, 50_818_468)]:
        bases[sc(s):min(length, sc(e))] = ord("N")
    _Backend(device).sync()
    meta["names"] = ["chr22"]
    meta["workload"] = f"S22 synthetic chr22-shaped record, {length} bp, seed {seed}"
    return bases, offsets, meta


def chr22_path():
    """The real chr22 FASTA of configs C1/C2 if this machine has it: $CRF_CHR22_FASTA, else benchmark/chr22.fa.gz of the
    reference checkout named by $CRF_REFERENCE_DIR (absent from it: .MISSING_LARGE_BLOBS:1), else None."""
    import os
    ref_dir = os.environ.get("CRF_REFERENCE_DIR")
    for path in (os.environ.get("CRF_CHR22_FASTA"), ref_dir and os.path.join(ref_dir, "benchmark", "chr22.fa.gz"),
                 "benchmark/chr22.fa.gz"):
        if path and os.path.isfile(path):
            return path
    return None


def chr22(device=None, scale=1.0):
    """Configs C1/C2: the real chr22 when it can be found (read by the native FASTA reader), else the stand-in S22.
    meta["workload"] says which."""
    path = chr22_path()
    if path is None or scale != 1.0:
        return s22(device=device, scale=scale)
    from . import _cabi
    with _cabi.Fasta(path) as fa:
        bases = fa.bases.copy()
        offsets = fa.offsets.copy()
        names = list(fa.names)
    if device is not None:
        import torch
        bases = torch.from_numpy(bases).to(device)
        torch.cuda.synchronize()
    return bases, offsets, {"names": names, "workload": f"chr22 from {path}, {int(offsets[-1])} bp"}


def sr(n_reads, read_len=150, device=None, seed=150):
    """n_reads x read_len reads (config C5): one planted STR per 512-base cell of the read
    stream (so roughly one read in three carries one), 0.1 % of bases N."""
    be = _Backend(device)
    total = n_reads * read_len
    bases, _, meta = generate_records([total], seed, device=device, kmax=20, lower_case=False, telomere=0,
                                      centromere_frac=0.0, n_gaps=0)
    chunk = 1 << 26
    for lo in range(0, total, chunk):
        p = be.arange(lo, min(total, lo + chunk))
        is_n = (hash32(((p * 0x27D4EB2F) + seed) & M32) % 1000) == 0
        seg = bases[lo:lo + p.shape[0]]
        n_byte = seg * 0 + ord("N")
        bases[lo:lo + p.shape[0]] = be.where(is_n, n_byte, seg)
    be.sync()
    offsets = np.arange(0, total + 1, read_len, dtype=np.uint64)
    meta["workload"] = f"SR {n_reads} reads x {read_len} bp, seed {seed}"
    return bases, offsets, meta


def sx(length, chunk, device=None, seed=4, kset=(1, 2, 3, 7, 16, 31, 32, 33, 50)):
    """One record with perfect repeats of 0.5 / 1 / 2.5 chunks whose start / end sit at offsets
    -k-1 .. +k+1 around multiples of `chunk` (config C4), plus a run to the last base and runs
    abutting N."""
    bases, offsets, meta = generate_records([length], seed, device=device, telomere=0, centromere_frac=0.0, n_gaps=0,
                                            lower_case=False)
    be = _Backend(device)
    rng = np.random.Generator(np.random.PCG64(seed))
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    cursor = chunk // 3
    planted = []
    for k in kset:
        for mult in (0.5, 1.0, 2.5):
            ln = int(chunk * mult) + int(rng.integers(-k - 1, k + 2))
            boundary = ((cursor // chunk) + 1) * chunk
            s = boundary + int(rng.integers(-k - 1, k + 2))
            if s + ln + chunk >= length:
                break
            unit = rng.integers(0, 4, size=k)
            if k > 1 and len(set(unit.tolist())) == 1:
                unit[0] = (unit[0] + 1) % 4
            reps = be.from_numpy(lut[unit])
            bases[s:s + ln] = reps[be.arange(0, ln) % k]
            planted.append((s, s + ln, k))
            cursor = s + ln + chunk // 7
    # a run reaching the very last base, and N directly before / after a run
    bases[length - 5000:] = ord("G")
    if length > 40_000:
        bases[length - 20_000:length - 19_000] = ord("N")
        bases[length - 19_000:length - 15_000] = be.from_numpy(lut[np.array([0, 3])])[be.arange(0, 4000) % 2]
        bases[length - 15_000:length - 14_990] = ord("N")
    be.sync()
    meta["planted"] = planted
    meta["workload"] = f"SX chunk-crossing repeats, {length} bp, chunk {chunk}, seed {seed}"
    return bases, offsets, meta
