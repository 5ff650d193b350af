"""Records longer than one device load (crf_load_limit, about 2^32 positions).

Such a record is cut into partition units that go to several loads of one rank (multi.RankScan phases, on one GPU or
over --devices); each load reports its units as records of their own, rows stay 32-bit and unit-relative on the device,
and the host adds the units' origins in 64 bits (api.scan_arrays, the CLI through crf_write_rows_at).

CPU tests patch the load limit down to a few thousand positions and answer the scans with a closed form of what
crf_scan documents (include/crf.h), so that several loads, load cuts and stitched runs appear on records of a few
kilobases.  The -m gpu tests scan one record of 2^32 + 150 Mbp on the device."""
import argparse
import os
import random
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, cli, multi, partition  # noqa: E402
from oracle import oracle  # noqa: E402
from tests.fake_ctx import FakeContext, FakeSeq, FakeXchg, unpack_planes  # noqa: E402
from tests.helpers import ns, random_seq  # noqa: E402
from tests.test_host_cpu import _ClosedFormSeq, _runs_single_copy  # noqa: E402

KMIN, KMAX, MR, MS = 1, 10, 3, 9
LIMIT, CHUNK, HALO = 1500, 300, 64


# ---- CPU stand-in: per-unit closed form of crf_scan, loads checked against the patched limit ---------------------------

class _ClosedFormUnits(FakeSeq):
    def scan(self, kmin, kmax, min_repeats, min_span, flags=0, **knobs):
        rows = []
        for i, u in enumerate(self.units):
            text = bytes(u).upper()
            if min_repeats == 1:
                st, en, kk = _runs_single_copy(text, kmin, kmax, min_span)
            else:
                cf = _ClosedFormSeq(text)
                cf.scan(kmin, kmax, min_repeats, min_span, flags=flags)
                st, en, kk = cf.rows[:, 0], cf.rows[:, 1], cf.rows[:, 2]
            for a, b, c in zip(st.tolist(), en.tolist(), kk.tolist()):
                if self.own_lo[i] <= a < self.own_hi[i]:
                    rows.append((i, a, b, c))
        self._rows = np.array(rows, dtype=np.int64).reshape(-1, 4)
        self._open = np.zeros((0, 5), np.uint32)
        self._apply_map()
        return len(rows)


class _Ctx(FakeContext):
    """Records every load's layout size (sum of length + max_motif_cap) so the tests can hold them to the limit."""

    def __init__(self):
        self.loads = []

    def _seq(self, bases, starts, lens, own_lo, own_hi, cap):
        self.loads.append(int(sum(int(n) + cap for n in lens)))
        return _ClosedFormUnits(bases, starts, lens, own_lo, own_hi)

    def load(self, bases, offsets=None, max_motif_cap=50, on_device=False):
        n = len(bases)
        offsets = np.array([0, n], dtype=np.uint64) if offsets is None else np.asarray(offsets, dtype=np.uint64)
        return self._seq(bases, offsets[:-1], np.diff(offsets.astype(np.int64)), None, None, max_motif_cap)

    def load_ranges(self, bases, starts, lengths, own_lo=None, own_hi=None, max_motif_cap=50, on_device=False):
        return self._seq(bases, starts, lengths, own_lo, own_hi, max_motif_cap)

    def load_packed(self, planes, offsets=None, max_motif_cap=50, ranges=None):
        text = unpack_planes(planes)
        if ranges is not None:
            return self._seq(text, *ranges, max_motif_cap)
        return self.load(text, offsets, max_motif_cap)


@pytest.fixture
def small_loads(monkeypatch):
    """Load limit LIMIT, units of CHUNK + HALO: a record of a few kbp needs several loads."""
    ctxs = []

    def get_context(device=None):
        ctxs.append(_Ctx())
        return ctxs[-1]
    monkeypatch.setattr(_cabi, "load_limit", lambda cap: LIMIT)
    monkeypatch.setattr(partition, "DEFAULT_CHUNK", CHUNK)
    monkeypatch.setattr(partition, "DEFAULT_HALO", HALO)
    monkeypatch.setattr(api, "get_context", get_context)
    monkeypatch.setattr(multi._cabi, "Xchg", FakeXchg)
    monkeypatch.setattr(FakeXchg, "dist", None)
    return ctxs


def long_record(seed, n):
    """Repeat-rich text with periodic runs longer than the halo every ~700 bp (some cross a load cut) and one that runs
    to the last base."""
    rng = random.Random(seed)
    parts, total = [], 0
    while total < n - 400:
        piece = random_seq(rng, rng.randint(300, 700), alphabets=["ACGT", "ACGTN", "ACGTacgtNn"])
        unit = "".join(rng.choice("ACGT") for _ in range(rng.randint(1, KMAX)))
        piece += unit * (HALO // len(unit) + rng.randint(2, 40))
        parts.append(piece)
        total += len(piece)
    text = "".join(parts)[:n - 150] + "GA" * 75
    for i, c in enumerate(load_cuts(n, KMAX)[0]):                        # a run three halos long across every load cut
        unit = "ACCGT"[:1 + i % 5]
        text = text[:c - HALO] + (unit * (3 * HALO))[:3 * HALO] + text[c + 2 * HALO:]
    return text


def load_cuts(n, kmax, mr=MR, ms=MS, world=1):
    plan, phases = partition.plan_loads([n], world, 1, LIMIT, chunk=CHUNK,
                                        halo=max(HALO, partition.halo_needed(kmax, mr, ms)), kmax=kmax,
                                        min_repeats=mr, min_span=ms)
    return [plan.units[b].u0 for b in plan.bounds[1:-1]], phases


def test_scan_arrays_dtypes_follow_the_record_length(small_loads):
    seq = long_record(1, 5000)
    start, end, k = api.scan_arrays(seq[:1000].encode(), KMIN, KMAX, MR, MS)
    assert start.dtype == np.uint32 and end.dtype == np.uint32 and len(small_loads[-1].loads) == 1
    start, end, k = api.scan_arrays(seq.encode(), KMIN, KMAX, MR, MS)
    assert start.dtype == np.uint64 and end.dtype == np.uint64
    assert len(small_loads[-1].loads) > 2 and max(small_loads[-1].loads) <= LIMIT


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_detect_repeats_full_mode_over_several_loads(small_loads, seed):
    seq = long_record(seed, 6000 + 1000 * seed)
    fs = ns(min_motif_size=KMIN, max_motif_size=KMAX, min_repeats=MR, min_span=MS)
    want = oracle.detect_repeats(seq, fs)
    assert api.detect_repeats(seq, fs) == want
    loads = small_loads[-1].loads
    assert len(loads) >= 4 and max(loads) <= LIMIT
    cuts, phases = load_cuts(len(seq), KMAX)
    assert phases == len(loads) and len(cuts) == phases - 1
    crossing = [(s, e) for s, e, _ in want if any(s < c < e for c in cuts)]
    assert crossing and any(e - s > HALO for s, e in crossing)             # runs across load cuts, longer than the halo
    assert want[-1][1] == len(seq)                                         # a run to the last base


@pytest.mark.parametrize("min_repeats,kmin,min_span", [(3, 1, 9), (2, 1, 5), (1, 2, 5), (1, 1, 4)])
def test_detect_repeats_interval_mode_over_several_loads(small_loads, min_repeats, kmin, min_span):
    seq = long_record(7, 7000)
    rng = random.Random(min_repeats * 100 + min_span)
    checked = 0
    for a, b in [(0, 6000), (40, 5200), (1234, 7000), (700, 6900)] + [(rng.randint(0, 500), rng.randint(5000, 7000))]:
        fs = ns(min_motif_size=kmin, max_motif_size=KMAX, min_repeats=min_repeats, min_span=min_span,
                interval_start_0based=a, interval_end=b)
        try:
            want, exc = oracle.detect_repeats(seq, fs), None
        except (AssertionError, IndexError) as e:
            want, exc = None, type(e)
        if exc is not None:
            with pytest.raises(exc):
                api.detect_repeats(seq, fs)
            continue
        assert api.detect_repeats(seq, fs) == want, (a, b)
        checked += 1
    assert checked >= 3
    assert any(len(c.loads) > 2 for c in small_loads)                      # the main scan went over several loads


def test_detect_repeats_single_copy_full_mode_over_several_loads(small_loads):
    seq = long_record(11, 6500)
    fs = ns(min_motif_size=2, max_motif_size=KMAX, min_repeats=1, min_span=6)
    assert api.detect_repeats(seq, fs) == oracle.detect_repeats(seq, fs)
    assert any(len(c.loads) > 2 for c in small_loads)


def _fasta(path, records):
    path.write_text("".join(f">{n}\n" + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)) for n, s in records))


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_cli_bed_of_a_record_longer_than_a_load(small_loads, tmp_path, monkeypatch, capsys, devices):
    """FASTA -> BED: one record far above the (patched) load limit between two short ones, on one rank and on two
    thread ranks (--devices 0,0): the BED is the oracle's rows, the stdout counts are per record."""
    rng = random.Random(5)
    records = [("short1", random_seq(rng, 400)), ("long", long_record(13, 9000)), ("short2", random_seq(rng, 250))]
    _fasta(tmp_path / "in.fa", records)
    want, counts = [], []
    for name, seq in records:
        rows = oracle.detect_repeats(seq, ns(min_motif_size=KMIN, max_motif_size=KMAX, min_repeats=MR, min_span=MS))
        want += [f"{name}\t{s}\t{e}\t{m}\n" for s, e, m in rows]
        counts.append(len(rows))
    monkeypatch.chdir(tmp_path)
    argv = [str(tmp_path / "in.fa"), "-max", str(KMAX), "-o", "out"] + (["--devices", devices] if devices else [])
    assert cli.main(argv) == 0
    assert (tmp_path / "out.bed").read_text() == "".join(want)
    out = capsys.readouterr().out
    for (name, seq), c in zip(records, counts):
        assert f"Processing {name} ({len(seq):,d} bp)\nFound {c:,d} repeats\n" in out
    assert any(len(c.loads) > 2 for c in small_loads)


def test_planner_on_a_five_gigabase_record():
    """No data: the plan of one 5e9-base record at the library's own limit, on one and on two ranks."""
    limit = _cabi.load_limit(50)
    n = 5_000_000_000
    for world in (1, 2):
        plan, phases = partition.plan_loads([n], world, 1, limit, chunk=partition.DEFAULT_CHUNK,
                                            halo=partition.DEFAULT_HALO, kmax=50, min_repeats=3, min_span=9)
        assert phases == (2 if world == 1 else 1)                          # 5e9 bp: two loads in all
        assert all(partition.load_positions(plan, v, 50) <= limit for v in range(phases * world))
        owned = [(u.u0, u.u1) for u in plan.units]
        assert owned[0][0] == 0 and owned[-1][1] == n and all(a[1] == b[0] for a, b in zip(owned, owned[1:]))
        assert all(u.d0 == max(0, u.u0 - 1) and u.d1 == min(n, u.u1 + partition.DEFAULT_HALO) for u in plan.units)
        assert all(u.d1 - u.d0 < 2 ** 32 for u in plan.units)
    # unit-relative rows -> record coordinates, exact above 2^32
    high = [u for u in plan.units if u.d0 > 2 ** 32][:3] + [plan.units[-1]]
    idx = np.array([u.index for u in high], dtype=np.uint32)
    st = np.array([0, 1, 2 ** 20, 5], dtype=np.uint32)
    en = np.array([u.d1 - u.d0 for u in high], dtype=np.uint32)
    rec, g_st, g_en, _ = multi.unit_rows_to_records(plan.units, idx, st, en, np.ones(4, np.uint32))
    assert g_st.dtype == np.uint64 and g_en.dtype == np.uint64 and not rec.any()
    assert g_st.tolist() == [u.d0 + int(s) for u, s in zip(high, st.tolist())]
    assert g_en.tolist() == [u.d1 for u in high] and g_en[-1] == n


def test_writer_origins_above_two_to_the_32(tmp_path):
    names = ["u0", "u1", "u2", "u3"]
    text = b"acgtNNACGTACGTAC" * 8
    offsets = np.array([0, 16, 32, 48], dtype=np.uint64)
    origin = np.array([2 ** 32 - 1, 2 ** 32, 2 ** 33 + 12345, 0], dtype=np.uint64)
    rec = np.array([0, 0, 1, 2, 2, 3], dtype=np.uint32)
    st = np.array([0, 5, 3, 1, 2, 4], dtype=np.uint32)
    en = np.array([9, 2 ** 32 - 1, 12, 10, 14, 13], dtype=np.uint32)
    k = np.array([1, 3, 2, 4, 1, 3], dtype=np.uint32)
    for tsv in (False, True):
        _cabi.write_rows(str(tmp_path / "at"), names, text, offsets, rec, st, en, k, tsv=tsv, origin=origin)
        want = ["start_0based\tend\tmotif\n"] if tsv else []
        for r, s, e, kk in zip(rec.tolist(), st.tolist(), en.tolist(), k.tolist()):
            motif = text[int(offsets[r]) + s:int(offsets[r]) + s + kk].decode().upper()
            o = int(origin[r])
            want.append(("" if tsv else f"{names[r]}\t") + f"{o + s}\t{o + e}\t{motif}\n")
        assert (tmp_path / "at").read_text() == "".join(want)
        # origin = NULL (and all-zero origins) write what crf_write_rows writes, byte for byte
        _cabi.write_rows(str(tmp_path / "plain"), names, text, offsets, rec, st, en, k, tsv=tsv)
        _cabi.write_rows(str(tmp_path / "zero"), names, text, offsets, rec, st, en, k, tsv=tsv,
                         origin=np.zeros(4, np.uint64))
        assert (tmp_path / "plain").read_bytes() == (tmp_path / "zero").read_bytes()
    _cabi.write_rows(str(tmp_path / "plain"), names, text, offsets, rec, st, en, k)
    rc = _cabi.lib().crf_write_rows_at(os.fsencode(str(tmp_path / "null")), 0, 0, b"u0\0u1\0u2\0u3\0", text,
                                           offsets.ctypes.data, None, rec.ctypes.data, st.ctypes.data, en.ctypes.data,
                                           k.ctypes.data, len(rec), None)
    assert rc == _cabi.CRF_OK and (tmp_path / "null").read_bytes() == (tmp_path / "plain").read_bytes()


def test_writer_origins_under_sanitizers(tmp_path):
    """tests/fuzz_rows_at.cpp: csrc/crf_rows.h without the CUDA runtime under ASan + UBSan, on enough rows for several
    formatting threads: origin = NULL is byte-identical to crf_write_rows, origins up to 3 x (2^32 - 1) print as
    snprintf prints them."""
    if not shutil.which("g++"):
        pytest.skip("no g++")
    exe = str(tmp_path / "fuzz_rows_at")
    built = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                            "-pthread", "-I", os.path.join(ROOT, "colab-repeat-finder_b200", "csrc"),
                            "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "fuzz_rows_at.cpp"), "-o", exe],
                           capture_output=True, text=True)
    if built.returncode != 0:
        pytest.skip("sanitizer build not available here: " + built.stderr[-300:])
    run = subprocess.run([exe, str(tmp_path), "300000"], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-4000:]
    assert "ok 300000 rows" in run.stdout


# ---- on the GPU: one record of 2^32 + 150 Mbp ----------------------------------------------------------------------------

BIG = (1 << 32) + 150_000_000
T32 = 1 << 32
GPU_FS = dict(min_motif_size=1, max_motif_size=50, min_repeats=3, min_span=9)


def _plant(host, at, unit, n):
    host[at:at + n] = np.frombuffer((unit * (n // len(unit) + 1)).encode()[:n], dtype=np.uint8)


@pytest.fixture(scope="module")
def big_record():
    """The record on the host, with: repeats whose start, first mismatch or end sit at 2^32 +- (k+1), N blocks at and around
    2^32, runs straddling every load cut of the default plan (one of them 2 Mbp: longer than the 1 Mbp halo) and a run to
    the last base.  Also returns the load cuts."""
    from crf_b200 import synth
    bases, _, _ = synth.long_record(BIG, device="cuda:0")
    host = bases.cpu().numpy()
    del bases
    plan, phases = partition.plan_loads([BIG], 1, 1, _cabi.load_limit(50), chunk=partition.DEFAULT_CHUNK,
                                        halo=partition.DEFAULT_HALO, kmax=50, min_repeats=3, min_span=9)
    assert phases == 2
    cuts = [plan.units[b].u0 for b in plan.bounds[1:-1]]
    for c in cuts:
        _plant(host, c - 1_000_500, "ACG", 2_000_000)                     # longer than the halo, across the cut
        _plant(host, c + 3_000_000 - 20, "TTAGG", 45)                    # (the next unit's cut: a plain chunk boundary)
    for i, k in enumerate((1, 7, 31, 50)):
        base = T32 - 400_000 + i * 100_000
        unit = "".join("ACGT"[(j * 7 + i) % 4] for j in range(k - 1)) + "T" if k > 1 else "C"
        _plant(host, T32 - (k + 1) - i * 20_000 - 40_000, unit, 4 * k + 3)   # starts at ... - (k+1)
        _plant(host, base, unit, 5 * k)
    _plant(host, T32 - 58, "AC", 52)                                     # start 2^32 - 58, first mismatch 2^32 - (1+1) - 4
    _plant(host, T32 + 8, "CAGTACA", 3 * 7)                              # starts at 2^32 + (k+1), k = 7
    _plant(host, T32 - 3 * 50 + 51, "".join("ACGT"[(j * 5) % 4] for j in range(49)) + "A", 150)   # ends at 2^32 + 51
    host[T32 - 1000:T32 - 900] = ord("N")
    host[T32 - 1:T32 + 1] = ord("N")
    host[T32 + 300:T32 + 5000] = ord("n")
    _plant(host, BIG - 777, "GAT", 777)                                  # to the last base
    return host, cuts


@pytest.mark.gpu
def test_gpu_record_above_two_to_the_32_row_by_row(big_record, tmp_path, monkeypatch):
    """api.scan_arrays over two loads (start / end uint64) = the oracle row by row; interval mode across 2^32 with
    min_repeats 3 and 1 = the oracle with the same interval; the CLI BED of the record between two short ones = the
    oracle's rows, byte-identical with --devices 0,0 (two ranks on one GPU) and over two GPUs when there are two."""
    import torch
    host, cuts = big_record
    st, en, k = api.scan_arrays(host, 1, 50, 3, 9)
    assert st.dtype == np.uint64 and en.dtype == np.uint64
    o_s, o_e, o_m, _ = oracle.detect_repeats_by_k(host, ns(**GPU_FS), arrays=True)
    assert len(st) == len(o_s) > 8_000_000
    assert np.array_equal(st.astype(np.int64), o_s) and np.array_equal(en.astype(np.int64), o_e)
    assert np.array_equal(k.astype(np.int64), o_m.astype(np.int64))
    assert o_e[-1] == BIG and (o_s > T32).sum() > 100_000
    for c in cuts:
        assert ((o_s < c) & (o_e > c) & (o_e - o_s > partition.DEFAULT_HALO)).any()
    # interval mode across 2^32 (the probe and main scans are short here: they fit one load)
    raw = host.tobytes()
    for mr, kmin, ms in ((3, 1, 9), (1, 2, 5)):
        fs = ns(min_motif_size=kmin, max_motif_size=50, min_repeats=mr, min_span=ms,
                interval_start_0based=T32 - 200_000, interval_end=T32 + 150_000)
        want = oracle.detect_repeats(raw, fs)
        assert len(want) > 100 and api.detect_repeats(raw, fs) == want
    del raw
    # the CLI: FASTA with the record between two short ones
    rng = random.Random(9)
    shorts = [random_seq(rng, 5000), random_seq(rng, 3000)]
    fa = tmp_path / "big.fa"
    with open(fa, "wb") as f:
        f.write(b">short1\n" + shorts[0].encode() + b"\n>big desc\n")
        f.write(memoryview(host))
        f.write(b"\n>short2\n" + shorts[1].encode() + b"\n")
    lines = []
    for s0, e0, m0 in oracle.detect_repeats(shorts[0], ns(**GPU_FS)):
        lines.append(f"short1\t{s0}\t{e0}\t{m0}\n")
    upper = np.where((host >= ord("a")) & (host <= ord("z")), host - 32, host).astype(np.uint8)
    lines += [f"big\t{a}\t{b}\t{upper[a:a + m].tobytes().decode()}\n" for a, b, m in zip(o_s.tolist(), o_e.tolist(), o_m.tolist())]
    del upper
    for s0, e0, m0 in oracle.detect_repeats(shorts[1], ns(**GPU_FS)):
        lines.append(f"short2\t{s0}\t{e0}\t{m0}\n")
    want = "".join(lines).encode()
    del lines
    monkeypatch.chdir(tmp_path)
    runs = [("one", None), ("loop", "0,0")] + ([("two", "0,1")] if torch.cuda.device_count() > 1 else [])
    for name, devices in runs:
        assert cli.main([str(fa), "-o", name] + (["--devices", devices] if devices else [])) == 0
        assert (tmp_path / f"{name}.bed").read_bytes() == want, name
        os.remove(tmp_path / f"{name}.bed")


@pytest.mark.gpu
def test_gpu_patched_limit_multi_load_equals_single_load(monkeypatch):
    """A load limit patched to 64 Mbp on a 300 Mbp record: one unit per load, nine loads on one GPU, rows bit for bit those of the ordinary
    single-load scan of the same record (which the real limit allows)."""
    from crf_b200 import synth
    bases, offsets, _ = synth.generate_records([300_000_000], 77, device="cuda:0", n_satellites=40)
    host = bases.cpu().numpy()
    del bases
    with api.get_context().load(host, max_motif_cap=50) as seq:
        n = seq.scan(1, 50, 3, 9)
        _, want_s, want_e, want_k = seq.fetch(n)
    monkeypatch.setattr(_cabi, "load_limit", lambda cap: 64_000_000)
    st, en, k = api.scan_arrays(host, 1, 50, 3, 9)
    assert st.dtype == np.uint64 and len(st) == n > 500_000
    assert np.array_equal(st, want_s.astype(np.uint64)) and np.array_equal(en, want_e.astype(np.uint64))
    assert np.array_equal(k, want_k)
