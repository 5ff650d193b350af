"""Many intervals in one pass: crf_interval_stop, intervals.detect_repeats_intervals and the CLI's --intervals.

CPU tests run the host half with stand-ins (tests/fake_ctx.py: the scan is the C oracle; interval_stop is the reference's
lock-step loop run on the loaded prefix) and compare with per-interval api.detect_repeats on the same stand-ins.  The
-m gpu tests run the kernels."""
import gzip
import os
import random
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, cli, intervals, synth  # noqa: E402
from tests.fake_ctx import FakeContext, FakeSeq  # noqa: E402
from tests.helpers import load_golden, ns, random_seq  # noqa: E402


# ---- stand-ins ------------------------------------------------------------------------------------------------------

def _stop_literal(s, end_position, kmin, kmax, full_len=None):
    """prf:66-74 word for word, trackers reduced to their run length, on s = the first len(s) bases of a sequence of
    full_len bases: only t <= len(s) - 1 - kmax can be decided when the prefix is shorter (-2 past that), -1 = to the end."""
    W = len(s)
    L = W if full_len is None else full_len
    if end_position >= L - 1:
        return -1
    t_last = L - 1 if W == L else W - 1 - kmax
    run = {k: 1 for k in range(kmin, kmax + 1)}
    for t in range(t_last + 1):
        for k in run:
            if t < L - k:
                run[k] = run[k] + 1 if (s[t] == s[t + k] and s[t] != ord("N")) else 1
        if t > end_position and not any(v >= k + 1 for k, v in run.items()):
            return t
    return -1 if W == L else -2


def _runs_single_copy(s, kmin, kmax, min_span):
    """crf_scan with min_repeats == 1 as include/crf.h states it (what tests/test_host_cpu.py uses)."""
    L, arr = len(s), np.frombuffer(s, dtype=np.uint8)
    rows = []
    for k in range(kmin, min(kmax, L - 1) + 1):
        m = (arr[:L - k] == arr[k:]) & (arr[:L - k] != ord("N"))
        edge = np.diff(np.concatenate([[0], m.astype(np.int8), [0]]))
        for st, i0 in zip(np.flatnonzero(edge == 1).tolist(), np.flatnonzero(edge == -1).tolist()):
            if i0 - st >= max(min_span - k, k - 1, 1) and s[st + k - 1] != ord("N") and api._is_primitive(s[st:st + k]):
                rows.append((st, i0 + k, k))
    rows.sort()
    cols = np.array(rows, dtype=np.uint32).reshape(-1, 3)
    return cols[:, 0], cols[:, 1], cols[:, 2]


class StopSeq(FakeSeq):
    def interval_stop(self, kmin, kmax, end_pos, full_len):
        return np.array([_stop_literal(bytes(u).upper(), int(e), kmin, kmax, int(f))
                         for u, e, f in zip(self.units, end_pos, full_len)], dtype=np.int64)


class StopContext(FakeContext):
    loads = 0

    def load_packed(self, planes, offsets=None, max_motif_cap=50, ranges=None):
        from tests.fake_ctx import unpack_planes
        StopContext.loads += 1
        return StopSeq(unpack_planes(planes), *ranges)


@pytest.fixture
def stand_ins(monkeypatch):
    monkeypatch.setattr(api, "get_context", lambda device=None: StopContext())
    monkeypatch.setattr(api, "_interval_stop_position",
                        lambda ctx, s, e, kmin, kmax, knobs: (lambda t: None if t == -1 else t)(
                            _stop_literal(bytes(s).upper(), e, kmin, kmax)))
    real_scan_arrays = api.scan_arrays

    def scan_arrays(s, kmin, kmax, min_repeats, span, device=None, **kw):
        if min_repeats == 1:
            return _runs_single_copy(bytes(s).upper(), kmin, kmax, span)
        return real_scan_arrays(s, kmin, kmax, min_repeats, span, device=device, **kw)
    monkeypatch.setattr(api, "scan_arrays", scan_arrays)
    StopContext.loads = 0


def _outcome(fn):
    try:
        return fn(), None
    except (AssertionError, IndexError, ValueError, NotImplementedError) as e:
        return None, (type(e), str(e))


def _per_interval(seq, ivs, fs):
    """What detect_repeats_intervals must give: detect_repeats once per interval; the first exception, if any."""
    out = []
    for a, b in ivs:
        got, exc = _outcome(lambda: api.detect_repeats(seq, intervals._settings_for(fs, a, b)))
        if exc:
            return None, exc
        out.append(got)
    return out, None


def _seeded_intervals(rng, n, count):
    out = []
    for _ in range(count):
        kind = rng.random()
        if kind < 0.1:
            a = b = rng.randint(0, n)
        elif kind < 0.2:
            a, b = rng.randint(0, n), n                                  # touches the end
        elif kind < 0.3:
            a, b = 0, rng.randint(0, n)                                  # touches the start
        else:
            a = rng.randint(0, n)
            b = rng.randint(a, n)
        out.append((a, b))
    return out


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_vectorised_n_trim_equals_api_n_trim():
    rng = random.Random(11)
    checked = 0
    for case in range(60):
        n = rng.randint(1, 700)
        seq = random_seq(rng, n, exotic=True)
        if case % 4 == 0:
            seq = "N" * rng.randint(1, 30) + seq[:max(0, n - 60)] + "n" * rng.randint(1, 30)      # N at both ends
        raw = seq.encode()
        n = len(raw)
        planes = _cabi.pack_ascii(raw).with_runs()
        ivs = _seeded_intervals(rng, n, 90)
        nruns = [i for i in range(n) if raw[i] in b"Nn"]
        for _ in range(10):                                              # a or b inside an N block
            if nruns:
                p = rng.choice(nruns)
                ivs.append((p, rng.randint(p, n)))
                ivs.append((rng.randint(0, p), p + 1))
        ivs = [(a, b) for a, b in ivs if a < b]
        a = np.array([x for x, _ in ivs], dtype=np.int64)
        b = np.array([y for _, y in ivs], dtype=np.int64)
        a2, b2, lt = intervals.n_trim(*intervals.n_runs(planes), np.zeros_like(a), a, b, np.full_like(a, n))
        want = np.array([api._n_trim(raw, x, y) for x, y in ivs], dtype=np.int64).reshape(-1, 3)
        assert np.array_equal(np.stack([a2, b2, lt], axis=1), want), seq
        checked += len(ivs)
    assert checked >= 5000


def test_n_trim_in_a_multi_record_source():
    """Records back to back: an N run that crosses a record boundary must not carry a trim into the next record."""
    recs = [b"ACGTNNNN", b"NNNNACGTRYNN", b"N", b"ACnnGT"]
    planes = _cabi.pack_ascii(b"".join(recs)).with_runs()
    offs = np.cumsum([0] + [len(r) for r in recs])
    for r, raw in enumerate(recs):
        for a in range(len(raw)):
            for b in range(a + 1, len(raw) + 1):
                got = intervals.n_trim(*intervals.n_runs(planes), [offs[r]], [a], [b], [len(raw)])
                assert tuple(int(x[0]) for x in got) == api._n_trim(raw, a, b), (raw, a, b)


@pytest.mark.parametrize("name", ["fuzz_interval.json", "fuzz_interval_long.json", "fuzz_interval_tail.json"])
def test_batched_equals_per_interval_detect_repeats(stand_ins, name):
    rng = random.Random(name)
    n_rows = n_exc = n_single = 0
    exc_types = set()
    for case in load_golden(name):
        st = dict(case["settings"])
        golden = (st.pop("interval_start_0based"), st.pop("interval_end"))
        seq = case["seq"]
        modes = [st["min_repeats"]] + rng.sample([1, 2, 3], 1)
        for mr in modes:
            fs = ns(**{**st, "min_repeats": mr})
            ivs = [golden] + _seeded_intervals(rng, len(seq), 20)
            if rng.random() < 0.2:
                ivs.append((rng.randint(0, len(seq)), len(seq) + rng.randint(1, 5)))          # IndexError, like prf
            want, want_exc = _per_interval(seq, ivs, fs)
            got, got_exc = _outcome(lambda: intervals.detect_repeats_intervals(seq, ivs, fs))
            assert got_exc == want_exc, (name, case["settings"], mr)
            if want_exc:
                n_exc += 1
                exc_types.add(want_exc[0])
                ok = [iv for iv in ivs if _outcome(lambda: api.detect_repeats(seq, intervals._settings_for(fs, *iv)))[1] is None]
                want, _ = _per_interval(seq, ok, fs)
                got = intervals.detect_repeats_intervals(seq, ok, fs)
            assert got == want, (name, case["settings"], mr)
            n_rows += sum(len(x) for x in got)
            n_single += mr == 1
    assert n_rows > 1000 and n_exc >= 5 and n_single >= 5
    assert IndexError in exc_types


def test_satellite_across_the_interval_end_takes_several_rounds(stand_ins):
    """A 120 kbp satellite straddling the interval end: the loop only breaks where it ends, far beyond every window
    but the last few; rows must still equal the single-interval path."""
    rng = random.Random(3)
    left = random_seq(rng, 3000, alphabets=["ACGT"])
    unit = "ACGGTTCAGT"
    sat = unit * 12_000
    seq = left + sat + random_seq(rng, 2000, alphabets=["ACGT"])
    fs = ns(min_motif_size=2, max_motif_size=12, min_repeats=3, min_span=9)
    ivs = [(100, 3500), (2900, 3100), (0, 1000), (3050, 3060)]
    want, _ = _per_interval(seq, ivs, fs)
    got = intervals.detect_repeats_intervals(seq, ivs, fs)
    assert got == want
    assert intervals.last_stats["rounds"] >= 4
    assert any(e - s >= 100_000 for rows in got for s, e, _ in rows)


def _write_fasta(path, recs, gz=False):
    text = "".join(f">{n}\n" + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)) for n, s in recs)
    if gz:
        with gzip.open(path, "wt") as f:
            f.write(text)
    else:
        path.write_text(text)


def _per_line_cli(tmp_path, capsys, fa, lines, flags):
    """Concatenation of the BED files and stdout of one -i run per line."""
    bed, out = [], []
    for chrom, a, b in lines:
        assert cli.main([str(fa), *flags, "-i", f"{chrom}:{a}-{b}", "-o", str(tmp_path / "one")]) == 0
        bed.append((tmp_path / "one.bed").read_bytes())
        text = capsys.readouterr().out
        assert text.endswith("Wrote results to one.bed\n")
        out.append(text[:-len("Wrote results to one.bed\n")])
    return b"".join(bed), "".join(out)


def _glue_fasta(tmp_path, gz):
    rng = random.Random(8)
    recs = [("chrA", random_seq(rng, 3000)), ("chrB desc", random_seq(rng, 400)), ("chrC", random_seq(rng, 5000, exotic=True)),
            ("chrA", random_seq(rng, 100)), ("chrE", "N" * 50 + random_seq(rng, 700) + "n" * 40)]
    fa = tmp_path / ("glue.fa.gz" if gz else "glue.fa")
    _write_fasta(fa, recs, gz)
    lines = []
    for _ in range(40):
        name, s = rng.choice(recs)
        name = name.split()[0]
        a = rng.randint(0, len(s))
        lines.append((name, a, rng.choice([rng.randint(a, len(s)), len(s) + 100, a + rng.randint(0, 300)])))
    return fa, lines


@pytest.mark.parametrize("gz", [False, True])
def test_cli_intervals_equals_per_line_runs(tmp_path, monkeypatch, capsys, stand_ins, gz):
    monkeypatch.chdir(tmp_path)
    fa, lines = _glue_fasta(tmp_path, gz)
    flags = ["-min", "2", "-max", "12", "--min-repeats", "2", "--min-span", "8"]
    want_bed, want_out = _per_line_cli(tmp_path, capsys, fa, lines, flags)
    bed = tmp_path / "lines.bed"
    bed.write_text("# comment\ntrack name=x\nbrowser position chrA:1-2\n\n" +
                   "".join(f"{c}\t{a}\t{b}\tname{i}\t0\t+\n" for i, (c, a, b) in enumerate(lines)))
    assert cli.main([str(fa), *flags, "--intervals", str(bed), "-o", str(tmp_path / "sub" / "many")]) == 0
    assert (tmp_path / "many.bed").read_bytes() == want_bed
    assert capsys.readouterr().out == want_out + "Wrote results to many.bed\n"
    assert want_bed.count(b"\n") > 50


def test_cli_intervals_small_load_limit_groups_and_falls_back(tmp_path, monkeypatch, capsys, stand_ins):
    monkeypatch.chdir(tmp_path)
    fa, lines = _glue_fasta(tmp_path, False)
    lines.append(("chrC", 0, 5000))                                      # its prefix alone outgrows the patched limit
    flags = ["-min", "1", "-max", "9"]
    want_bed, want_out = _per_line_cli(tmp_path, capsys, fa, lines, flags)
    bed = tmp_path / "lines.bed"
    bed.write_text("".join(f"{c} {a} {b}\n" for c, a, b in lines))
    real = intervals.scan_intervals
    monkeypatch.setattr(intervals, "scan_intervals", lambda *a, **kw: real(*a[:-1], load_limit=3000))
    StopContext.loads = 0
    assert cli.main([str(fa), *flags, "--intervals", str(bed), "-o", "many"]) == 0
    assert (tmp_path / "many.bed").read_bytes() == want_bed
    assert capsys.readouterr().out == want_out + "Wrote results to many.bed\n"
    assert intervals.last_stats["too_long"] >= 1 and intervals.last_stats["loads"] >= 3


def test_cli_intervals_argument_errors(tmp_path, monkeypatch, capsys, stand_ins):
    monkeypatch.chdir(tmp_path)
    fa, _ = _glue_fasta(tmp_path, False)
    bed = tmp_path / "x.bed"
    for text, msg in (("chrA 1 10\nchrZ 1 10\n", "Chromosome chrZ not found in the input FASTA file"),
                      ("chrA 1 10\nchrA 1\n", "line 2"), ("chrA one 10\n", "line 1")):
        bed.write_text(text)
        with pytest.raises(SystemExit) as e:
            cli.main([str(fa), "--intervals", str(bed)])
        assert e.value.code == 2 and msg in capsys.readouterr().err
        assert not (tmp_path / "glue.bed").exists()
    bed.write_text("chrA 1 10\n")
    for argv in ([str(fa), "--intervals", str(bed), "-i", "chrA:1-10"], ["ACGTACGT", "--intervals", str(bed)]):
        with pytest.raises(SystemExit) as e:
            cli.main(argv)
        assert e.value.code == 2 and "--interval" in capsys.readouterr().err


# ---- GPU ------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_interval_stop_kernel_against_the_literal_loop():
    rng = random.Random(2027)
    ctx = api.get_context(0)
    n_cases = n_undecided = n_to_end = n_tail = 0
    for batch in range(8):
        kmin = rng.choice([1, 2, 3, 7, 30])
        kmax = kmin + rng.choice([0, 1, 5, 15, 49, 120, 199 - kmin])
        text, starts, W, F, E, want = [], [], [], [], [], []
        pos = 0
        for _ in range(400):
            n = rng.randint(1, 900)
            s = random_seq(rng, n, exotic=rng.random() < 0.3)
            if rng.random() < 0.5:
                unit = "".join(rng.choice("ACGT") for _ in range(rng.randint(1, kmax + 3)))
                p = rng.randint(0, len(s))
                s = s[:p] + unit * rng.randint(2, 40) + s[p:]
            raw = s.encode()
            f = len(raw)
            e = rng.choice([rng.randint(0, f), max(0, f - rng.randint(0, 2 * kmax + 2)), rng.randint(0, f // 3)])
            w = f if rng.random() < 0.6 else rng.randint(0, f)
            T = _stop_literal(raw[:w].upper(), e, kmin, kmax, f)
            if w < f:                                                  # UNDECIDED exactly when the full answer is beyond
                full = _stop_literal(raw.upper(), e, kmin, kmax)
                assert (T == -2) == (full == -1 or full > w - 1 - kmax) or e >= f - 1
                assert T == -2 or T == full
            text.append(raw)
            starts.append(pos)
            pos += f
            W.append(w)
            F.append(f)
            E.append(e)
            want.append(T)
            n_undecided += T == -2
            n_to_end += T == -1 and e < f - 1
            n_tail += f - 2 * kmax <= e < f - 1
        planes = _cabi.pack_ascii(b"".join(text)).with_runs()
        with ctx.load_packed(planes, max_motif_cap=kmax, ranges=(starts, W, None, None)) as seq:
            got = seq.interval_stop(kmin, kmax, E, F)
        bad = [(i, text[i], W[i], E[i], int(got[i]), want[i]) for i in range(len(want)) if got[i] != want[i]]
        assert not bad, (kmin, kmax, bad[:3])
        n_cases += len(want)
    assert n_cases >= 3000 and n_undecided > 50 and n_to_end > 50 and n_tail > 50
    with ctx.load_packed(_cabi.pack_ascii(b"ACGTACGT").with_runs(), max_motif_cap=4, ranges=([0], [8], None, None)) as seq:
        with pytest.raises(ValueError):
            seq.interval_stop(1, 4, [0], [7])                            # loaded prefix longer than the sequence
        with pytest.raises(ValueError):
            seq.interval_stop(1, 5, [0], [8])                            # above max_motif_cap


@pytest.mark.gpu
def test_detect_repeats_intervals_against_the_oracle():
    from oracle import oracle
    rng = random.Random(44)
    n_rows = 0
    for case in range(12):
        n = rng.choice([500, 5000, 70_000])
        seq = random_seq(rng, n, exotic=case % 3 == 0)
        kmin = rng.choice([1, 2, 4])
        fs = ns(min_motif_size=kmin, max_motif_size=kmin + rng.choice([5, 30, 49]), min_repeats=rng.choice([2, 3, 4]),
                min_span=rng.choice([1, 9, 20]))
        ivs = [iv for iv in _seeded_intervals(rng, n, 80) if iv[1] < n or iv[0] > 0]
        want = []
        for a, b in ivs:
            try:
                want.append(oracle.detect_repeats(seq, intervals._settings_for(fs, a, b)))
            except AssertionError:
                want.append(None)
        ok = [iv for iv, w in zip(ivs, want) if w is not None]
        got = intervals.detect_repeats_intervals(seq, ok, fs, device=0)
        assert got == [w for w in want if w is not None], (case, fs)
        assert len(ok) >= 50
        n_rows += sum(len(x) for x in got)
    assert n_rows > 2000


@pytest.mark.gpu
def test_cli_intervals_reference_vectors_in_one_load(tmp_path, monkeypatch, capsys):
    """The reference-generated interval cases, grouped by filter settings, as one multi-record FASTA + BED each."""
    monkeypatch.chdir(tmp_path)
    groups = {}
    for name in ("fuzz_interval.json", "fuzz_interval_long.json", "fuzz_interval_tail.json"):
        for case in load_golden(name):
            st = dict(case["settings"])
            if "raises" in case or st["min_repeats"] == 1:
                continue
            a, b = st.pop("interval_start_0based"), st.pop("interval_end")
            groups.setdefault(tuple(sorted(st.items())), []).append((case["seq"], a, b, case["result"]))
    n_checked = 0
    for gi, (key, cases) in enumerate(groups.items()):
        st = dict(key)
        fa = tmp_path / f"g{gi}.fa"
        _write_fasta(fa, [(f"r{i}", c[0]) for i, c in enumerate(cases)])
        bed = tmp_path / f"g{gi}.bed.txt"
        bed.write_text("".join(f"r{i}\t{c[1]}\t{c[2]}\n" for i, c in enumerate(cases)))
        flags = ["-min", str(st["min_motif_size"]), "-max", str(st["max_motif_size"]), "--min-repeats",
                 str(st["min_repeats"]), "--min-span", str(st["min_span"])]
        assert cli.main([str(fa), *flags, "--intervals", str(bed), "-o", f"out{gi}"]) == 0
        capsys.readouterr()
        want = "".join(f"r{i}\t{s}\t{e}\t{m}\n" for i, c in enumerate(cases) for s, e, m in c[3])
        assert (tmp_path / f"out{gi}.bed").read_text() == want, key
        n_single = sum(c[1] >= min(c[2], len(c[0])) for c in cases)         # a >= b: the single-interval path
        st = intervals.last_stats                                            # one load per window round
        assert st["loads"] == st["rounds"] and st["fallback"] == n_single
        n_checked += len(cases)
    assert n_checked > 600


@pytest.mark.gpu
def test_cli_intervals_500kb_tiling_of_s22(tmp_path, monkeypatch, capsys):
    """What the Hail pipeline does with --interval per 500 kb tile (before its sort | uniq), in one run.  The per-tile
    BED lines are made by api.detect_repeats on the record, which is all the -i path does with a line."""
    monkeypatch.chdir(tmp_path)
    bases, _, _ = synth.s22(device="cuda:0")
    raw = bases.cpu().numpy().tobytes()
    del bases
    fa = tmp_path / "s22.fa"
    with open(fa, "wb") as f:
        f.write(b">chr22\n" + b"".join(raw[i:i + 60] + b"\n" for i in range(0, len(raw), 60)))
    tiles = [(a, min(a + 500_000, len(raw))) for a in range(0, len(raw), 500_000)]
    fs = ns(min_motif_size=1, max_motif_size=6, min_repeats=3, min_span=9)
    per_tile = ["".join(f"chr22\t{s}\t{e}\t{m}\n" for s, e, m in api.detect_repeats(raw, intervals._settings_for(fs, a, b), device=0))
                for a, b in tiles]
    want = "".join(per_tile)
    bed = tmp_path / "tiles.bed.txt"
    bed.write_text("".join(f"chr22\t{a}\t{b}\n" for a, b in tiles))
    assert cli.main([str(fa), "-min", "1", "-max", "6", "--intervals", str(bed), "-o", "tiles"]) == 0
    assert (tmp_path / "tiles.bed").read_text() == want
    out = capsys.readouterr().out
    assert out.count("Processing chr22 (500,000 bp)\n") == len(tiles) - 1 and out.endswith("Wrote results to tiles.bed\n")
    assert len(tiles) > 100 and want.count("\n") > 40_000
    # the command line itself, one -i run per tile, on a seeded sample of the tiles (the leading N block and the last,
    # shorter tile included)
    sample = sorted({0, 21, len(tiles) - 1} | set(random.Random(22).sample(range(len(tiles)), 5)))
    lines = out.splitlines(keepends=True)
    for t in sample:
        a, b = tiles[t]
        assert cli.main([str(fa), "-min", "1", "-max", "6", "-i", f"chr22:{a}-{b}", "-o", "one"]) == 0
        assert (tmp_path / "one.bed").read_text() == per_tile[t], tiles[t]
        assert capsys.readouterr().out == "".join(lines[2 * t:2 * t + 2]) + "Wrote results to one.bed\n"


@pytest.mark.gpu
def test_interval_above_2_32_on_a_long_record(tmp_path, monkeypatch, capsys):
    """One interval 2^32 + 12 kbp into a record (synth.long_record salts every 2^32-block, so a position read 2^32 off
    is caught): rows = the oracle on that slice (the loop breaks long before the slice ends), printed + 2^32.  Then the
    whole record as a second line: its prefix outgrows one load, so it goes through the single-interval path, and its rows
    run past 2^32; the BED file and stdout must equal those of the two -i runs."""
    from oracle import oracle
    monkeypatch.chdir(tmp_path)
    n = (1 << 32) + 2_000_000
    bases, _, _ = synth.long_record(n, device="cuda:0")
    raw = bases.cpu().numpy()
    del bases
    a, b = (1 << 32) + 12_345, (1 << 32) + 212_345
    fs = ns(min_motif_size=1, max_motif_size=20, min_repeats=3, min_span=9)
    sl = raw[a:a + 400_000].tobytes()
    want = [(s + a, e + a, m) for s, e, m in oracle.detect_repeats(sl, intervals._settings_for(fs, 0, b - a))]
    fa = tmp_path / "long.fa"
    with open(fa, "wb") as f:
        f.write(b">big\n")
        for i in range(0, len(raw), 1 << 26):
            f.write(memoryview(raw[i:i + (1 << 26)]))
            f.write(b"\n")
    del raw
    bed = tmp_path / "one.bed.txt"
    bed.write_text(f"big\t{a}\t{b}\n")
    assert cli.main([str(fa), "-max", "20", "--intervals", str(bed), "-o", "long"]) == 0
    got = (tmp_path / "long.bed").read_text()
    assert got == "".join(f"big\t{s}\t{e}\t{m}\n" for s, e, m in want) and len(want) > 100
    capsys.readouterr()
    bed.write_text(f"big\t{a}\t{b}\nbig\t0\t{n}\n")
    want_bed, want_out = b"", ""
    for lo, hi in ((a, b), (0, n)):
        assert cli.main([str(fa), "-max", "20", "-i", f"big:{lo}-{hi}", "-o", "one"]) == 0
        want_bed += (tmp_path / "one.bed").read_bytes()
        want_out += capsys.readouterr().out.replace("Wrote results to one.bed\n", "")
    assert cli.main([str(fa), "-max", "20", "--intervals", str(bed), "-o", "long"]) == 0
    assert intervals.last_stats["too_long"] == 1 and intervals.last_stats["fallback"] == 1
    got = (tmp_path / "long.bed").read_bytes()
    assert got == want_bed
    assert capsys.readouterr().out == want_out + "Wrote results to long.bed\n"
    tail = [int(x.split(b"\t")[1]) for x in got.splitlines()[-1000:]]
    assert min(tail) >= 1 << 32                                            # rows written above 2^32
