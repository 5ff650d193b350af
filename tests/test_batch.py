"""Many sequences in one pass: batch.detect_repeats_batch and batch.scan_batch.

CPU tests run the host half with the stand-ins of tests/test_intervals.py (the scan is the C oracle, crf_interval_stop the
reference's lock-step loop on the loaded prefix, min_repeats == 1 the closed form crf_scan documents) and compare with one
api.detect_repeats call per sequence on the same stand-ins.  The -m gpu tests run the kernels."""
import os
import random
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, batch, intervals, synth  # noqa: E402
from tests.fake_ctx import FakeContext  # noqa: E402
from tests.helpers import load_golden, ns, random_seq  # noqa: E402
from tests.test_intervals import StopContext, stand_ins  # noqa: E402,F401 (stand_ins: fixture)

EXC = (AssertionError, IndexError, ValueError, NotImplementedError, AttributeError)


class BatchContext(StopContext):
    """StopContext (ranged loads of interval prefixes) plus the whole-record loads of full mode."""

    def load_packed(self, planes, offsets=None, max_motif_cap=50, ranges=None):
        if ranges is not None:
            return super().load_packed(planes, offsets, max_motif_cap, ranges)
        StopContext.loads += 1
        return FakeContext.load_packed(self, planes, offsets, max_motif_cap)


@pytest.fixture
def batch_stand_ins(stand_ins, monkeypatch):  # noqa: F811
    monkeypatch.setattr(api, "get_context", lambda device=None: BatchContext())


def _outcome(fn):
    try:
        return fn(), None
    except EXC as e:
        return None, (type(e), str(e))


def _loop(seqs, fs):
    """What detect_repeats_batch must give: detect_repeats once per sequence; the first exception, if any."""
    out = []
    for s in seqs:
        got, exc = _outcome(lambda: api.detect_repeats(s, fs))
        if exc:
            return None, exc
        out.append(got)
    return out, None


def _check(seqs, fs):
    """batch == loop on seqs, then on the sequences that do not raise alone.  Returns (rows, raised)."""
    want = _loop(seqs, fs)
    assert _outcome(lambda: batch.detect_repeats_batch(seqs, fs)) == want, fs
    if want[1] is None:
        return sum(len(x) for x in want[0]), False
    ok = [s for s in seqs if _outcome(lambda: api.detect_repeats(s, fs))[1] is None]
    want_ok, _ = _loop(ok, fs)
    assert batch.detect_repeats_batch(iter(ok), fs) == want_ok, fs
    return sum(len(x) for x in want_ok), True


# ---- CPU ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["kat.json", "fuzz_full.json", "fuzz_interval.json", "fuzz_interval_long.json",
                                  "fuzz_interval_tail.json", "fuzz_minrep1.json"])
def test_batch_equals_per_sequence_detect_repeats_on_the_golden_vectors(batch_stand_ins, name):
    """Every sequence of the file in one batch (every third one as bytes), under settings taken from the file's cases,
    each in its own min_repeats mode and one other."""
    rng = random.Random(name)
    cases = load_golden(name)
    seqs = [c["seq"].encode() if i % 3 == 1 else c["seq"] for i, c in enumerate(cases)]
    n_rows = n_raised = n_batched = 0
    for case in rng.sample(cases, min(len(cases), 5)):
        own = case["settings"]["min_repeats"]
        for mr in [own] + rng.sample([m for m in (1, 2, 3) if m != own], 1):
            fs = ns(**{**case["settings"], "min_repeats": mr})
            rows, raised = _check(seqs, fs)
            n_rows += rows
            n_raised += raised
            n_batched += mr > 1 and batch.last_stats["fallback"] < len(seqs)
    assert n_rows > 100 and n_batched >= 3
    if "interval" in name:
        assert n_raised >= 3                             # interval_end beyond most of the file's sequences: IndexError


def _odd_sequences(rng):
    return ["ACGTACGTACGTACGTTTTTTTTTTTTG", b"acgtacgtACGTacgtnnnnAAAAAAAAAAAAaaaaaaa", "", b"", "N" * 40, b"n" * 7,
            "RYRYRYRYRYRYKMKMKMKMKMKM" + "ACG" * 9, b"WWWWWWWWWWSSSSSSSSSSBDHVBDHVBDHV",
            "ACGT" + "é" * 12 + "acgacgacgacgACG",             # latin-1 beyond ASCII: upper-cased on the host
            random_seq(rng, 3000, exotic=True), random_seq(rng, 400).encode(), "a" * 30 + "N" + "a" * 30, "T"]


def test_batch_mixed_input(batch_stand_ins):
    """str and bytes, lower case, IUPAC and latin-1 letters, empty and all-N sequences; full and interval mode, all
    min_repeats modes.  A non-latin-1 string raises NotImplementedError as detect_repeats does (first raising sequence)."""
    rng = random.Random(5)
    seqs = _odd_sequences(rng)
    n_rows = 0
    for mr in (1, 2, 3):
        base = dict(min_motif_size=1, max_motif_size=12, min_repeats=mr, min_span=9 if mr > 1 else 5)
        for extra in ({}, {"interval_start_0based": 2}, {"interval_start_0based": 0, "interval_end": 1}, {"interval_end": 0}):
            rows, raised = _check(seqs, ns(**base, **extra))
            n_rows += rows
            for bad in ("ACGTĀĀĀ", "straße"):          # outside latin-1 / upper case grows
                got = _outcome(lambda: batch.detect_repeats_batch(seqs + [bad] + seqs, ns(**base, **extra)))
                assert got == _loop(seqs + [bad] + seqs, ns(**base, **extra))
                assert raised or got[1][0] is NotImplementedError
    assert n_rows > 100
    assert batch.detect_repeats_batch([], ns(min_motif_size=0)) == []              # the loop never reads the settings
    with pytest.raises(ValueError, match="min_motif_size"):
        batch.detect_repeats_batch(["ACGT"], ns(min_motif_size=0, max_motif_size=3, min_repeats=2, min_span=1))


def test_first_raising_sequence_wins(batch_stand_ins):
    fs = ns(min_motif_size=1, max_motif_size=6, min_repeats=2, min_span=4, interval_start_0based=0, interval_end=50)
    long_ = "ACG" * 40
    cases = [
        ([long_, long_, "ACGT" * 5, long_, "ACĀ", "A" * 10], IndexError),       # b > len: IndexError, before the bad text
        ([long_, "ACĀ", "ACGT" * 5], NotImplementedError),                      # bad text before the short sequence
        ([long_, "", long_], IndexError),
    ]
    for seqs, exc in cases:
        want = _loop(seqs, fs)
        assert want[1][0] is exc
        assert _outcome(lambda: batch.detect_repeats_batch(seqs, fs)) == want
    # prf:77-78: interval_end equals the length of the trimmed string, but the loop breaks before its end; that
    # AssertionError comes before a later sequence's IndexError, and after an earlier one's
    fs = ns(min_motif_size=1, max_motif_size=3, min_repeats=2, min_span=4, interval_start_0based=5, interval_end=25)
    asserting = "ACGTTGCAACGTAGCTAGGATCCATGCAAT"
    assert _loop([asserting], fs)[1][0] is AssertionError
    for seqs in ([long_, asserting, "ACG"], ["ACG", asserting, long_]):
        assert _outcome(lambda: batch.detect_repeats_batch(seqs, fs)) == _loop(seqs, fs)


def test_small_load_limit_groups_and_falls_back(batch_stand_ins, monkeypatch):
    rng = random.Random(17)
    seqs = [random_seq(rng, rng.choice([0, rng.randint(1, 300), rng.randint(300, 1500)])) for _ in range(40)]
    seqs[23] = random_seq(rng, 5000)                      # alone longer than one (patched) load
    monkeypatch.setattr(batch, "_load_limit", lambda kmax: 3000)
    fs = ns(min_motif_size=1, max_motif_size=9, min_repeats=3, min_span=9)
    want, _ = _loop(seqs, fs)
    StopContext.loads = 0
    assert batch.detect_repeats_batch(seqs, fs) == want and sum(len(x) for x in want) > 50
    assert batch.last_stats["fallback"] == 1 and batch.last_stats["loads"] >= 5
    assert StopContext.loads == batch.last_stats["loads"]
    # interval mode: the long sequence's prefix outgrows the load too
    fs_iv = ns(min_motif_size=1, max_motif_size=9, min_repeats=3, min_span=9, interval_start_0based=0)
    want, _ = _loop(seqs, fs_iv)
    assert batch.detect_repeats_batch(seqs, fs_iv) == want
    assert batch.last_stats["fallback"] >= 1 and batch.last_stats["loads"] >= 5
    # scan_batch itself refuses the long record and points to detect_repeats_batch
    blob = "".join(seqs).encode()
    offsets = np.concatenate([[0], np.cumsum([len(s) for s in seqs])])
    with pytest.raises(NotImplementedError, match="record 23 .*detect_repeats_batch"):
        batch.scan_batch(blob, offsets, fs)


def test_scan_batch_columns(batch_stand_ins):
    """Host input: the columns are the per-record rows of detect_repeats, sorted by (record, start, end); offsets may
    start past 0 and be any integer array; refusals and malformed input."""
    rng = random.Random(23)
    recs = [random_seq(rng, rng.randint(0, 900), exotic=True).encode() for _ in range(60)]
    text = b"xx" + b"".join(recs)
    offsets = 2 + np.concatenate([[0], np.cumsum([len(r) for r in recs])]).astype(np.uint64)
    fs = ns(min_motif_size=2, max_motif_size=15, min_repeats=2, min_span=6)
    want = [(i, s, e, len(m)) for i, r in enumerate(recs) for s, e, m in api.detect_repeats(r, fs)]
    for bases in (text, bytearray(text), np.frombuffer(text, dtype=np.uint8)):
        cols = batch.scan_batch(bases, offsets, fs)
        assert all(isinstance(c, np.ndarray) and c.dtype == np.uint32 for c in cols)
        assert list(zip(*(c.tolist() for c in cols))) == want and len(want) > 100
    assert all(c.size == 0 for c in batch.scan_batch(b"", [0], fs))
    assert all(c.size == 0 for c in batch.scan_batch(b"ACGT", [0, 0, 0], fs))
    for bad_fs in (ns(**vars(fs), interval_end=100), ns(**{**vars(fs), "min_repeats": 1})):
        with pytest.raises(NotImplementedError, match="detect_repeats_batch"):
            batch.scan_batch(text, offsets, bad_fs)
    for bad in ([[0, 4]], [3, 2], [0, len(text) + 1], [-1, 3], [], [0.0, 2.0]):
        with pytest.raises(ValueError):
            batch.scan_batch(text, bad, fs)


# ---- GPU ------------------------------------------------------------------------------------------------------------

DEFAULTS = dict(min_motif_size=1, max_motif_size=50, min_repeats=3, min_span=9)


def _planted(rng, n):
    """A sequence of n symbols with repeats of every kind planted in it (mixed case, N runs, IUPAC letters)."""
    s = list(random_seq(rng, n, exotic=True))
    for _ in range(max(1, n // 2000)):
        unit = "".join(rng.choice("ACGT") for _ in range(rng.randint(1, 50)))
        rep = (unit * (rng.randint(60, 2000) // len(unit) + 2))
        p = rng.randint(0, n)
        s[p:p + len(rep)] = rep
    return "".join(s)[:n]


@pytest.mark.gpu
def test_batch_of_reads_and_of_long_sequences_against_the_oracle():
    from oracle import oracle
    n_reads = 100_000
    bases, offsets, _ = synth.sr(n_reads)
    reads = [bases[int(offsets[i]):int(offsets[i + 1])].tobytes() for i in range(n_reads)]
    reads = [r.decode() if i % 2 else r for i, r in enumerate(reads)]
    fs = ns(**{**DEFAULTS, "max_motif_size": 20})
    got = batch.detect_repeats_batch(reads, fs, device=0)
    assert batch.last_stats == {"loads": 1, "fallback": 0}
    want = [oracle.detect_repeats(r, fs) for r in reads]
    assert got == want and sum(map(len, got)) > 10_000
    rng = random.Random(70)
    seqs = [_planted(rng, rng.choice([rng.randint(1, 5000), rng.randint(5000, 70_000)])) for _ in range(300)]
    seqs = [s.encode() if i % 3 == 0 else s for i, s in enumerate(seqs)]
    got = batch.detect_repeats_batch(seqs, ns(**DEFAULTS), device=0)
    want = [oracle.detect_repeats_by_k(s, ns(**DEFAULTS)) for s in seqs]
    assert got == want and sum(map(len, got)) > 20_000


@pytest.mark.gpu
def test_batch_with_interval_attributes_equals_detect_repeats():
    """Every sequence is an interval of itself; in some of them the interval ends inside a satellite of tens of kbp, so the
    stop position is found only after several window rounds."""
    rng = random.Random(71)
    seqs = []
    for i in range(200):
        s = _planted(rng, rng.randint(3000, 20_000))
        if i % 4 == 0:
            unit = "".join(rng.choice("ACGT") for _ in range(rng.randint(2, 12)))
            s = s[:2500] + unit * (rng.randint(5_000, 60_000) // len(unit)) + s[2500:]
        seqs.append(s if i % 2 else s.encode())
    for extra in ({"interval_start_0based": 100, "interval_end": 2900}, {"interval_start_0based": 1000},
                  {"interval_end": 2600}):
        fs = ns(**{**DEFAULTS, "max_motif_size": 20}, **extra)
        want = [api.detect_repeats(s, fs, device=0) for s in seqs]
        assert batch.detect_repeats_batch(seqs, fs, device=0) == want, extra
        assert batch.last_stats["fallback"] == 0
        if extra.get("interval_end") == 2900:
            assert intervals.last_stats["rounds"] >= 4 and sum(map(len, want)) > 2_000


@pytest.mark.gpu
def test_scan_batch_ten_million_reads_from_host_and_from_a_tensor():
    """Config C5: 10 M reads x 150 bp, motif 1-20.  From host bytes: the oracle's rows, checked the way
    test_all_ten_million_reads_row_by_row checks them (the reads as one string with max_motif_size N's between them); from
    the CUDA tensor: bit-identical columns, on the device."""
    import torch
    from oracle import oracle
    n_reads, rl, gap = 10_000_000, 150, 20
    bases, offsets, _ = synth.sr(n_reads, device="cuda:0")
    host = bases.cpu().numpy()
    fs = ns(**{**DEFAULTS, "max_motif_size": 20})
    rec, st, en, k = batch.scan_batch(host.tobytes(), offsets, fs, device=0)
    assert batch.last_stats["loads"] == 1 and rec.size > 500_000
    gapped = np.full((n_reads, rl + gap), ord("N"), dtype=np.uint8)
    gapped[:, :rl] = host.reshape(n_reads, rl)
    o_s, o_e, o_m, _ = oracle.detect_repeats_by_k(gapped.reshape(-1), fs, arrays=True)
    del gapped
    o_rec = o_s // (rl + gap)
    assert np.array_equal(rec.astype(np.int64), o_rec)
    assert np.array_equal(st.astype(np.int64), o_s - o_rec * (rl + gap))
    assert np.array_equal(en.astype(np.int64), o_e - o_rec * (rl + gap))
    assert np.array_equal(k.astype(np.int64), o_m.astype(np.int64))
    torch.cuda.synchronize()
    dev = batch.scan_batch(bases, torch.from_numpy(offsets.astype(np.int64)), fs)
    assert all(t.is_cuda and t.dtype == torch.uint32 for t in dev)
    for t, h in zip(dev, (rec, st, en, k)):
        assert np.array_equal(t.cpu().numpy(), h)
    # bases written on torch's stream just before the call: the load must see them
    shifted = torch.roll(bases, 75)
    want = batch.scan_batch(shifted.cpu().numpy(), offsets, fs)
    shifted = torch.roll(bases, 75)
    got = batch.scan_batch(shifted, offsets, fs, device=0)
    assert all(np.array_equal(t.cpu().numpy(), h) for t, h in zip(got, want))


@pytest.mark.gpu
def test_several_loads_and_the_fallback_on_the_gpu(monkeypatch):
    """A patched load limit: several groups (rows mapped to the batch's record numbers by crf_seq_set_output_map), host and
    tensor input alike, and one sequence above the limit through api.detect_repeats."""
    import torch
    rng = random.Random(72)
    seqs = [_planted(rng, rng.randint(0, 20_000)) for _ in range(120)]
    seqs[50] = _planted(rng, 150_000)
    monkeypatch.setattr(batch, "_load_limit", lambda kmax: 100_000)
    fs = ns(**DEFAULTS)
    want = [api.detect_repeats(s, fs, device=0) for s in seqs]
    assert batch.detect_repeats_batch(seqs, fs, device=0) == want
    assert batch.last_stats["fallback"] == 1 and batch.last_stats["loads"] >= 10
    fit = seqs[:50] + seqs[51:]
    blob = "".join(fit).encode()
    offsets = np.concatenate([[0], np.cumsum([len(s) for s in fit])])
    host = batch.scan_batch(blob, offsets, fs, device=0)
    assert batch.last_stats["loads"] >= 10
    assert list(zip(*(c.tolist() for c in host))) == [(i, s, e, len(m)) for i, f in enumerate(fit)
                                                      for s, e, m in api.detect_repeats(f, fs, device=0)]
    dev = batch.scan_batch(torch.frombuffer(bytearray(blob), dtype=torch.uint8).to("cuda:0"), offsets, fs)
    assert all(np.array_equal(t.cpu().numpy(), h) for t, h in zip(dev, host))
    with pytest.raises(NotImplementedError, match="detect_repeats_batch"):
        batch.scan_batch("".join(seqs).encode(), np.concatenate([[0], np.cumsum([len(s) for s in seqs])]), fs, device=0)
    assert _cabi.load_limit(50) > 4_000_000_000                                   # the library's own limit is untouched
