"""Per-base repeat masks: crf_mask_rows, the masked FASTA writer, mask.repeat_mask and the CLI's --mask.

The mask of a record is the union of the rows detect_repeats gives for it (mask[p] = 1 iff some row has s <= p < e).  CPU
tests check the writer against a Python statement of the format, the writer under sanitizers, and the CLI glue with the
scan and crf_mask_rows replaced by stand-ins (the oracle, numpy).  The -m gpu tests run the kernels."""
import os
import random
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, batch, cli, mask, synth  # noqa: E402
from oracle import oracle  # noqa: E402
from tests.fake_ctx import FakeContext  # noqa: E402
from tests.helpers import ns, random_seq  # noqa: E402


def union(n, start, end):
    """bool[n]: the union of the ranges [start[i], end[i])."""
    d = np.zeros(n + 1, np.int64)
    np.add.at(d, np.asarray(start, np.int64), 1)
    np.add.at(d, np.asarray(end, np.int64), -1)
    return np.cumsum(d[:-1]) > 0


def words_of(bits):
    """bool mask -> uint32 words, bit p & 31 of word p >> 5 (the layout of crf_mask_rows)."""
    packed = np.packbits(np.asarray(bits, bool), bitorder="little")
    packed = np.concatenate([packed, np.zeros(-packed.size % 4, np.uint8)])
    return packed.view(np.uint32)


def masked_fasta(names, records, masks, hard, width=60):
    """The masked FASTA format, stated one base at a time."""
    out = []
    for name, rec, m in zip(names, records, masks):
        out.append(b">" + name + b"\n")
        line = bytearray()
        for c, x in zip(rec, m):
            if x:
                c = ord("N") if hard else c + 32 if ord("A") <= c <= ord("Z") else c
            line.append(c)
            if len(line) == width:
                out.append(bytes(line) + b"\n")
                line = bytearray()
        if line:
            out.append(bytes(line) + b"\n")
    return b"".join(out)


def write_fasta(path, records, width=60):
    path.write_bytes(b"".join(b">" + n + b"\n" + b"".join(s[i:i + width] + b"\n" for i in range(0, len(s), width))
                              for n, s in records))


# ---- CPU: the writer ------------------------------------------------------------------------------------------------

def _writer_case(tmp_path, names, records, masks, hard, width, lead=b""):
    blob = lead + b"".join(records)
    offsets = len(lead) + np.concatenate([[0], np.cumsum([len(r) for r in records])]).astype(np.uint64)
    bits = np.concatenate([np.zeros(len(lead), bool)] + [np.asarray(m, bool) for m in masks])
    path = tmp_path / "out.fa"
    n = _cabi.write_fasta_masked(str(path), names, np.frombuffer(blob, np.uint8) if blob else b"", offsets, words_of(bits),
                                 hard=hard, line_width=width)
    want = masked_fasta([x.encode() for x in names], records, masks, hard, width)
    assert path.read_bytes() == want and n == len(want), (hard, width)


@pytest.mark.parametrize("hard", [False, True])
def test_writer_matches_the_format(tmp_path, hard):
    """Lower-case input, IUPAC letters and other bytes, empty records, line widths that do and do not divide the record
    lengths, records that start inside a mask word, and bases before the first record."""
    rng = random.Random(3)
    records = [random_seq(rng, 120, alphabets=["ACGTacgtNn"]).encode(), b"", b"ACGTRYKMSWBDHVNacgtrykm-*.\xe9" * 7,
               random_seq(rng, 61).encode(), b"", b"", b"A", random_seq(rng, 1000, exotic=True).encode(), b""]
    names = [f"r{i}" if i % 2 else f"record_{i}" for i in range(len(records))]
    for width in (60, 1, 7, 120, 1000, 1001):
        masks = [np.array([rng.random() < 0.4 for _ in r], bool) for r in records]
        _writer_case(tmp_path, names, records, masks, hard, width)
        _writer_case(tmp_path, names, records, masks, hard, width, lead=b"xyz")
        _writer_case(tmp_path, names, records, [np.ones(len(r), bool) for r in records], hard, width)
    _writer_case(tmp_path, ["e1", "e2"], [b"", b""], [[], []], hard, 60)
    _writer_case(tmp_path, [], [], [], hard, 60)


def test_writer_on_many_records_and_threads(tmp_path):
    """10^5 records (15 Mbp: the writer formats slices of 2^20 bases on several threads) against the Python statement."""
    n_rec, rl = 100_000, 150
    rng = np.random.default_rng(5)
    blob = np.frombuffer(b"ACGTacgtNR", np.uint8)[rng.integers(0, 10, n_rec * rl)]
    bits = rng.random(n_rec * rl) < 0.3
    offsets = np.arange(0, n_rec * rl + 1, rl, dtype=np.uint64)
    names = [f"read{i}" for i in range(n_rec)]
    for hard in (False, True):
        path = tmp_path / "reads.fa"
        _cabi.write_fasta_masked(str(path), names, blob, offsets, words_of(bits), hard=hard)
        text = blob.copy()
        if hard:
            text[bits] = ord("N")
        else:
            up = bits & (text >= ord("A")) & (text <= ord("Z"))
            text[up] += 32
        body = np.full((n_rec, rl + 3), ord("\n"), np.uint8)          # 150 bp at 60 per line: 60 + 60 + 30, 3 line breaks
        rows = text.reshape(n_rec, rl)
        body[:, 0:60], body[:, 61:121], body[:, 122:152] = rows[:, :60], rows[:, 60:120], rows[:, 120:]
        want = b"".join(f">read{i}\n".encode() + body[i].tobytes() for i in range(n_rec))
        assert path.read_bytes() == want


def test_writer_refusals(tmp_path):
    offsets = np.array([0, 4], np.uint64)
    with pytest.raises(ValueError):
        _cabi.write_fasta_masked(str(tmp_path / "x.fa"), ["a"], b"ACGT", offsets, np.zeros(1, np.uint32), line_width=0)
    with pytest.raises(ValueError):
        _cabi.write_fasta_masked(str(tmp_path / "x.fa"), ["a"], b"ACGT", np.array([0, 5], np.uint64), np.zeros(1, np.uint32))
    with pytest.raises(ValueError):
        _cabi.write_fasta_masked(str(tmp_path / "no" / "dir.fa"), ["a"], b"ACGT", offsets, np.zeros(1, np.uint32))
    if os.path.exists("/dev/full"):                                         # a short write is an error, not a shorter file
        with pytest.raises(OSError, match="failed"):
            _cabi.write_fasta_masked("/dev/full", ["a"], b"ACGT" * 50_000, np.array([0, 200_000], np.uint64),
                                     np.zeros(6250, np.uint32))


def test_mask_writer_under_sanitizers(tmp_path):
    """tests/fuzz_mask_writer.cpp: csrc/crf_fasta_out.h without the CUDA runtime under ASan + UBSan."""
    if not shutil.which("g++"):
        pytest.skip("no g++")
    exe = str(tmp_path / "fuzz_mask_writer")
    built = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                            "-pthread", "-I", os.path.join(ROOT, "colab-repeat-finder_b200", "csrc"),
                            "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "fuzz_mask_writer.cpp"), "-o", exe],
                           capture_output=True, text=True)
    if built.returncode != 0:
        pytest.skip("sanitizer build not available here: " + built.stderr[-300:])
    run = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-4000:]
    assert "ok 48 files" in run.stdout


# ---- CPU: the command line with stand-ins -----------------------------------------------------------------------------

class MaskContext(FakeContext):
    """FakeContext (the oracle as scan) with crf_mask_rows in numpy."""

    def mask_rows(self, record, start, end, dst_offset, mask_bits, n_rows=None, mask=None):
        record, start, end = (np.asarray(a, np.int64) for a in (record, start, end))
        dst = np.asarray(dst_offset, np.uint64).astype(np.int64)
        assert (end >= start).all() and (record < dst.size).all() and (dst[record] + end <= mask_bits).all()
        return words_of(union(int(mask_bits), dst[record] + start, dst[record] + end))


def mask_from_bed(bed_text, names, records):
    """Per record, the union of the BED rows written for it."""
    rows = {}
    for line in bed_text.splitlines():
        c, s, e, _ = line.split("\t")
        rows.setdefault(c, []).append((int(s), int(e)))
    return [union(len(r), [a for a, _ in rows.get(n, [])], [b for _, b in rows.get(n, [])]) for n, r in zip(names, records)]


def _glue_records(rng):
    return [(b"chrA", random_seq(rng, 3000).encode()), (b"chrB", random_seq(rng, 50).encode()), (b"empty", b""),
            (b"chrC", random_seq(rng, 7000, exotic=True).encode()), (b"chrD", (b"acgt" * 30 + b"AC" * 40) * 9)]


def _check_cli_mask(tmp_path, capsys, records, argv, kind):
    assert cli.main(argv + ["--mask", kind]) == 0
    names = [n for n, _ in records]
    masks = mask_from_bed((tmp_path / "out.bed").read_text(), [n.decode() for n in names], [s for _, s in records])
    assert (tmp_path / "out.masked.fa").read_bytes() == masked_fasta(names, [s for _, s in records], masks, kind == "hard")
    out = capsys.readouterr().out
    assert out.endswith("Wrote results to out.bed\nWrote masked sequence to out.masked.fa\n")
    return sum(int(m.sum()) for m in masks)


def test_cli_mask_glue_with_stand_ins(tmp_path, monkeypatch, capsys):
    """--mask soft|hard: the masked FASTA is the file with the union of the BED rows the same run writes masked; the BED
    and stdout are what a run without --mask gives.  Load limits of one load, several groups, and one record per load
    (records longer than a load: unit-relative rows, the unit origin in dst_offset)."""
    rng = random.Random(8)
    records = _glue_records(rng)
    write_fasta(tmp_path / "in.fa", records)
    monkeypatch.setattr(api, "get_context", lambda device=None: MaskContext())
    monkeypatch.chdir(tmp_path)
    argv = [str(tmp_path / "in.fa"), "-max", "12", "-o", str(tmp_path / "sub" / "out")]
    real_limit = _cabi.load_limit(12)
    for limit in (real_limit, 3500, 1):
        monkeypatch.setattr(_cabi, "load_limit", lambda cap, limit=limit: limit)
        assert cli.main(argv) == 0
        plain_bed, plain_out = (tmp_path / "out.bed").read_bytes(), capsys.readouterr().out
        for kind in ("soft", "hard"):
            masked = _check_cli_mask(tmp_path, capsys, records, argv, kind)
            assert (tmp_path / "out.bed").read_bytes() == plain_bed and masked > 500
        assert not (tmp_path / "sub").exists() and "Wrote masked" not in plain_out


def test_cli_mask_with_min_repeats_1(tmp_path, monkeypatch, capsys):
    """The per-record --min-repeats 1 loop: its rows are painted too; a run that raises leaves no masked file (the BED
    file behaves as without --mask)."""
    rng = random.Random(9)
    records = _glue_records(rng)
    write_fasta(tmp_path / "in.fa", records)
    monkeypatch.setattr(api, "get_context", lambda device=None: MaskContext())
    monkeypatch.setattr(api, "detect_repeats", lambda seq, fs, device=None: oracle.detect_repeats(seq, fs))
    monkeypatch.chdir(tmp_path)
    argv = [str(tmp_path / "in.fa"), "-max", "8", "--min-repeats", "1", "--min-span", "4", "-o", "out"]
    assert _check_cli_mask(tmp_path, capsys, records, argv, "soft") > 500
    calls = []

    def raising(seq, fs, device=None):
        calls.append(1)
        if len(calls) == 3:
            raise IndexError("string index out of range")
        return oracle.detect_repeats(seq, fs)
    monkeypatch.setattr(api, "detect_repeats", raising)
    os.remove(tmp_path / "out.masked.fa")
    with pytest.raises(IndexError):
        cli.main(argv + ["--mask", "hard"])
    assert not (tmp_path / "out.masked.fa").exists() and (tmp_path / "out.bed").exists()


def test_cli_mask_argument_errors(tmp_path, monkeypatch, capsys):
    write_fasta(tmp_path / "in.fa", [(b"c", b"ACGT" * 20)])
    (tmp_path / "l.bed").write_text("c\t0\t10\n")
    monkeypatch.chdir(tmp_path)
    for argv in (["ACGTACGT", "--mask", "soft"], [str(tmp_path / "in.fa"), "-i", "c:0-10", "--mask", "soft"],
                 [str(tmp_path / "in.fa"), "--intervals", str(tmp_path / "l.bed"), "--mask", "hard"],
                 [str(tmp_path / "in.fa"), "--mask", "lower"]):
        with pytest.raises(SystemExit) as e:
            cli.main(argv)
        assert e.value.code == 2
        assert "--mask" in capsys.readouterr().err
    assert not list(tmp_path.glob("*.masked.fa")) and not list(tmp_path.glob("*.tsv"))


# ---- GPU --------------------------------------------------------------------------------------------------------------

def _rows_for(rng, lengths, n_rows):
    """Random rows over records of the given lengths: 1 base to several Mbp, many overlapping, some at record ends."""
    rec = np.array([rng.randrange(len(lengths)) for _ in range(n_rows)], np.uint32)
    start, end = np.zeros(n_rows, np.uint32), np.zeros(n_rows, np.uint32)
    for i, r in enumerate(rec.tolist()):
        n = lengths[r]
        span = min(n, rng.choice([1, rng.randint(1, 40), rng.randint(30, 300), rng.randint(200, 20_000),
                                  rng.randint(1_000_000, 5_000_000), 0]))
        a = rng.choice([0, n - span, rng.randint(0, n - span)])
        start[i], end[i] = a, a + span
    return rec, start, end


@pytest.mark.gpu
def test_mask_rows_against_the_numpy_union():
    """Host and device rows, host and device masks; records not word-aligned; rows of 0 bases to 5 Mbp."""
    import torch
    ctx = api.get_context(0)
    rng = random.Random(11)
    lengths = [rng.randint(1, 100) for _ in range(50)] + [rng.randint(1000, 100_000) for _ in range(40)] + \
              [5_000_003, 7_777_777, 33]
    dst = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.uint64) + 5       # 5 leading bits nobody covers
    n_bits = int(dst[-1]) + lengths[-1] + 17
    for n_rows in (1, 1000, 300_000):
        rec, start, end = _rows_for(rng, lengths, n_rows)
        want = words_of(union(n_bits, dst[rec].astype(np.int64) + start, dst[rec].astype(np.int64) + end))
        got = ctx.mask_rows(rec, start, end, dst, n_bits)
        assert np.array_equal(got, want), n_rows
        order = np.random.default_rng(n_rows).permutation(n_rows)                  # row order does not matter
        assert np.array_equal(ctx.mask_rows(rec[order], start[order], end[order], dst, n_bits), want)
        cols = [torch.from_numpy(a.astype(np.int32)).to("cuda:0") for a in (rec, start, end)]
        for rows_dev in (False, True):
            out = torch.full((want.size,), -1, dtype=torch.int32, device="cuda:0")   # every word is written
            args = [c.data_ptr() for c in cols] if rows_dev else [rec, start, end]
            ctx.mask_rows(*args, dst, n_bits, n_rows=n_rows, mask=out.data_ptr())
            assert np.array_equal(out.cpu().numpy().view(np.uint32), want)
        got = ctx.mask_rows(*[c.data_ptr() for c in cols], dst, n_bits, n_rows=n_rows)
        assert np.array_equal(got, want)
    assert ctx.mask_rows(np.zeros(0), np.zeros(0), np.zeros(0), dst, 100).tolist() == [0, 0, 0, 0]


@pytest.mark.gpu
def test_mask_rows_above_two_to_the_32():
    """A mask of 2^33 bits and no scan: destinations around 2^32 and up to its last bit."""
    import torch
    ctx = api.get_context(0)
    n_bits = 1 << 33
    dst = np.array([0, (1 << 32) - 7, 1 << 32, (1 << 33) - 3_000_000, (1 << 33) - 10], np.uint64)
    rec = np.array([0, 1, 1, 2, 2, 3, 4, 4, 1], np.uint32)
    start = np.array([5, 0, 3, 0, 100, 0, 0, 9, 0], np.uint32)
    end = np.array([40, 7, 20, 2_500_000, 2_600_000, 3_000_000, 10, 10, 0], np.uint32)
    want = np.zeros(n_bits // 32, np.uint32)
    for r, s, e in zip(rec.tolist(), start.tolist(), end.tolist()):
        a, b = int(dst[r]) + s, int(dst[r]) + e
        lo, hi = a // 32 * 32, -(-b // 32) * 32
        want[lo // 32:hi // 32] |= words_of(union(hi - lo, [a - lo], [b - lo]))
    out = torch.full((n_bits // 32,), -1, dtype=torch.int32, device="cuda:0")
    ctx.mask_rows(rec, start, end, dst, n_bits, mask=out.data_ptr())
    got = out.cpu().numpy().view(np.uint32)
    assert np.array_equal(got, want)
    assert int(np.unpackbits(got[got != 0].view(np.uint8)).sum()) == 35 + (2_600_000 + 7) + 3_000_000
    del out
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_mask_rows_refuses_bad_rows():
    """end < start, record >= n_records, a range past mask_bits: CRF_ERR_ARG (ValueError), from host and device rows."""
    import torch
    ctx = api.get_context(0)
    dst = np.array([0, 100], np.uint64)
    good = (np.array([0, 1, 1], np.uint32), np.array([3, 0, 50], np.uint32), np.array([90, 100, 100], np.uint32))
    assert ctx.mask_rows(*good, dst, 200).size == 7
    bad = {"ends before it starts": (1, 60, 59), "n_records": (2, 0, 1), "past mask_bits": (1, 50, 101)}
    for message, row in bad.items():
        cols = [np.append(c, v).astype(np.uint32) for c, v in zip(good, row)]
        with pytest.raises(ValueError, match=message):
            ctx.mask_rows(*cols, dst, 200)
        dev = [torch.from_numpy(c.astype(np.int32)).to("cuda:0") for c in cols]
        with pytest.raises(ValueError, match=message):
            ctx.mask_rows(*[d.data_ptr() for d in dev], dst, 200, n_rows=4)
    with pytest.raises(ValueError, match="past mask_bits"):                            # dst + end wraps past 2^64
        ctx.mask_rows(np.zeros(1, np.uint32), np.zeros(1, np.uint32), np.ones(1, np.uint32),
                      np.array([2 ** 64 - 1], np.uint64), 200)
    assert ctx.mask_rows(*good, dst, 200).size == 7                                    # the context is still fine


DEFAULTS = dict(min_motif_size=1, max_motif_size=50, min_repeats=3, min_span=9)


def _oracle_mask(text, offsets, fs):
    """The union of the oracle's rows of every record, from one oracle call over the records with max_motif_size N's
    between them (no run crosses an N), as tests/test_batch.py checks scan_batch."""
    offsets = np.asarray(offsets, np.int64)
    gap = int(fs.max_motif_size)
    src = np.frombuffer(text, np.uint8)
    lengths = np.diff(offsets)
    at = np.concatenate([[0], np.cumsum(lengths + gap)])                    # record r starts at at[r] in the gapped text
    gapped = np.full(int(at[-1]), ord("N"), np.uint8)
    for r in range(lengths.size):
        gapped[at[r]:at[r] + lengths[r]] = src[offsets[r]:offsets[r + 1]]
    s, e, _, _ = oracle.detect_repeats_by_k(gapped, fs, arrays=True)
    r = np.searchsorted(at, s, side="right") - 1
    assert (e <= at[r] + lengths[r]).all()
    return union(len(text), s - at[r] + offsets[r], e - at[r] + offsets[r])


def _both(text, offsets, fs, **kw):
    """repeat_mask from host bytes and from a CUDA tensor: must be bit-identical; returns the host result."""
    import torch
    host = mask.repeat_mask(text, offsets, fs, **kw)
    assert isinstance(host, np.ndarray) and host.dtype == bool and host.shape == (len(text),)
    dev = mask.repeat_mask(torch.frombuffer(bytearray(text), dtype=torch.uint8).to("cuda:0"), offsets, fs, **kw)
    assert dev.is_cuda and dev.dtype == torch.bool and dev.shape == (len(text),)
    assert np.array_equal(dev.cpu().numpy(), host)
    return host


@pytest.mark.gpu
def test_repeat_mask_of_reads_and_long_sequences_against_the_oracle():
    from oracle import oracle as orc  # noqa: F401 (built C oracle)
    n_reads = 100_000
    bases, offsets, _ = synth.sr(n_reads)
    text = bases.tobytes()
    fs = ns(**{**DEFAULTS, "max_motif_size": 20})
    got = _both(text, offsets, fs, device=0)
    assert mask.last_stats["loads"] == 1 and mask.last_stats["rows"] > 10_000
    want = _oracle_mask(text, offsets, fs)
    assert np.array_equal(got, want) and want.sum() > 100_000
    rng = random.Random(70)
    from tests.test_batch import _planted
    seqs = [_planted(rng, rng.choice([rng.randint(1, 5000), rng.randint(5000, 70_000)])).encode() for _ in range(300)]
    text = b"NNN" + b"".join(seqs) + b"acgt"                                  # bases outside every record stay False
    offsets = 3 + np.concatenate([[0], np.cumsum([len(s) for s in seqs])])
    got = _both(text, offsets, ns(**DEFAULTS), device=0)
    want = _oracle_mask(text, offsets, ns(**DEFAULTS))
    assert np.array_equal(got, want) and want.sum() > 200_000
    assert not got[:3].any() and not got[-4:].any()
    with pytest.raises(NotImplementedError, match="detect_repeats_batch"):
        mask.repeat_mask(text, offsets, ns(**{**DEFAULTS, "min_repeats": 1}), device=0)
    with pytest.raises(NotImplementedError, match="detect_repeats_batch"):
        mask.repeat_mask(text, offsets, ns(**DEFAULTS, interval_end=100), device=0)


@pytest.mark.gpu
def test_repeat_mask_over_several_loads(monkeypatch):
    from tests.test_batch import _planted
    rng = random.Random(72)
    seqs = [_planted(rng, rng.randint(0, 20_000)).encode() for _ in range(120)]
    monkeypatch.setattr(batch, "_load_limit", lambda kmax: 100_000)
    text = b"".join(seqs)
    offsets = np.concatenate([[0], np.cumsum([len(s) for s in seqs])])
    got = _both(text, offsets, ns(**DEFAULTS), device=0)
    assert mask.last_stats["loads"] >= 10
    assert np.array_equal(got, _oracle_mask(text, offsets, ns(**DEFAULTS)))
    assert len(text) > 1_000_000                                            # as one record: ten times the patched limit
    with pytest.raises(NotImplementedError, match="longer than one device load"):
        mask.repeat_mask(text, [0, len(text)], ns(**DEFAULTS), device=0)


@pytest.mark.gpu
@pytest.mark.parametrize("devices,kind", [(None, "soft"), ("0,0", "hard")])
def test_cli_masked_fasta_of_s22_against_the_oracle(tmp_path, monkeypatch, capsys, devices, kind):
    monkeypatch.chdir(tmp_path)
    bases, _, _ = synth.s22(device="cuda:0")
    raw = bases.cpu().numpy().tobytes()
    del bases
    write_fasta(tmp_path / "s22.fa", [(b"chr22", raw)])
    fs = ns(min_motif_size=1, max_motif_size=6, min_repeats=3, min_span=9)
    argv = [str(tmp_path / "s22.fa"), "-min", "1", "-max", "6", "-o", "s22", "--mask", kind]
    assert cli.main(argv + (["--devices", devices] if devices else [])) == 0
    want_mask = _oracle_mask(raw, [0, len(raw)], fs)
    assert (tmp_path / "s22.masked.fa").read_bytes() == _fast_masked_fasta(b"chr22", raw, want_mask, kind == "hard")
    assert want_mask.sum() > 500_000
    assert capsys.readouterr().out.endswith("Wrote masked sequence to s22.masked.fa\n")


def _fast_masked_fasta(name, raw, m, hard):
    text = np.frombuffer(raw, np.uint8).copy()
    if hard:
        text[m] = ord("N")
    else:
        text[m & (text >= ord("A")) & (text <= ord("Z"))] += 32
    t = text.tobytes()
    return b">" + name + b"\n" + b"".join(t[i:i + 60] + b"\n" for i in range(0, len(t), 60))


@pytest.mark.gpu
def test_cli_mask_with_min_repeats_1_on_the_gpu(tmp_path, monkeypatch, capsys):
    rng = random.Random(12)
    records = _glue_records(rng)
    write_fasta(tmp_path / "in.fa", records)
    monkeypatch.chdir(tmp_path)
    argv = [str(tmp_path / "in.fa"), "-max", "8", "--min-repeats", "1", "--min-span", "4", "-o", "out"]
    assert _check_cli_mask(tmp_path, capsys, records, argv, "soft") > 500
    bed = (tmp_path / "out.bed").read_text()
    want = []
    for name, seq in records:
        want += [f"{name.decode()}\t{s}\t{e}\t{m}\n" for s, e, m in
                 oracle.detect_repeats(seq, ns(min_motif_size=1, max_motif_size=8, min_repeats=1, min_span=4))]
    assert bed == "".join(want)
