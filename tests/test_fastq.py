"""FASTQ input: the native reader (crf_fasta_open on a file whose first byte that is not whitespace is '@'), the masked
FASTQ writer (crf_write_fastq_masked) and the command line on FASTQ files.

CPU tests check the reader against a Python statement of the parse rules, the writer against a Python statement of the
format, both under sanitizers (tests/fuzz_fastq.cpp), and the CLI glue with the scan replaced by the oracle.  The -m gpu
tests run the scan on reads files: the BED of a FASTQ file is byte-identical to the BED of the same reads as FASTA."""
import gzip
import os
import random
import shutil
import struct
import subprocess
import sys
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, cli, fasta, synth  # noqa: E402
from oracle import oracle  # noqa: E402
from tests.helpers import ns, random_seq  # noqa: E402
from tests.test_intervals import stand_ins  # noqa: E402,F401 (the scan and crf_interval_stop as stand-ins)
from tests.test_mask import MaskContext, mask_from_bed, words_of  # noqa: E402


# ---- the format, stated in Python ------------------------------------------------------------------------------------

def parse_fastq(text):
    """The parse rules: a record is a header line '@name ...' (name = first whitespace-delimited token), sequence lines up
    to a line starting with '+', then quality lines until they hold as many bytes as the sequence.  A line is its bytes up
    to '\\n' or the end, without one trailing '\\r'.  Whitespace between records is skipped.  Returns [(name, seq, qual)];
    raises ValueError(f"FASTQ record {n}: ...") for the first fault."""
    lines = text.split(b"\n")
    lines = [ln[:-1] if ln.endswith(b"\r") else ln for ln in lines]
    ends_with_newline = text.endswith(b"\n")
    if ends_with_newline:
        lines.pop()
    out, i, n_lines = [], 0, len(lines)

    def fail(why):
        raise ValueError(f"FASTQ record {len(out) + 1}: {why}")
    while True:
        # whitespace between records (blank lines, or blank bytes before the '@')
        while i < n_lines and lines[i].strip(b" \t\r\n\v\f") == b"":
            i += 1
        if i == n_lines:
            return out
        line = lines[i].lstrip(b" \t\r\n\v\f")
        if not line.startswith(b"@"):
            fail("text that is not whitespace before its '@' header")
        name = line[1:].split()[0] if line[1:].split() else b""
        i += 1
        seq = []
        while True:
            if i >= n_lines:
                fail("the file ends inside the record")
            if lines[i].startswith(b"+"):
                i += 1
                break
            seq.append(lines[i])
            i += 1
        seq = b"".join(seq)
        qual = b""
        while len(qual) < len(seq):
            if i >= n_lines:
                fail("the file ends inside the record")
            if len(qual) + len(lines[i]) > len(seq):
                fail("its quality is longer than its sequence")
            if any(c < 33 or c > 126 for c in lines[i]):
                fail("a quality byte outside '!'..'~'")
            qual += lines[i]
            i += 1
        out.append((name, seq, qual))


def fastq_bytes(reads, eol=b"\n", desc=False):
    """4-line FASTQ of (name, seq, qual) reads."""
    return b"".join(b"@" + n + (b" 1:N:0:ACGT" if desc and k % 2 else b"") + eol + s + eol + b"+" + eol + q + eol
                    for k, (n, s, q) in enumerate(reads))


def fasta_bytes(reads):
    return b"".join(b">" + n + b"\n" + s + b"\n" for n, s, *_ in reads)


def bgzf(raw, block=65280, level=1):
    """bgzip's container (gzip members of <= 64 KiB with a 'BC' extra field holding the member's size, then the empty
    end-of-file block), the members compressed on several threads."""
    def member(chunk):
        comp = zlib.compressobj(level, zlib.DEFLATED, -15)
        data = comp.compress(chunk) + comp.flush()
        return (b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\0\xff" + struct.pack("<H", 6) + b"BC" +
                struct.pack("<HH", 2, 12 + 6 + len(data) + 8 - 1) + data + struct.pack("<II", zlib.crc32(chunk), len(chunk)))
    with ThreadPoolExecutor(16) as ex:
        parts = list(ex.map(member, (raw[i:i + block] for i in range(0, len(raw), block))))
    return b"".join(parts) + member(b"")


def random_quals(rng, n):
    """Seeded qualities whose first byte is often '@', '+' or '>'."""
    q = bytes(rng.randrange(33, 127) for _ in range(n))
    return (rng.choice(b"@+>I").to_bytes(1, "big") + q[1:]) if n and rng.random() < 0.6 else q


def random_reads(rng, n, max_len=200):
    reads = []
    for i in range(n):
        L = 0 if rng.random() < 0.05 else rng.randint(1, max_len)
        reads.append((f"read{i}".encode(), random_seq(rng, L, exotic=True).encode(), random_quals(rng, L)))
    return reads


def read_back(path, threads=0, qualities=True):
    with _cabi.Fasta(str(path), n_threads=threads, qualities=qualities) as fa:
        assert fa.format == "fastq"
        assert fa.total_bases == int(fa.offsets[-1]) == len(fa.bases)
        out = [(n.encode(), fa.record(i).tobytes(),
                fa.quals[int(fa.offsets[i]):int(fa.offsets[i + 1])].tobytes() if qualities else None)
               for i, n in enumerate(fa.names)]
        if not qualities:
            assert fa.quals is None
    return out


def check_reader(path, text, threads=(1, 16)):
    want = parse_fastq(text)
    for t in threads:
        assert read_back(path, t) == want, (path, t)
        assert [r[:2] for r in read_back(path, t, qualities=False)] == [r[:2] for r in want]
    return want


# ---- CPU: the reader -------------------------------------------------------------------------------------------------

def test_python_statement_on_hand_made_cases():
    got = parse_fastq(b"\n  @r1 desc\nAC\nGT\n+r1\n@@\r\n+>\n\n@e\n\n+\n\n@r3\r\nN\r\n+\r\n>")
    assert got == [(b"r1", b"ACGT", b"@@+>"), (b"e", b"", b""), (b"r3", b"N", b">")]


def test_reader_containers_and_line_ends(tmp_path):
    """Plain, gzip, multi-member gzip and BGZF; LF and CRLF; descriptions; quality lines starting with '@', '+' and '>';
    empty reads; lower-case, IUPAC and N bases."""
    rng = random.Random(1)
    reads = random_reads(rng, 400)
    reads[3] = (b"empty", b"", b"")
    reads[7] = (b"q_at", b"ACGT", b"@III")
    reads[8] = (b"q_plus", b"acgt", b"+III")
    reads[9] = (b"q_gt", b"RYKN", b">III")
    for eol in (b"\n", b"\r\n"):
        text = fastq_bytes(reads, eol, desc=True)
        assert [r for r in parse_fastq(text)] == reads
        containers = {"plain.fq": text, "plain.fq.gz": gzip.compress(text, 6),
                      "members.fq.gz": gzip.compress(text[:5000], 1) + gzip.compress(text[5000:], 9),
                      "blocks.fastq.bgz": bgzf(text, block=4000)}
        for name, blob in containers.items():
            (tmp_path / name).write_bytes(blob)
            assert check_reader(tmp_path / name, text) == reads, (name, eol)


def test_reader_multi_line_records_and_blank_lines(tmp_path):
    rng = random.Random(2)
    reads = random_reads(rng, 200, 300)
    parts = []
    for k, (n, s, q) in enumerate(reads):
        cut = [0] + sorted(rng.sample(range(1, len(s)), min(len(s) - 1, rng.randint(0, 3)))) + [len(s)] if s else [0, 0]
        parts.append(b"@" + n + b"\n" + b"".join(s[a:b] + b"\n" for a, b in zip(cut, cut[1:])) + b"+\n")
        qcut = [0] + sorted(rng.sample(range(1, len(q)), min(len(q) - 1, rng.randint(0, 3)))) + [len(q)] if q else [0]
        parts.append(b"".join(q[a:b] + b"\n" for a, b in zip(qcut, qcut[1:])))
        if k % 9 == 0:
            parts.append(b"\n \t\n")
    text = b"\n\n" + b"".join(parts) + b"\n\n"
    assert parse_fastq(text) == reads
    (tmp_path / "multi.fq").write_bytes(text)
    check_reader(tmp_path / "multi.fq", text)
    (tmp_path / "multi.fq.gz").write_bytes(gzip.compress(text))
    check_reader(tmp_path / "multi.fq.gz", text)


def test_reader_across_many_pieces_and_the_serial_fall_back(tmp_path):
    """~2 x 10^5 reads of random lengths (~70 MB of text: 9 pieces of the threaded path), and the same file with one
    record on several lines in the middle (the whole text then goes to the serial parser): the same records."""
    rng = np.random.default_rng(3)
    n = 220_000
    lengths = rng.integers(0, 300, n)
    lengths[rng.random(n) < 0.01] = 0
    total = int(lengths.sum())
    bases = np.frombuffer(b"ACGTNacgtR", np.uint8)[rng.integers(0, 10, total)].tobytes()
    quals = rng.integers(33, 127, total, dtype=np.uint8)
    starts = np.concatenate([[0], np.cumsum(lengths)])
    firsts = starts[:-1][lengths > 0]
    quals[firsts] = np.frombuffer(b"@+>", np.uint8)[rng.integers(0, 3, firsts.size)]
    quals = quals.tobytes()
    reads = [(f"SRR{i}.{i}".encode(), bases[starts[i]:starts[i + 1]], quals[starts[i]:starts[i + 1]]) for i in range(n)]
    text = fastq_bytes(reads, desc=True)
    assert len(text) > 8 * (8 << 20)
    (tmp_path / "big.fq").write_bytes(text)
    for t in (1, 16):
        assert read_back(tmp_path / "big.fq", t) == reads
    mid = next(i for i in range(n // 2, n) if lengths[i] > 10)
    name, s, q = reads[mid]
    one_multi = (fastq_bytes(reads[:mid], desc=True) + b"@" + name + b"\n" + s[:5] + b"\n" + s[5:] + b"\n+\n" + q[:3] +
                 b"\n" + q[3:] + b"\n" + fastq_bytes(reads[mid + 1:], desc=True))
    (tmp_path / "big_multi.fq").write_bytes(one_multi)
    for t in (1, 16):
        assert read_back(tmp_path / "big_multi.fq", t) == reads


ERRORS = [
    (b"@r1\nACGT\n+\nIIII\n@r2\nACGT\n+\nII", 2, "ends inside"),
    (b"@r1\nACGT\n+\nIIII\n@r2\nACGT\n", 2, "ends inside"),
    (b"@r1\nACGT", 1, "ends inside"),
    (b"@r1\nACGT\n+\nIIII\n@r2\nAC\n+\nIII\n", 2, "longer than its sequence"),
    (b"@r1\nACGT\n+\nII\nIII\n", 1, "longer than its sequence"),
    (b"@r1\nACGT\n+\nIIII\n@r2\nAC\n+\nI \n", 2, "outside"),
    (b"@r1\nACGT\n+\nII\x7fI\n", 1, "outside"),
    (b"@r1\nACGT\n+\nIIII\n@r2\nAC\n+\nII\nACGT\n", 3, "not whitespace before"),
    (b"@r1\nACGT\n+\nIIII\nIIII\n", 2, "not whitespace before"),
    (b"\n\n  @r1\nACGT\n+\nIIII\n>r2\nACGT\n", 2, "not whitespace before"),
]


@pytest.mark.parametrize("text,record,why", ERRORS)
def test_reader_errors_name_the_record(tmp_path, text, record, why):
    """Every fault is a ValueError naming the 1-based record, with the same message at 1 and 16 threads."""
    with pytest.raises(ValueError, match=f"FASTQ record {record}: .*{why}"):
        parse_fastq(text)
    path = tmp_path / "bad.fq"
    path.write_bytes(text)
    msgs = []
    for t in (1, 16):
        with pytest.raises(ValueError, match=f"FASTQ record {record}: .*{why}") as e:
            _cabi.Fasta(str(path), n_threads=t)
        msgs.append(str(e.value))
    assert msgs[0] == msgs[1]
    (tmp_path / "bad.fq.gz").write_bytes(gzip.compress(text))
    with pytest.raises(ValueError, match=f"FASTQ record {record}: .*{why}"):
        _cabi.Fasta(str(tmp_path / "bad.fq.gz"))


def test_fasta_files_are_read_as_before(tmp_path):
    """Only a text whose first byte that is not whitespace is '@' is FASTQ: FASTA (with '@' and '+' lines inside
    records) keeps its format and records."""
    text = b">c1 x\nACGT\n@@\n+\n>c2\n\nNN\n"
    (tmp_path / "a.fa").write_bytes(text)
    with fasta.open_fasta(str(tmp_path / "a.fa"), qualities=True) as fa:
        assert fa.format == "fasta" and fa.quals is None
        assert fa.names == ["c1", "c2"] and fa.bases.tobytes() == b"ACGT@@+NN"
    assert [(r.name, r.seq) for r in fasta.read_fasta(str(tmp_path / "a.fa"))] == [("c1", b"ACGT@@+"), ("c2", b"NN")]
    (tmp_path / "r.fq").write_bytes(b"  \n@x y\nAC\n+\n!!\n")
    assert [(r.name, r.seq) for r in fasta.read_fasta(str(tmp_path / "r.fq"))] == [("x", b"AC")]


def test_fastq_harness_under_sanitizers(tmp_path):
    """tests/fuzz_fastq.cpp: the reader with pieces of 1-97 bytes and the masked FASTQ writer, without the CUDA runtime,
    under ASan + UBSan."""
    if not shutil.which("g++"):
        pytest.skip("no g++")
    exe = str(tmp_path / "fuzz_fastq")
    built = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                            "-pthread", "-I", os.path.join(ROOT, "colab-repeat-finder_b200", "csrc"),
                            "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "fuzz_fastq.cpp"), "-o", exe,
                            "-lz"], capture_output=True, text=True)
    if built.returncode != 0:
        pytest.skip("sanitizer build not available here: " + built.stderr[-300:])
    run = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-4000:]
    assert "ok 60 texts" in run.stdout and "16 files" in run.stdout


# ---- CPU: the masked FASTQ writer ------------------------------------------------------------------------------------

def masked_fastq(reads, masks, hard):
    """The masked FASTQ format, stated one base at a time."""
    out = []
    for (name, seq, qual), m in zip(reads, masks):
        s = bytes(ord("N") if x and hard else c + 32 if x and ord("A") <= c <= ord("Z") else c for c, x in zip(seq, m))
        out.append(b"@" + name + b"\n" + s + b"\n+\n" + qual + b"\n")
    return b"".join(out)


@pytest.mark.parametrize("hard", [False, True])
def test_fastq_writer_matches_the_format(tmp_path, hard):
    rng = random.Random(4)
    for n_reads in (0, 1, 5, 300, 40_000):                 # 40 000 reads of <= 300 bp: several threads and waves
        reads = random_reads(rng, n_reads, 300) if n_reads < 1000 else \
            [(f"r{i}".encode(), bytes(rng.choice(b"ACGTacgtNR") for _ in range(rng.randint(0, 300))), None)
             for i in range(n_reads)]
        reads = [(n, s, q if q is not None else bytes(73 for _ in s)) for n, s, q in reads]
        lead = b"xy"
        blob, qblob = lead + b"".join(s for _, s, _ in reads), b"qq" + b"".join(q for _, _, q in reads)
        offsets = len(lead) + np.concatenate([[0], np.cumsum([len(s) for _, s, _ in reads])]).astype(np.uint64)
        masks = [np.array([rng.random() < 0.4 for _ in s], bool) for _, s, _ in reads]
        bits = np.concatenate([np.zeros(len(lead), bool)] + masks)
        path = tmp_path / "out.fq"
        n = _cabi.write_fastq_masked(str(path), [r[0].decode() for r in reads], np.frombuffer(blob, np.uint8), qblob,
                                     offsets, words_of(bits), hard=hard)
        want = masked_fastq(reads, masks, hard)
        assert path.read_bytes() == want and n == len(want), n_reads


def test_fastq_writer_refusals(tmp_path):
    offsets = np.array([0, 4], np.uint64)
    with pytest.raises(ValueError, match="quals"):
        _cabi.write_fastq_masked(str(tmp_path / "x.fq"), ["a"], b"ACGT", b"III", offsets, np.zeros(1, np.uint32))
    with pytest.raises(ValueError):
        _cabi.write_fastq_masked(str(tmp_path / "x.fq"), ["a"], b"ACGT", b"IIII", np.array([0, 5], np.uint64),
                                 np.zeros(1, np.uint32))
    with pytest.raises(ValueError):
        _cabi.write_fastq_masked(str(tmp_path / "no" / "dir.fq"), ["a"], b"ACGT", b"IIII", offsets, np.zeros(1, np.uint32))
    if os.path.exists("/dev/full"):                                         # a short write is an error, not a shorter file
        with pytest.raises(OSError, match="failed"):
            _cabi.write_fastq_masked("/dev/full", ["a"], b"ACGT" * 50_000, b"I" * 200_000, np.array([0, 200_000], np.uint64),
                                     np.zeros(6250, np.uint32))


# ---- CPU: the command line with stand-ins -----------------------------------------------------------------------------

def _glue_reads(rng):
    reads = [(b"chrA", random_seq(rng, 3000).encode()), (b"chrB", random_seq(rng, 50).encode()), (b"empty", b""),
             (b"chrC", random_seq(rng, 7000, exotic=True).encode()), (b"chrD", (b"acgt" * 30 + b"AC" * 40) * 9)]
    reads += [(f"read{i}".encode(), random_seq(rng, rng.randint(0, 150)).encode()) for i in range(300)]
    return [(n, s, random_quals(rng, len(s))) for n, s in reads]


def _run(capsys, argv):
    assert cli.main(argv) == 0
    return capsys.readouterr().out


def test_cli_fastq_bed_equals_fasta_bed(tmp_path, monkeypatch, capsys):
    """The BED and stdout of a FASTQ file are byte-identical to those of the FASTA file of the same reads: whole file in
    one load, several load groups, records longer than a load, and the per-record --min-repeats 1 loop."""
    rng = random.Random(5)
    all_reads = _glue_reads(rng)
    monkeypatch.setattr(api, "get_context", lambda device=None: MaskContext())
    monkeypatch.setattr(api, "detect_repeats", lambda seq, fs, device=None: oracle.detect_repeats(seq, fs))
    monkeypatch.chdir(tmp_path)
    real_limit = _cabi.load_limit(12)
    # (--min-repeats 1 as the reference runs it raises IndexError on reads of a few bases, FASTA or FASTQ: not those)
    for extra in (["-max", "12"], ["-max", "8", "--min-repeats", "1", "--min-span", "4"]):
        reads = all_reads if len(extra) == 2 else [r for r in all_reads if len(r[1]) == 0 or len(r[1]) >= 10]
        (tmp_path / "r.fa").write_bytes(fasta_bytes(reads))
        (tmp_path / "r.fq").write_bytes(fastq_bytes(reads, desc=True))
        (tmp_path / "r.fq.gz").write_bytes(gzip.compress(fastq_bytes(reads, b"\r\n")))
        for limit in (real_limit, 3500, 1):
            monkeypatch.setattr(_cabi, "load_limit", lambda cap, limit=limit: limit)
            outs, beds = [], []
            for src in ("r.fa", "r.fq", "r.fq.gz"):
                outs.append(_run(capsys, [str(tmp_path / src), "-o", "out"] + extra))
                beds.append((tmp_path / "out.bed").read_bytes())
            assert beds[0] == beds[1] == beds[2] and len(beds[0]) > 1000, (extra, limit)
            assert outs[0] == outs[1] == outs[2]
            if len(extra) > 2:
                break


def test_cli_default_prefix_for_fastq(tmp_path, monkeypatch, capsys):
    reads = [(b"r1", b"ACACACACACACAC", b"I" * 14)]
    monkeypatch.setattr(api, "get_context", lambda device=None: MaskContext())
    monkeypatch.chdir(tmp_path)
    text = fastq_bytes(reads)
    for name, blob, bed in (("reads.fq", text, "reads.bed"), ("reads.fq.gz", gzip.compress(text), "reads.bed"),
                            ("s.fastq", text, "s.bed"), ("s.fastq.bgz", bgzf(text), "s.bed"),
                            ("s.fastq.gz", gzip.compress(text), "s.bed"), ("x.txt", text, "x.txt.bed"),
                            ("my.fastqc.fq", text, "my.fastqc.bed")):
        (tmp_path / "in").mkdir(exist_ok=True)
        (tmp_path / "in" / name).write_bytes(blob)
        out = _run(capsys, [str(tmp_path / "in" / name)])
        assert out.endswith(f"Wrote results to {bed}\n"), name
        assert (tmp_path / bed).read_text() == "r1\t0\t14\tAC\n"
        os.remove(tmp_path / bed)
    # FASTA input keeps the reference's (unanchored) regex
    (tmp_path / "in" / "g.fasta.gz").write_bytes(gzip.compress(fasta_bytes(reads)))
    assert _run(capsys, [str(tmp_path / "in" / "g.fasta.gz")]).endswith("Wrote results to g.bed\n")
    assert cli.default_prefix("reads.fastq.gz", "fasta") == "readsstq.gz"
    assert cli.default_prefix("reads.fastq.gz", "fastq") == "reads"


@pytest.mark.parametrize("kind", ["soft", "hard"])
def test_cli_mask_on_fastq(tmp_path, monkeypatch, capsys, kind):
    """--mask on FASTQ writes <basename(prefix)>.masked.fq: the reads with the union of the BED rows masked, names and
    qualities as read; the BED and stdout are what the FASTA file gives."""
    rng = random.Random(6)
    reads = _glue_reads(rng)
    (tmp_path / "r.fa").write_bytes(fasta_bytes(reads))
    (tmp_path / "r.fq.gz").write_bytes(gzip.compress(fastq_bytes(reads, desc=True)))
    monkeypatch.setattr(api, "get_context", lambda device=None: MaskContext())
    monkeypatch.chdir(tmp_path)
    for limit in (None, 3500):
        if limit:
            monkeypatch.setattr(_cabi, "load_limit", lambda cap: limit)
        fa_out = _run(capsys, [str(tmp_path / "r.fa"), "-max", "12", "--mask", kind])
        fa_bed = (tmp_path / "r.bed").read_bytes()
        fq_out = _run(capsys, [str(tmp_path / "r.fq.gz"), "-max", "12", "--mask", kind])
        assert (tmp_path / "r.bed").read_bytes() == fa_bed
        assert fq_out == fa_out.replace("r.masked.fa", "r.masked.fq")
        assert fq_out.endswith("Wrote results to r.bed\nWrote masked sequence to r.masked.fq\n")
        masks = mask_from_bed(fa_bed.decode(), [n.decode() for n, _, _ in reads], [s for _, s, _ in reads])
        assert sum(int(m.sum()) for m in masks) > 500
        assert (tmp_path / "r.masked.fq").read_bytes() == masked_fastq(reads, masks, kind == "hard")


def test_cli_interval_and_intervals_on_read_names(tmp_path, monkeypatch, capsys, stand_ins):
    rng = random.Random(7)
    reads = _glue_reads(rng)
    (tmp_path / "r.fa").write_bytes(fasta_bytes(reads))
    (tmp_path / "r.fq").write_bytes(fastq_bytes(reads))
    (tmp_path / "l.bed").write_text("chrA\t100\t2000\nread3\t0\t100\nchrD\t5\t400\nchrA\t0\t50\n")
    monkeypatch.chdir(tmp_path)
    for opt in (["-i", "chrA:100-2000"], ["-i", "chrD:0-400"], ["--intervals", str(tmp_path / "l.bed")]):
        outs, beds = [], []
        for src in ("r.fa", "r.fq"):
            outs.append(_run(capsys, [str(tmp_path / src), "-max", "10", "-o", "o"] + opt))
            beds.append((tmp_path / "o.bed").read_bytes())
        assert beds[0] == beds[1] and len(beds[0]) > 50, opt
        assert outs[0] == outs[1]
    with pytest.raises(SystemExit):
        cli.main([str(tmp_path / "r.fq"), "-i", "nosuch:0-10"])


# ---- GPU --------------------------------------------------------------------------------------------------------------

DEFAULTS = dict(min_motif_size=1, max_motif_size=20, min_repeats=3, min_span=9)


def c5_files(tmp_path, n_reads, containers=("fq",)):
    """Config C5 reads (synth.sr) with seeded qualities, written as FASTA (one line per read) and as FASTQ in the given
    containers ("fq", "fq.gz", "fq.bgz").  Returns (host bases, offsets, quals, {container: path})."""
    bases, offsets, _ = synth.sr(n_reads, device="cuda:0")
    host = bases.cpu().numpy()
    del bases
    rl = 150
    rng = np.random.default_rng(150)
    quals = rng.integers(33, 127, (n_reads, rl), dtype=np.uint8)
    quals[:, 0] = np.frombuffer(b"@+>I", np.uint8)[rng.integers(0, 4, n_reads)]
    idx = np.arange(n_reads, dtype=np.int64)
    name = np.empty((n_reads, 9), np.uint8)
    name[:, 0] = ord("r")
    for d in range(8):
        name[:, 8 - d] = ord("0") + (idx // 10 ** d) % 10
    reads = host.reshape(n_reads, rl)
    fa = np.empty((n_reads, 1 + 9 + 1 + rl + 1), np.uint8)
    fa[:, 0], fa[:, 1:10], fa[:, 10], fa[:, 11:11 + rl], fa[:, -1] = ord(">"), name, 10, reads, 10
    paths = {"fa": tmp_path / "reads.fa"}
    fa.tofile(paths["fa"])
    del fa
    fq = np.empty((n_reads, 1 + 9 + 1 + rl + 3 + rl + 1), np.uint8)
    fq[:, 0], fq[:, 1:10], fq[:, 10], fq[:, 11:11 + rl] = ord("@"), name, 10, reads
    fq[:, 11 + rl:14 + rl] = np.frombuffer(b"\n+\n", np.uint8)
    fq[:, 14 + rl:14 + 2 * rl], fq[:, -1] = quals, 10
    text = fq.reshape(-1)
    for c in containers:
        paths[c] = tmp_path / f"reads.{c}"
        if c == "fq":
            text.tofile(paths[c])
        elif c == "fq.gz":
            paths[c].write_bytes(gzip.compress(text.tobytes(), 1))
        else:
            paths[c].write_bytes(bgzf(text.tobytes()))
    del fq, text
    return host, offsets, quals.reshape(-1), paths


def oracle_bed(tmp_path, host, n_reads, rl=150):
    """The oracle's rows for the reads (one oracle call over the reads with max_motif_size N's between them, as
    test_all_ten_million_reads_row_by_row checks them), written by the native row writer."""
    gap = DEFAULTS["max_motif_size"]
    gapped = np.full((n_reads, rl + gap), ord("N"), dtype=np.uint8)
    gapped[:, :rl] = host.reshape(n_reads, rl)
    o_s, o_e, o_m, _ = oracle.detect_repeats_by_k(gapped.reshape(-1), ns(**DEFAULTS), arrays=True)
    del gapped
    o_rec = o_s // (rl + gap)
    path = tmp_path / "oracle.bed"
    names = b"".join(f"r{i:08d}".encode() + b"\0" for i in range(n_reads))
    _cabi.write_rows(str(path), names, host, np.arange(0, n_reads * rl + 1, rl, dtype=np.uint64), o_rec,
                     o_s - o_rec * (rl + gap), o_e - o_rec * (rl + gap), o_m)
    return path.read_bytes()


def _cli_bed(tmp_path, src, extra=()):
    """The CLI in a process of its own (stdout to a file: a reads file prints two lines per read)."""
    out = tmp_path / "stdout.txt"
    with open(out, "wb") as f:
        subprocess.run([sys.executable, os.path.join(ROOT, "perfect_repeat_finder.py"), str(src), "-min", "1", "-max", "20",
                        "-o", "out", *extra], stdout=f, check=True, cwd=tmp_path)
    return (tmp_path / "out.bed").read_bytes(), out.read_bytes()


@pytest.mark.gpu
def test_c5_reads_as_fastq_plain_gzip_bgzf(tmp_path):
    n_reads = 100_000
    host, _, _, paths = c5_files(tmp_path, n_reads, ("fq", "fq.gz", "fq.bgz"))
    want_bed, want_out = _cli_bed(tmp_path, paths["fa"])
    assert want_bed == oracle_bed(tmp_path, host, n_reads) and want_bed.count(b"\n") > 10_000
    for c in ("fq", "fq.gz", "fq.bgz"):
        bed, out = _cli_bed(tmp_path, paths[c])
        assert bed == want_bed, c
        assert out == want_out, c


@pytest.mark.gpu
def test_all_ten_million_c5_reads_as_fastq(tmp_path):
    n_reads = 10_000_000
    host, _, _, paths = c5_files(tmp_path, n_reads)
    fa_bed, fa_out = _cli_bed(tmp_path, paths["fa"])
    fq_bed, fq_out = _cli_bed(tmp_path, paths["fq"])
    assert fq_bed == fa_bed and fq_out == fa_out
    del fa_out, fq_out
    assert fa_bed == oracle_bed(tmp_path, host, n_reads) and fa_bed.count(b"\n") > 500_000


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["soft", "hard"])
def test_cli_mask_on_c5_fastq(tmp_path, kind):
    """The sequence lines of the masked FASTQ are the masked FASTA's records; names and qualities are the input's."""
    n_reads = 100_000
    host, _, quals, paths = c5_files(tmp_path, n_reads, ("fq.gz",))
    _cli_bed(tmp_path, paths["fa"], ("--mask", kind))
    fa_lines = (tmp_path / "out.masked.fa").read_bytes().split(b"\n")
    _cli_bed(tmp_path, paths["fq.gz"], ("--mask", kind))
    fq_lines = (tmp_path / "out.masked.fq").read_bytes().split(b"\n")
    assert len(fq_lines) == 4 * n_reads + 1 and fq_lines[-1] == b""
    names = [f"r{i:08d}".encode() for i in range(n_reads)]
    assert fq_lines[0:-1:4] == [b"@" + n for n in names]
    assert fa_lines[0:-1:4] == [b">" + n for n in names]                 # 150 bp at 60 per line: 3 lines per record
    masked = [b"".join(fa_lines[4 * i + 1:4 * i + 4]) for i in range(n_reads)]
    assert fq_lines[1:-1:4] == masked
    assert fq_lines[2:-1:4] == [b"+"] * n_reads
    assert b"".join(fq_lines[3:-1:4]) == quals.tobytes()
    text = np.frombuffer(b"".join(masked), np.uint8)
    assert int(((text >= ord("a")) & (text <= ord("z"))).sum() + (text == ord("N")).sum()) > 100_000


@pytest.mark.gpu
def test_open_fasta_on_fastq_feeds_scan_batch_and_repeat_mask(tmp_path):
    import torch
    from crf_b200 import batch, mask
    n_reads = 100_000
    _, _, quals, paths = c5_files(tmp_path, n_reads, ("fq.bgz",))
    fs = ns(**DEFAULTS)
    with fasta.open_fasta(str(paths["fa"])) as fa, fasta.open_fasta(str(paths["fq.bgz"]), qualities=True) as fq:
        assert fq.format == "fastq" and fq.quals.tobytes() == quals.tobytes()
        assert np.array_equal(fa.offsets, fq.offsets) and fa.names_blob == fq.names_blob
        want = batch.scan_batch(fa.bases, fa.offsets, fs, device=0)
        got = batch.scan_batch(fq.bases, fq.offsets, fs, device=0)
        assert all(np.array_equal(a, b) for a, b in zip(got, want)) and want[0].size > 10_000
        m_fa = mask.repeat_mask(fa.bases, fa.offsets, fs, device=0)
        m_fq = mask.repeat_mask(fq.bases, fq.offsets, fs, device=0)
        assert np.array_equal(m_fa, m_fq) and m_fa.sum() > 100_000
        dev = torch.from_numpy(fq.bases.copy()).to("cuda:0")
        assert torch.equal(mask.repeat_mask(dev, fq.offsets, fs, device=0).cpu(), torch.from_numpy(m_fa))
