"""BAM input: the native reader (crf_fasta_open on a BGZF file whose first inflated bytes are "BAM\\1"), the rows writer that
reads the motif from the 4-bit codes (crf_write_rows_nibbles), the GPU load from the codes (crf_seq_load_nibbles) and the
command line on unaligned BAM files.

The file has its own small BAM writer (BGZF blocks of at most 64 KiB with the 'BC' extra field, records across block
boundaries, the 28-byte end-of-file block) and a Python statement of what `samtools fastq -n` writes.  A BAM file must give
what the FASTQ reader gives on that FASTQ: offsets, names, bases and qualities.  CPU tests check the reader, the packed form,
malformed records, the memory bound, the writer and the CLI glue with the scan replaced by the oracle; tests/fuzz_bam.cpp
runs the reader under sanitizers.  The -m gpu tests check that the rows of a BAM load equal those of the ASCII load of the
decoded text and the oracle's, and that a BAM file gives the BED file of its FASTQ."""
import os
import random
import shutil
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, cli  # noqa: E402
from oracle import oracle  # noqa: E402
from tests.helpers import ns  # noqa: E402
from tests.test_intervals import StopContext, stand_ins  # noqa: E402,F401 (stand_ins: fixture)
from tests.test_mask import MaskContext  # noqa: E402

LETTERS = b"=ACMGRSVTWYHKDBN"
CODE = {c: i for i, c in enumerate(LETTERS)}
COMP = bytes(LETTERS[int(f"{i:04b}"[::-1], 2)] for i in range(16))     # complement: the code's 4-bit bit-reversal
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


# ---- the format, stated in Python --------------------------------------------------------------------------------------

class Read:
    """One BAM record: name (bytes), flag, bases (letters of =ACMGRSVTWYHKDBN), qualities (list of 0..93, or None:
    absent), n_cigar_op, tags (raw bytes)."""

    def __init__(self, name, flag, seq, qual=None, n_cigar=0, tags=b""):
        self.name, self.flag, self.seq, self.qual, self.n_cigar, self.tags = name, flag, seq, qual, n_cigar, tags


def pack_seq(seq):
    """Letters -> BAM seq bytes, the first base in the high nibble, a padding nibble 0."""
    c = np.frombuffer(bytes(LETTERS.index(x) for x in seq), np.uint8) if seq else np.zeros(0, np.uint8)
    c = np.concatenate([c, np.zeros(len(c) & 1, np.uint8)]).reshape(-1, 2)
    return ((c[:, 0] << 4) | c[:, 1]).astype(np.uint8).tobytes()


def record_bytes(r, l_seq=None, block_size=None, l_read_name=None):
    seq = pack_seq(r.seq)
    n = len(r.seq)
    qual = bytes(r.qual) if r.qual is not None else b"\xff" * n
    name = r.name + b"\0"
    body = struct.pack("<iiBBHHHiiii", -1, -1, len(name) if l_read_name is None else l_read_name, 255, 4680, r.n_cigar,
                       r.flag, n if l_seq is None else l_seq, -1, -1, 0)
    body += name + b"\0\0\0\0" * r.n_cigar + seq + qual + r.tags
    return struct.pack("<I", len(body) if block_size is None else block_size) + body


def bam_stream(reads, text=b"@HD\tVN:1.6\tSO:unknown\n", refs=((b"chr1", 1000),)):
    head = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    head += b"".join(struct.pack("<i", len(n) + 1) + n + b"\0" + struct.pack("<i", z) for n, z in refs)
    return head + b"".join(record_bytes(r) for r in reads)


def bgzf(raw, block=65280, eof=True, level=6):
    """BGZF: gzip members of at most 64 KiB, each with a 'BC' extra field holding its size minus 1, then the 28-byte
    end-of-file block.  Records cross the block boundaries wherever they fall."""
    out = []
    for i in range(0, len(raw), block):
        chunk = raw[i:i + block]
        comp = zlib.compressobj(level, zlib.DEFLATED, -15)
        data = comp.compress(chunk) + comp.flush()
        out.append(b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\0\xff" + struct.pack("<H", 6) + b"BC" +
                   struct.pack("<HH", 2, 12 + 6 + len(data) + 8 - 1) + data +
                   struct.pack("<II", zlib.crc32(chunk), len(chunk)))
        assert len(out[-1]) <= 65536
    return b"".join(out) + (EOF_BLOCK if eof else b"")


def samtools_fastq(reads):
    """What `samtools fastq -n` writes: records with (flag & 0x900) == 0 in file order, '@' + read name, the bases
    reverse-complemented when flag & 0x10, '+', qualities + 33 (reversed with them; '"' each when absent)."""
    out = []
    for r in reads:
        if r.flag & 0x900:
            continue
        seq = r.seq
        q = bytes(x + 33 for x in r.qual) if r.qual is not None else b'"' * len(seq)
        if r.flag & 0x10:
            seq = bytes(COMP[LETTERS.index(c)] for c in reversed(seq))
            q = q[::-1]
        out.append(b"@" + r.name + b"\n" + seq + b"\n+\n" + q + b"\n")
    return b"".join(out)


def nibble_form(reads):
    """(nib, rec_byte, exotic) the reader must give: the kept reads' codes (reverse complements applied, padding 0), each
    from a byte, and (position << 8 | letter) of the codes other than A, C, G, T, N."""
    nib, rec_byte, ex, pos = [], [], [], 0
    for r in reads:
        if r.flag & 0x900:
            continue
        seq = bytes(COMP[LETTERS.index(c)] for c in reversed(r.seq)) if r.flag & 0x10 else r.seq
        rec_byte.append(sum(len(b) for b in nib))
        nib.append(pack_seq(seq))
        ex += [((pos + i) << 8) | c for i, c in enumerate(seq) if c not in b"ACGTN"]
        pos += len(seq)
    return b"".join(nib), np.array(rec_byte, np.uint64), np.array(ex, np.uint64)


def random_read(rng, i, max_len=300, exotic=0.02):
    n = 0 if rng.random() < 0.05 else rng.randint(1, max_len)
    seq = bytes(rng.choice(LETTERS) if rng.random() < exotic else rng.choice(b"ACGTACGTN") for _ in range(n))
    qual = None if rng.random() < 0.2 else [rng.randint(0, 93) for _ in range(n)]
    flag = rng.choice([0x4, 0x4 | 0x10, 0x0, 0x10, 0x100, 0x800, 0x4 | 0x1 | 0x40, 0x4 | 0x1 | 0x80, 0x910, 0x4 | 0x1 | 0x80 | 0x10])
    name = (b"q%d_" % i) + bytes(rng.choice(b"abcdefghij:/|") for _ in range(rng.choice([0, 3, 30, 250])))
    return Read(name[:254], flag, seq, qual, n_cigar=rng.choice([0, 0, 2]), tags=rng.choice([b"", b"RGZgrp1\0", b"NMi\x05\0\0\0"]))


def read_back(path, threads=0, qualities=True):
    with _cabi.Fasta(str(path), n_threads=threads, qualities=qualities) as fa:
        q = fa.quals.tobytes() if fa.quals is not None else None
        return fa.format, fa.offsets.copy(), fa.names, fa.bases.tobytes(), q


def check_against_fastq(tmp_path, reads, blob=None, threads=(1, 16)):
    """The reader on the BAM equals the reader on the FASTQ samtools writes: offsets, names, bases and qualities."""
    bam = tmp_path / "t.bam"
    bam.write_bytes(bgzf(bam_stream(reads)) if blob is None else blob)
    fq = tmp_path / "t.fq"
    fq.write_bytes(samtools_fastq(reads))
    _, off, names, text, quals = read_back(fq, 1)
    for t in threads:
        fmt, b_off, b_names, b_text, b_quals = read_back(bam, t)
        assert fmt == "bam"
        assert np.array_equal(b_off, off) and b_names == names and b_text == text and b_quals == quals, t
    nib, rec_byte, ex = nibble_form(reads)
    with _cabi.Fasta(str(bam)) as fa:
        src = fa.nibbles()
        assert src.nib.tobytes() == nib and np.array_equal(src.rec_byte, rec_byte) and np.array_equal(src.exotic, ex)
        assert fa.quals is None
    return len(off) - 1


# ---- CPU: the reader ----------------------------------------------------------------------------------------------------

def test_python_statement_on_hand_made_reads():
    reads = [Read(b"a", 0x4, b"ACGTN", [0, 1, 2, 3, 40]), Read(b"b", 0x10, b"AACM", [1, 2, 3, 4]),
             Read(b"s", 0x100, b"AAA"), Read(b"u", 0x800, b"CCC"), Read(b"e", 0x4, b""), Read(b"c", 0x4, b"GT")]
    assert samtools_fastq(reads) == b"@a\nACGTN\n+\n!\"#$I\n@b\nKGTT\n+\n%$#\"\n@e\n\n+\n\n@c\nGT\n+\n\"\"\n"
    assert COMP == b"=TGKCYSBAWRDMHVN"
    nib, rec_byte, ex = nibble_form(reads)
    assert nib == bytes([0x12, 0x48, 0xF0, 0xC4, 0x88, 0x48]) and rec_byte.tolist() == [0, 3, 5, 5]
    assert ex.tolist() == [(5 << 8) | ord("K")]


def test_reader_flags_lengths_codes_and_names(tmp_path):
    """Flags 0x4, 0x10, 0x100, 0x800 and paired 0x1/0x40/0x80; odd and even lengths, l_seq == 0 and all 16 codes; absent
    qualities and 254-character names, on 1 and 16 threads."""
    rng = random.Random(1)
    reads = [random_read(rng, i) for i in range(600)]
    reads.append(Read(b"x" * 254, 0x4, LETTERS * 3, list(range(48))))
    reads.append(Read(b"rc", 0x10, LETTERS, None))
    reads.append(Read(b"empty", 0x4, b""))
    assert check_against_fastq(tmp_path, reads) > 300


def test_reader_many_reads_and_small_windows(tmp_path, monkeypatch):
    """10^5 short reads, with the default window and with windows of one block or a few (records span them)."""
    rng = np.random.default_rng(2)
    n = 100_000
    lengths = rng.integers(0, 160, n)
    codes = np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, int(lengths.sum()))]
    reads, at = [], 0
    for i, z in enumerate(lengths.tolist()):
        reads.append(Read(b"r%d" % i, [0x4, 0x14, 0x104][i % 3], codes[at:at + z].tobytes(),
                          rng.integers(0, 60, z).tolist() if i % 5 else None))
        at += z
    blob = bgzf(bam_stream(reads), level=1)
    for window in (None, "1", "150000"):
        if window:
            monkeypatch.setenv("CRF_BAM_WINDOW", window)
        assert check_against_fastq(tmp_path, reads, blob, threads=(4,)) == n - n // 3


def test_reader_block_layouts(tmp_path, monkeypatch):
    """Small blocks (every record across a boundary), no end-of-file block, a large header and reference list."""
    rng = random.Random(3)
    reads = [random_read(rng, i, max_len=3000) for i in range(200)]
    text = b"@HD\tVN:1.6\n" + b"@CO\t" + b"z" * 200_000 + b"\n"
    refs = [(b"contig%d" % i, 1000 + i) for i in range(5000)]
    monkeypatch.setenv("CRF_BAM_WINDOW", "1")
    for blob in (bgzf(bam_stream(reads), block=1000), bgzf(bam_stream(reads), eof=False),
                 bgzf(bam_stream(reads, text, refs), block=7777)):
        check_against_fastq(tmp_path, reads, blob, threads=(1, 5))


def test_empty_bam_and_formats_kept_apart(tmp_path):
    (tmp_path / "e.bam").write_bytes(bgzf(bam_stream([])))
    with _cabi.Fasta(str(tmp_path / "e.bam")) as fa:
        assert fa.format == "bam" and fa.n_records == 0 and fa.bases.size == 0
        assert fa.nibbles().nib.size == 0
    (tmp_path / "g.fa").write_bytes(b">chr1\nACGT\n")
    with _cabi.Fasta(str(tmp_path / "g.fa")) as fa:
        with pytest.raises(ValueError, match="not a BAM file"):
            fa.nibbles()
    (tmp_path / "g.fq.bgz").write_bytes(bgzf(b"@r\nACGT\n+\nIIII\n"))
    with _cabi.Fasta(str(tmp_path / "g.fq.bgz")) as fa:
        assert fa.format == "fastq" and fa.bases.tobytes() == b"ACGT"


def test_magic_spanning_blocks_is_bam(tmp_path):
    """A BGZF file whose first blocks hold fewer than 4 bytes each is still BAM: the magic is read across blocks."""
    reads = [Read(b"a", 4, b"ACGTAC", [30] * 6), Read(b"b", 0x14, b"GGA")]
    stream = bam_stream(reads)
    blob = bgzf(stream[:1], eof=False) + bgzf(b"", eof=False) + bgzf(stream[1:3], eof=False) + bgzf(stream[3:])
    assert check_against_fastq(tmp_path, reads, blob, threads=(1,)) == 2


def test_source_extent_is_checked():
    """A NibbleSource or TwoBitSource whose records run past its host bytes is refused before anything is read."""
    offsets = np.array([0, 5, 9], np.uint64)
    _cabi._check_extent("nib", np.zeros(5, np.uint8), np.array([0, 3], np.uint64), offsets, 2)
    with pytest.raises(ValueError, match="past the end of nib"):
        _cabi._check_extent("nib", np.zeros(4, np.uint8), np.array([0, 3], np.uint64), offsets, 2)
    with pytest.raises(ValueError, match="past the end of dna"):
        _cabi._check_extent("dna", b"\0" * 3, np.array([0, 3], np.uint64), offsets, 4)
    _cabi._check_extent("nib", np.zeros(0, np.uint8), np.array([7, 7], np.uint64), np.zeros(3, np.uint64), 2)


def test_bam_in_plain_gzip_is_refused(tmp_path):
    import gzip
    (tmp_path / "p.bam").write_bytes(gzip.compress(bam_stream([Read(b"a", 4, b"ACGT")])))
    with pytest.raises(ValueError, match="plain gzip, not BGZF"):
        _cabi.Fasta(str(tmp_path / "p.bam"))


def _bad_cases():
    good = [Read(b"one", 4, b"ACGTACGT", [30] * 8), Read(b"two", 4, b"GATTACA", [20] * 7), Read(b"three", 4, b"CCCC")]
    head = bam_stream([])

    def with_second(**kw):
        return head + record_bytes(good[0]) + record_bytes(good[1], **kw) + record_bytes(good[2])
    rb = record_bytes(good[1])
    no_nul = rb[:4 + 32 + 3] + b"X" + rb[4 + 32 + 4:]
    stream = head + record_bytes(good[0]) + record_bytes(good[1]) + record_bytes(good[2])
    return [
        ("block_size < 32", with_second(block_size=20), 2, "block_size is less than 32"),
        ("l_read_name 0", with_second(l_read_name=0), 2, "l_read_name is 0"),
        ("no NUL", head + record_bytes(good[0]) + no_nul + record_bytes(good[2]), 2, "does not end with a NUL"),
        ("l_seq negative", with_second(l_seq=-3), 2, "l_seq is negative"),
        ("l_seq too long", with_second(l_seq=100), 2, "fields run past its block_size"),
        ("n_cigar_op", head + record_bytes(good[0]) + record_bytes(Read(b"two", 4, b"GA", n_cigar=0))[:4 + 12] +
         struct.pack("<H", 60000) + record_bytes(Read(b"two", 4, b"GA"))[4 + 14:] + record_bytes(good[2]), 2,
         "fields run past its block_size"),
        ("block_size past the data", with_second(block_size=10 ** 6), 2, "runs past the end of the data"),
        ("truncated", stream[:-5], 3, "runs past the end of the data"),
        ("trailing bytes", stream + b"\1\0", 4, "the data ends inside the record"),
    ]


@pytest.mark.parametrize("what,stream,record,why", _bad_cases(), ids=[c[0] for c in _bad_cases()])
def test_reader_errors_name_the_record(tmp_path, monkeypatch, what, stream, record, why):
    for window in ("1", "33554432"):
        monkeypatch.setenv("CRF_BAM_WINDOW", window)
        (tmp_path / "bad.bam").write_bytes(bgzf(stream, block=50))
        with pytest.raises(ValueError, match=rf"BAM record {record}: .*{why}"):
            _cabi.Fasta(str(tmp_path / "bad.bam"))


def test_reader_header_errors(tmp_path):
    good = bam_stream([Read(b"a", 4, b"ACGT")])
    for data, why in ((good[:10], "truncated"), (good[:4] + struct.pack("<i", -1) + good[8:], "l_text is negative"),
                      (good[:4] + struct.pack("<i", 10 ** 6) + good[8:], "the text runs past"),
                      (bam_stream([], refs=[(b"c", 5)])[:-3], "reference list runs past")):
        (tmp_path / "h.bam").write_bytes(bgzf(data))
        with pytest.raises(ValueError, match=f"BAM header: .*{why}"):
            _cabi.Fasta(str(tmp_path / "h.bam"))
    blob = bytearray(bgzf(good))
    blob[30] ^= 0xFF                                               # inside the first block's compressed data
    (tmp_path / "c.bam").write_bytes(bytes(blob))
    with pytest.raises(ValueError, match="corrupt BGZF block"):
        _cabi.Fasta(str(tmp_path / "c.bam"))


def test_peak_memory_stays_below_the_inflated_size(tmp_path):
    """A BAM whose tags inflate to 400 MB is read in windows: the reader's peak RSS grows by far less than that."""
    tag = b"XZZ" + b"k" * (2 << 20) + b"\0"
    reads = [Read(b"r%d" % i, 4, b"ACGT" * 25, [30] * 100, tags=tag) for i in range(200)]
    stream = bam_stream(reads)
    assert len(stream) > 400 << 20
    (tmp_path / "big.bam").write_bytes(bgzf(stream, level=1))
    del stream
    script = (
        "import resource, sys\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'colab-repeat-finder_b200')!r})\n"
        "from crf_b200 import _cabi\n"
        "_cabi.lib()\n"
        "with _cabi.Fasta(sys.argv[2]) as fa: pass\n"
        "before = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss\n"
        "with _cabi.Fasta(sys.argv[1], qualities=True) as fa:\n"
        "    assert fa.n_records == 200 and fa.total_bases == 20000\n"
        "print(resource.getrusage(resource.RUSAGE_SELF).ru_maxrss - before)\n")
    (tmp_path / "warm.fq").write_bytes(b"@a\nACGT\n+\nIIII\n")
    out = subprocess.run([sys.executable, "-c", script, str(tmp_path / "big.bam"), str(tmp_path / "warm.fq")],
                         capture_output=True, text=True, check=True)
    grew_kib = int(out.stdout.strip())
    assert grew_kib < 120 * 1024, grew_kib                          # window 32 MiB + record 2 MiB, not 400 MB


def test_existing_callers_read_the_decoded_text(tmp_path):
    """crf_fasta_packed and read_fasta work on a BAM handle through its decoded text."""
    from crf_b200 import fasta
    from tests.fake_ctx import unpack_planes
    rng = random.Random(4)
    reads = [random_read(rng, i) for i in range(300)]
    (tmp_path / "r.bam").write_bytes(bgzf(bam_stream(reads)))
    (tmp_path / "r.fq").write_bytes(samtools_fastq(reads))
    with _cabi.Fasta(str(tmp_path / "r.bam")) as fa, _cabi.Fasta(str(tmp_path / "r.fq")) as fq:
        assert fa._bases is None
        pa, pq = fa.packed(), fq.packed()
        assert unpack_planes(pa).tobytes() == unpack_planes(pq).tobytes()
        assert np.array_equal(pa.exotic, pq.exotic)
    got, want = fasta.read_fasta(str(tmp_path / "r.bam")), fasta.read_fasta(str(tmp_path / "r.fq"))
    assert [(r.name, r.seq) for r in got] == [(r.name, r.seq) for r in want]


def test_bam_harness_under_sanitizers(tmp_path):
    """tests/fuzz_bam.cpp: random BAMs read on 1 and several threads against a C++ statement of samtools fastq -n, with
    truncations and flipped bits (every outcome the right content or CRF_ERR_ARG, never a fault), and
    crf_write_rows_nibbles against crf_write_rows, without the CUDA runtime, under AddressSanitizer and UBSan."""
    if not shutil.which("g++"):
        pytest.skip("no g++")
    exe = str(tmp_path / "fuzz_bam")
    built = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                            "-pthread", "-I", os.path.join(ROOT, "colab-repeat-finder_b200", "csrc"),
                            "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "fuzz_bam.cpp"), "-o", exe,
                            "-lz"], capture_output=True, text=True)
    assert built.returncode == 0, built.stderr[-4000:]
    run = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=900,
                         env={**os.environ, "ASAN_OPTIONS": "detect_leaks=1"})
    assert run.returncode == 0 and run.stdout.startswith("ok "), (run.stdout[-2000:], run.stderr[-4000:])


# ---- CPU: the rows writer -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tsv", [False, True])
def test_rows_nibbles_equals_rows_on_the_text(tmp_path, tsv):
    """150 000 rows (several formatting threads and waves), reverse reads and exotic codes among them: byte-identical to
    crf_write_rows on the decoded text."""
    rng = np.random.default_rng(8)
    reads = []
    for i in range(60):
        n = int(rng.integers(0, 20000))
        seq = np.frombuffer(LETTERS, np.uint8)[np.where(rng.random(n) < 0.05, rng.integers(0, 16, n),
                                                        np.array([1, 2, 4, 8])[rng.integers(0, 4, n)])].tobytes()
        reads.append(Read(b"read%d" % i, [0x4, 0x14][i % 2], seq))
    (tmp_path / "w.bam").write_bytes(bgzf(bam_stream(reads)))
    with _cabi.Fasta(str(tmp_path / "w.bam")) as fa:
        src = fa.nibbles()
        lengths = np.diff(fa.offsets.astype(np.int64))
        m = 150_000
        rec = np.sort(rng.choice(np.flatnonzero(lengths > 60), m))
        k = rng.integers(1, 51, m)
        start = (rng.random(m) * (lengths[rec] - k)).astype(np.int64)
        end = np.minimum(start + k * rng.integers(1, 4, m), lengths[rec])
        names = None if tsv else fa.names_blob
        a = _cabi.write_rows(str(tmp_path / "a"), names, fa.bases, fa.offsets, rec, start, end, k, tsv=tsv)
        b = _cabi.write_rows_nibbles(str(tmp_path / "b"), names, src.nib, src.rec_byte, rec, start, end, k, tsv=tsv)
        a2 = _cabi.write_rows(str(tmp_path / "a"), names, fa.bases, fa.offsets, rec[:10], start[:10], end[:10], k[:10],
                              tsv=tsv, append=True)
        b2 = _cabi.write_rows_nibbles(str(tmp_path / "b"), names, src.nib, src.rec_byte, rec[:10], start[:10], end[:10],
                                      k[:10], tsv=tsv, append=True)
    assert (a, a2) == (b, b2)
    assert (tmp_path / "a").read_bytes() == (tmp_path / "b").read_bytes() and a > 3_000_000


# ---- CPU: the command line with stand-ins -------------------------------------------------------------------------------

def _stand_in_load_nibbles(self, source, max_motif_cap=50, on_device=False):
    """The BAM load as a stand-in: decode the codes (the Python statement above) and load the text."""
    if isinstance(source, _cabi.Fasta):
        source = source.nibbles()
    nib = np.asarray(source.nib)
    codes = np.stack([nib >> 4, nib & 15], 1).reshape(-1)
    texts = [np.frombuffer(LETTERS, np.uint8)[codes[2 * b:2 * b + n]]
             for b, n in zip(source.rec_byte.tolist(), np.diff(source.offsets.astype(np.int64)).tolist())]
    BamMaskContext.loads_nibbles += 1
    return self.load(np.concatenate(texts + [np.zeros(0, np.uint8)]), source.offsets - source.offsets[0], max_motif_cap)


class BamMaskContext(MaskContext):
    loads_nibbles = 0
    load_nibbles = _stand_in_load_nibbles


class BamStopContext(StopContext):
    load_nibbles = _stand_in_load_nibbles


def _glue_reads(rng):
    def seq(n, exotic=0.0):
        return _repeat_rich(rng, n, exotic)
    reads = [Read(b"chrA", 4, seq(3000)), Read(b"chrB", 0x14, seq(50)), Read(b"empty", 4, b""),
             Read(b"chrC", 0x10, seq(7000, 0.01)), Read(b"chrD", 4, (b"ACGT" * 30 + b"AC" * 40) * 9),
             Read(b"sec", 0x100, seq(500)), Read(b"chrE", 4, b"N" * 30 + b"ACAC" * 20 + b"N" * 9)]
    reads += [Read(b"read%d" % i, rng.choice([4, 0x14, 0x4d, 0x8d, 0x900]), seq(rng.randint(0, 150)),
                   [rng.randint(0, 60) for _ in range(150)] if rng.random() < 0.7 else None) for i in range(300)]
    for r in reads:
        if r.qual is not None:
            r.qual = r.qual[:len(r.seq)] + [20] * (len(r.seq) - len(r.qual))
    return reads


def _run(capsys, argv):
    assert cli.main(argv) == 0
    return capsys.readouterr().out


def _write_pair(tmp_path, reads, stem="r"):
    (tmp_path / f"{stem}.fq").write_bytes(samtools_fastq(reads))
    (tmp_path / f"{stem}.bam").write_bytes(bgzf(bam_stream(reads)))


def _single_copy_ok(seq):
    try:
        oracle.detect_repeats(seq, ns(min_motif_size=1, max_motif_size=8, min_repeats=1, min_span=4))
        return True
    except IndexError:
        return False


def test_cli_bam_bed_equals_fastq_bed(tmp_path, monkeypatch, capsys):
    """BED and stdout of a BAM file equal those of its FASTQ: one load, several load groups, a record longer than a load
    (the decoded text's path), and --min-repeats 1."""
    rng = random.Random(21)
    reads = _glue_reads(rng)
    monkeypatch.setattr(api, "get_context", lambda device=None: BamMaskContext())
    monkeypatch.setattr(api, "detect_repeats", lambda seq, fs, device=None: oracle.detect_repeats(seq, fs))
    monkeypatch.chdir(tmp_path)
    real_limit = _cabi.load_limit(12)
    for extra in (["-max", "12"], ["-max", "8", "--min-repeats", "1", "--min-span", "4"]):
        kept = reads if len(extra) == 2 else [r for r in reads if _single_copy_ok(r.seq) and b"=" not in r.seq]
        _write_pair(tmp_path, kept)
        for limit in (real_limit, 7100, 3500, 1):
            monkeypatch.setattr(_cabi, "load_limit", lambda cap, limit=limit: limit)
            BamMaskContext.loads_nibbles = 0
            outs, beds = [], []
            for src in ("r.fq", "r.bam"):
                outs.append(_run(capsys, [str(tmp_path / src), "-o", "out"] + extra))
                beds.append((tmp_path / "out.bed").read_bytes())
            assert beds[0] == beds[1] and len(beds[0]) > 1000, (extra, limit)
            assert outs[0] == outs[1]
            if len(extra) == 2:                    # the codes' path (one load per group) unless a record exceeds a load
                assert BamMaskContext.loads_nibbles == 1 if limit == real_limit else \
                    (BamMaskContext.loads_nibbles > 1) == (limit == 7100)
            if len(extra) > 2:
                break


def test_cli_bam_interval_and_intervals(tmp_path, monkeypatch, capsys, stand_ins):
    rng = random.Random(22)
    _write_pair(tmp_path, _glue_reads(rng))
    monkeypatch.setattr(api, "get_context", lambda device=None: BamStopContext())
    (tmp_path / "l.bed").write_text("chrA\t100\t2000\nread3\t0\t100\nchrD\t5\t400\nchrA\t0\t50\n")
    monkeypatch.chdir(tmp_path)
    for opt in (["-i", "chrA:100-2000"], ["-i", "chrD:0-400"], ["--intervals", str(tmp_path / "l.bed")]):
        outs, beds = [], []
        for src in ("r.fq", "r.bam"):
            outs.append(_run(capsys, [str(tmp_path / src), "-max", "10", "-o", "o"] + opt))
            beds.append((tmp_path / "o.bed").read_bytes())
        assert beds[0] == beds[1] and len(beds[0]) > 50, opt
        assert outs[0] == outs[1]


@pytest.mark.parametrize("kind", ["soft", "hard"])
def test_cli_mask_on_bam(tmp_path, monkeypatch, capsys, kind):
    """--mask on BAM writes <prefix>.masked.fq from the decoded text and the qualities: the file its FASTQ gives."""
    rng = random.Random(23)
    reads = _glue_reads(rng)
    _write_pair(tmp_path, reads)
    monkeypatch.setattr(api, "get_context", lambda device=None: BamMaskContext())
    monkeypatch.chdir(tmp_path)
    for limit in (None, 3500):
        if limit:
            monkeypatch.setattr(_cabi, "load_limit", lambda cap: limit)
        fq_out = _run(capsys, [str(tmp_path / "r.fq"), "-max", "12", "--mask", kind])
        fq_bed, fq_masked = (tmp_path / "r.bed").read_bytes(), (tmp_path / "r.masked.fq").read_bytes()
        os.remove(tmp_path / "r.masked.fq")
        bam_out = _run(capsys, [str(tmp_path / "r.bam"), "-max", "12", "--mask", kind])
        assert (tmp_path / "r.bed").read_bytes() == fq_bed and bam_out == fq_out
        assert bam_out.endswith("Wrote results to r.bed\nWrote masked sequence to r.masked.fq\n")
        assert (tmp_path / "r.masked.fq").read_bytes() == fq_masked and fq_masked.count(b"\n") > 1000
        assert fq_masked != samtools_fastq(reads)


def test_cli_default_prefix_for_bam(tmp_path, monkeypatch, capsys):
    monkeypatch.setattr(api, "get_context", lambda device=None: BamMaskContext())
    monkeypatch.chdir(tmp_path)
    (tmp_path / "in").mkdir()
    blob = bgzf(bam_stream([Read(b"r1", 4, b"ACACACACACACAC")]))
    for name, bed in (("hifi.bam", "hifi.bed"), ("m.hifi_reads.bam", "m.hifi_reads.bed"), ("x.bam.bak", "x.bam.bak.bed"),
                      ("reads", "reads.bed"), ("my.fq.bam", "my.fq.bed")):
        (tmp_path / "in" / name).write_bytes(blob)
        out = _run(capsys, [str(tmp_path / "in" / name)])
        assert out.endswith(f"Wrote results to {bed}\n"), name
        assert (tmp_path / bed).read_text() == "r1\t0\t14\tAC\n"
        os.remove(tmp_path / bed)
    assert cli.default_prefix("a.fq.bam", "bam") == "a.fq" and cli.default_prefix("a.bam", "fastq") == "a.bam"


# ---- GPU ----------------------------------------------------------------------------------------------------------------

DEFAULTS = dict(min_motif_size=1, max_motif_size=50, min_repeats=3, min_span=9)


def _rows(seq):
    n = seq.scan(1, 50, 3, 9)
    return tuple(a.copy() for a in seq.fetch(n))


def _oracle_rows(text, offsets):
    out = [[], [], [], []]
    for r in range(len(offsets) - 1):
        s, e, m, _ = oracle.detect_repeats_by_k(np.frombuffer(text[int(offsets[r]):int(offsets[r + 1])], np.uint8),
                                                ns(**DEFAULTS), arrays=True)
        for col, vals in zip(out, (np.full(len(s), r), s, e, m)):
            col.append(np.asarray(vals, np.int64))
    return tuple(np.concatenate(c) if c else np.zeros(0, np.int64) for c in out)


def _check_load(path, with_oracle=True, tensor=False, records=None):
    ctx = api.get_context()
    with _cabi.Fasta(str(path), pinned=2) as fa:
        src = fa.nibbles()
        if tensor:
            import torch
            src = _cabi.NibbleSource(torch.from_numpy(src.nib.copy()).cuda(), src.rec_byte, src.offsets, src.exotic)
        first, last = records or (0, fa.n_records)
        with ctx.load_nibbles(src.records(first, last)) as seq:
            got = _rows(seq)
        b0, b1 = int(fa.offsets[first]), int(fa.offsets[last])
        text = fa.bases[b0:b1].tobytes()
        offsets = fa.offsets[first:last + 1] - np.uint64(b0)
        with ctx.load(fa.bases[b0:b1], offsets) as seq:
            want = _rows(seq)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    if with_oracle:
        for a, b in zip(got, _oracle_rows(text, offsets)):
            assert np.array_equal(a.astype(np.int64), b)
    return len(got[0])


def _repeat_rich(rng, n, exotic=0.0):
    parts, at = [], 0
    while at < n:
        unit = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(1, 12)))
        p = unit * rng.randint(1, 8) + bytes(rng.choice(LETTERS) if rng.random() < exotic else rng.choice(b"ACGTN")
                                             for _ in range(rng.randint(0, 40)))
        parts.append(p)
        at += len(p)
    return b"".join(parts)[:n]


@pytest.mark.gpu
def test_gpu_alignments_reverse_and_exotic_equal_ascii_load_and_oracle(tmp_path):
    """Records at both nibble phases (odd and even lengths before them) and every start within a 32-base word, reverse
    reads and exotic codes, empty records; also from a CUDA tensor, and a sub-range of the records."""
    rng = random.Random(30)
    reads = []
    for i, n in enumerate(list(range(10)) + list(range(28, 37)) + list(range(60, 69)) + [500, 3000, 0, 7, 20000] +
                          [rng.randint(0, 400) for _ in range(200)]):
        reads.append(Read(b"r%d" % i, [0x4, 0x14, 0x904][i % 3], _repeat_rich(rng, n, 0.01)))
    (tmp_path / "a.bam").write_bytes(bgzf(bam_stream(reads)))
    assert _check_load(tmp_path / "a.bam") > 200
    assert _check_load(tmp_path / "a.bam", tensor=True) > 200
    assert _check_load(tmp_path / "a.bam", records=(7, 150)) > 50


@pytest.mark.gpu
def test_gpu_hundred_thousand_reads(tmp_path):
    """10^5 reads of 150 bp, some with N's and exotic codes, a third reverse."""
    rng = np.random.default_rng(31)
    n, rl = 100_000, 150
    unit = rng.integers(0, 4, (n, 6))
    codes = np.where(rng.random((n, rl)) < 0.7, np.tile(unit, 25), rng.integers(0, 4, (n, rl)))
    letters = np.frombuffer(b"ACGT", np.uint8)[codes]
    letters[rng.random((n, rl)) < 0.002] = ord("N")
    letters[rng.random((n, rl)) < 0.0005] = ord("R")
    reads = [Read(b"q%d" % i, [0x4, 0x14, 0x4][i % 3], letters[i].tobytes(), rng.integers(0, 60, rl).tolist()) for i in range(n)]
    (tmp_path / "reads.bam").write_bytes(bgzf(bam_stream(reads), level=1))
    assert _check_load(tmp_path / "reads.bam", with_oracle=False) > 30_000
    assert _check_load(tmp_path / "reads.bam", with_oracle=False, tensor=True) > 30_000
    assert _check_load(tmp_path / "reads.bam", records=(0, 300)) > 50


@pytest.mark.gpu
def test_gpu_records_straddle_upload_chunks(tmp_path):
    """A span of 320 M positions (160 MB of codes: the chunked upload on the second stream, records across chunks),
    compared with the ASCII load; the oracle on one record."""
    rng = np.random.default_rng(32)
    reads = []
    for i in range(4):
        n = 80_000_001 + i
        c = np.repeat(rng.integers(0, 4, n // 8 + 1), 8)[:n]
        seq = np.frombuffer(b"ACGT", np.uint8)[c]
        seq[rng.integers(0, n, 50)] = ord("N")
        seq[rng.integers(0, n, 50)] = ord("Y")
        reads.append(Read(b"big%d" % i, [0x4, 0x14][i % 2], seq.tobytes()))
    reads.append(Read(b"small", 0x10, _repeat_rich(random.Random(3), 5000, 0.01)))
    (tmp_path / "big.bam").write_bytes(bgzf(bam_stream(reads), level=1))
    assert _check_load(tmp_path / "big.bam", with_oracle=False) > 10 ** 6
    assert _check_load(tmp_path / "big.bam", records=(4, 5)) > 10


def _cli(tmp_path, src, extra=()):
    out = tmp_path / "stdout.txt"
    with open(out, "wb") as f:
        subprocess.run([sys.executable, os.path.join(ROOT, "perfect_repeat_finder.py"), str(src), "-o", "out", *extra],
                       stdout=f, check=True, cwd=tmp_path)
    masked = tmp_path / "out.masked.fq"
    got = ((tmp_path / "out.bed").read_bytes(), out.read_bytes(), masked.read_bytes() if masked.exists() else None)
    if masked.exists():
        os.remove(masked)
    return got


@pytest.mark.gpu
def test_gpu_cli_bam_equals_fastq(tmp_path):
    """On one GPU a BAM gives the BED file and stdout of the same reads as FASTQ; -i, --intervals, --min-repeats 1 and
    --mask soft / hard on the BAM match the FASTQ's outputs."""
    rng = random.Random(40)
    reads = [Read(b"read%d" % i, [0x4, 0x14, 0x904, 0x4d][i % 4], _repeat_rich(rng, rng.randint(0, 2000), 0.002))
             for i in range(3000)]
    for r in reads:
        r.qual = [rng.randint(0, 60) for _ in r.seq] if rng.random() < 0.8 else None
    reads.append(Read(b"long", 0x10, _repeat_rich(rng, 300_000)))
    _write_pair(tmp_path, reads)
    (tmp_path / "l.bed").write_text("long\t100\t20000\nread5\t0\t100\nread9\t5\t400\n")
    single = [r for r in reads if not r.flag & 0x900 and len(r.seq) >= 10 and _single_copy_ok(r.seq) and b"=" not in r.seq]
    (tmp_path / "s.fq").write_bytes(samtools_fastq(single))
    (tmp_path / "s.bam").write_bytes(bgzf(bam_stream(single)))
    for stem, extra in (("r", []), ("r", ["-i", "long:100-20000"]), ("r", ["--intervals", str(tmp_path / "l.bed")]),
                        ("r", ["--mask", "soft"]), ("r", ["--mask", "hard"]),
                        ("s", ["-max", "8", "--min-repeats", "1", "--min-span", "4"])):
        want = _cli(tmp_path, tmp_path / f"{stem}.fq", extra)
        got = _cli(tmp_path, tmp_path / f"{stem}.bam", extra)
        assert got == want and want[0].count(b"\n") > 100, extra
