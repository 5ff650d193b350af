""".2bit input: the native reader (crf_fasta_open on a file that starts with the .2bit signature), the rows writer that reads
the motif from the packed bases (crf_write_rows_twobit), the GPU load from the packed bytes (crf_seq_load_2bit) and the
command line on .2bit files.

The file has its own small .2bit writer (both byte orders, both versions) and a Python statement of what twoBitToFa
writes.  CPU tests check the reader and the writer against them, both under sanitizers (tests/fuzz_twobit.cpp), and the CLI
glue with the scan replaced by the oracle.  The -m gpu tests check that the rows of a .2bit load equal those of the ASCII
load of the decoded text and the oracle's, and that a .2bit file gives the BED file of its FASTA."""
import hashlib
import json
import os
import random
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "colab-repeat-finder_b200"))

from crf_b200 import _cabi, api, cli  # noqa: E402
from oracle import oracle  # noqa: E402
from tests.helpers import ns, random_seq  # noqa: E402
from tests.test_intervals import StopContext, stand_ins  # noqa: E402,F401 (stand_ins: fixture)
from tests.test_mask import MaskContext, mask_from_bed, masked_fasta  # noqa: E402

SIG = 0x1A412743
CODE = {"T": 0, "C": 1, "A": 2, "G": 3}


# ---- the format, stated in Python --------------------------------------------------------------------------------------

class Rec:
    """One .2bit record: name, dnaSize, packed bases, N blocks and mask blocks as (start, size) in file order."""

    def __init__(self, name, size, packed, nblocks=(), mblocks=()):
        self.name, self.size, self.packed = name, size, bytes(packed)
        self.nblocks, self.mblocks = list(nblocks), list(mblocks)


def pack_codes(letters):
    """'TCAG' letters -> packed bytes, the first base in the top two bits."""
    codes = np.frombuffer(letters.encode(), np.uint8)
    lut = np.zeros(256, np.uint8)
    for c, v in CODE.items():
        lut[ord(c)] = v
    c = lut[codes]
    c = np.concatenate([c, np.zeros((-len(c)) % 4, np.uint8)]).reshape(-1, 4)
    return ((c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]).astype(np.uint8).tobytes()


def runs_of(flags, base=0):
    """(start, size) of the maximal runs of True."""
    f = np.concatenate([[False], np.asarray(flags, bool), [False]])
    d = np.flatnonzero(f[1:] != f[:-1])
    return [(base + int(a), int(b - a)) for a, b in zip(d[::2], d[1::2])]


def rec_from_text(name, text):
    """A record from text over ACGTN / acgtn (N bases stored as T, as faToTwoBit does)."""
    t = np.frombuffer(text.encode(), np.uint8)
    upper = (t & 0xDF).tobytes().decode()
    letters = upper.replace("N", "T")
    return Rec(name, len(text), pack_codes(letters), runs_of([c == "N" for c in upper]), runs_of(t >= ord("a")))


def twobit_bytes(recs, swap=False, version=0, order=None, reserved=0):
    """The .2bit file of recs; order: the order the records' data appear in the file (default: index order)."""
    e = ">" if swap else "<"
    off_fmt = "Q" if version else "I"
    order = list(range(len(recs))) if order is None else order
    index_size = 16 + sum(1 + len(r.name) + (8 if version else 4) for r in recs)
    data, where = [], [0] * len(recs)
    at = index_size
    for i in order:
        r = recs[i]
        hdr = struct.pack(e + "II", r.size, len(r.nblocks))
        hdr += struct.pack(e + "%dI" % len(r.nblocks), *[s for s, _ in r.nblocks])
        hdr += struct.pack(e + "%dI" % len(r.nblocks), *[z for _, z in r.nblocks])
        hdr += struct.pack(e + "I", len(r.mblocks))
        hdr += struct.pack(e + "%dI" % len(r.mblocks), *[s for s, _ in r.mblocks])
        hdr += struct.pack(e + "%dI" % len(r.mblocks), *[z for _, z in r.mblocks])
        hdr += struct.pack(e + "I", reserved)
        where[i] = at
        data.append(hdr + r.packed)
        at += len(hdr) + len(r.packed)
    head = [struct.pack(e + "IIII", SIG, version, len(recs), 0)]
    for r, w in zip(recs, where):
        head.append(bytes([len(r.name)]) + r.name + struct.pack(e + off_fmt, w))
    head = b"".join(head)
    assert len(head) == index_size
    return head + b"".join(data)


def merged(blocks):
    """Blocks (start, size) -> sorted, merged [a, b) runs."""
    out = []
    for a, b in sorted((s, s + z) for s, z in blocks if z):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return [tuple(x) for x in out]


def twobit_to_fa(rec):
    """What twoBitToFa writes for a record: T/C/A/G, N blocks as 'N', mask blocks lower-cased ('n' inside both)."""
    p = np.frombuffer(rec.packed, np.uint8)
    codes = np.stack([(p >> 6) & 3, (p >> 4) & 3, (p >> 2) & 3, p & 3], 1).reshape(-1)[:rec.size]
    t = np.frombuffer(b"TCAG", np.uint8)[codes].copy()
    for a, b in merged(rec.nblocks):
        t[a:b] = ord("N")
    for a, b in merged(rec.mblocks):
        t[a:b] |= 0x20
    return t.tobytes()


def expected(recs):
    """(text, offsets, names, N runs) the reader must give."""
    texts = [twobit_to_fa(r) for r in recs]
    offsets = np.concatenate([[0], np.cumsum([r.size for r in recs])]).astype(np.uint64)
    runs = [(int(offsets[i]) + a, int(offsets[i]) + b) for i, r in enumerate(recs) for a, b in merged(r.nblocks)]
    return b"".join(texts), offsets, [r.name for r in recs], np.array(runs, np.uint64).reshape(-1, 2)


def random_rec(rng, name, size, blocks=True):
    letters = "".join(rng.choice("TCAG") for _ in range(size))
    nb, mb = [], []
    if blocks and size:
        for lst in (nb, mb):
            for _ in range(rng.randint(0, 4)):
                s = rng.randint(0, size)
                lst.append((s, rng.randint(0, size - s)))          # may overlap, may come unsorted, may be empty
            if rng.random() < 0.5:
                lst.append((size - 1, 1))                          # at the record's end
            if rng.random() < 0.5:
                lst.append((0, min(size, rng.randint(1, 3))))      # at its start (adjacent to the previous record's end)
            rng.shuffle(lst)
    return Rec(name, size, pack_codes(letters), nb, mb)


def alignment_recs(rng):
    """Records of length 0-9 and around 32 and 64, so every byte and word alignment of a record start occurs."""
    sizes = list(range(10)) + list(range(28, 37)) + list(range(60, 69)) + [1, 3, 200, 0, 5, 1000, 7]
    return [random_rec(rng, b"r%d_%d" % (i, n), n) for i, n in enumerate(sizes)]


def read_back(path, threads=0):
    with _cabi.Fasta(str(path), n_threads=threads) as fa:
        tb = fa.twobit()
        runs = tb.runs.copy()
        return fa.format, fa.bases.tobytes(), fa.offsets.copy(), [n.encode() for n in fa.names], runs


def check_file(path, recs, threads=(1, 16)):
    text, offsets, names, runs = expected(recs)
    for t in threads:
        fmt, got_text, got_off, got_names, got_runs = read_back(path, t)
        assert fmt == "2bit"
        assert got_text == text, t
        assert np.array_equal(got_off, offsets) and got_names == names
        assert np.array_equal(got_runs, runs)


# ---- CPU: the reader ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("swap,version", [(False, 0), (True, 0), (False, 1), (True, 1)])
def test_reader_alignments_blocks_byte_orders_versions(tmp_path, swap, version):
    rng = random.Random(10 + 2 * swap + version)
    recs = alignment_recs(rng)
    order = list(range(len(recs)))
    rng.shuffle(order)                                             # data in another order than the index
    for o in (None, order):
        path = tmp_path / "a.2bit"
        path.write_bytes(twobit_bytes(recs, swap=swap, version=version, order=o))
        check_file(path, recs)


def test_reader_hand_made_blocks(tmp_path):
    """N and mask blocks at record ends, overlapping, unsorted and adjacent across records; 'n' inside both kinds."""
    recs = [Rec(b"a", 10, pack_codes("TCAGTCAGTC"), [(8, 2), (2, 3), (3, 4)], [(0, 3), (9, 1), (1, 1)]),
            Rec(b"b", 5, pack_codes("GGGGG"), [(0, 2)], [(0, 5)]),
            Rec(b"empty", 0, b""),
            Rec(b"c", 4, pack_codes("ACGT"), [(0, 0)], [(4, 0)])]
    path = tmp_path / "h.2bit"
    path.write_bytes(twobit_bytes(recs))
    fmt, text, offsets, names, runs = read_back(path)
    assert text == b"tcnNNNNGNn" + b"nnggg" + b"" + b"ACGT"
    assert offsets.tolist() == [0, 10, 15, 15, 19] and names == [b"a", b"b", b"empty", b"c"]
    assert runs.tolist() == [[2, 7], [8, 10], [10, 12]]            # merged within a record, not across records
    check_file(path, recs)


def test_reader_many_short_records(tmp_path):
    """10^6 short records (the index walk and the decode across many records per piece)."""
    rng = np.random.default_rng(3)
    n = 10 ** 6
    sizes = rng.integers(0, 12, n)
    letters = "".join(rng.choice(list("TCAG"), int(sizes.sum())))
    recs, at = [], 0
    for i, z in enumerate(sizes.tolist()):
        nb = [(0, 1)] if z and i % 7 == 0 else []
        mb = [(z - 1, 1)] if z and i % 5 == 0 else []
        recs.append(Rec(b"s%d" % i, z, pack_codes(letters[at:at + z]), nb, mb))
        at += z
    path = tmp_path / "many.2bit"
    path.write_bytes(twobit_bytes(recs, version=1))
    check_file(path, recs)


def test_reader_file_larger_than_one_piece(tmp_path):
    """One record of 11 M bases (several decode pieces) with N and mask blocks across the piece boundaries."""
    rng = np.random.default_rng(4)
    n = 11_000_003
    letters = np.frombuffer(b"TCAG", np.uint8)[rng.integers(0, 4, n)].tobytes().decode()
    nb = [(4_194_300, 10), (8_388_600, 20), (n - 5, 5)]
    mb = [(0, 4_194_310), (6_000_000, 3_000_000)]
    recs = [Rec(b"big", n, pack_codes(letters), nb, mb), rec_from_text(b"tail", "ACGTNNacgtnn")]
    path = tmp_path / "big.2bit"
    path.write_bytes(twobit_bytes(recs))
    check_file(path, recs)


def _bad_cases():
    good = [rec_from_text(b"one", "ACGTACGTNNNNacgt"), rec_from_text(b"two", "GATTACA"), rec_from_text(b"three", "CCCC")]
    blob = twobit_bytes(good)
    index_end = 16 + sum(1 + len(r.name) + 4 for r in good)
    rec2_off = struct.unpack_from("<I", blob, 16 + 1 + 3 + 4 + 1 + 3)[0]
    cases = [("truncated index", blob[:16 + 1 + 3 + 4 + 2], 2, "index is truncated")]
    b = bytearray(blob)
    struct.pack_into("<I", b, 16 + 1 + 3 + 4 + 1 + 3, len(blob) + 10)
    cases.append(("offset past the end", bytes(b), 2, "offset is past the end"))
    bad_block = [good[0], Rec(b"two", 7, good[1].packed, [(5, 3)]), good[2]]
    cases.append(("N block past dnaSize", twobit_bytes(bad_block), 2, "N block ends past its dnaSize"))
    bad_mask = [good[0], good[1], Rec(b"three", 4, good[2].packed, [], [(4, 1)])]
    cases.append(("mask block past dnaSize", twobit_bytes(bad_mask), 3, "mask block ends past its dnaSize"))
    cases.append(("shorter than its DNA", blob[:-1], 3, "shorter than its DNA"))
    b = bytearray(blob)
    struct.pack_into("<I", b, rec2_off + 4, 1 << 30)                 # an N block count past the end of the file
    cases.append(("block count", bytes(b), 2, "N blocks run past the end"))
    b = bytearray(blob)
    struct.pack_into("<I", b, 16 + 1 + 3 + 4 + 1 + 3, struct.unpack_from("<I", blob, 16 + 1 + 3)[0])   # two records, one place
    cases.append(("overlapping records", bytes(b), 2, "overlap those of record 1"))
    assert index_end < rec2_off
    return cases


@pytest.mark.parametrize("what,blob,record,why", _bad_cases(), ids=[c[0] for c in _bad_cases()])
def test_reader_errors_name_the_record(tmp_path, what, blob, record, why):
    path = tmp_path / "bad.2bit"
    path.write_bytes(blob)
    with pytest.raises(ValueError, match=rf"\.2bit record {record}: .*{why}"):
        _cabi.Fasta(str(path))


def test_reader_header_errors(tmp_path):
    blob = twobit_bytes([rec_from_text(b"x", "ACGT")])
    for data, why in ((blob[:4] + struct.pack("<I", 2) + blob[8:], "version 2"), (blob[:12], "header is truncated")):
        (tmp_path / "h.2bit").write_bytes(data)
        with pytest.raises(ValueError, match=why):
            _cabi.Fasta(str(tmp_path / "h.2bit"))


def test_index_and_packed_form_without_decoding(tmp_path):
    """offsets, names and the packed form come from the index; bases decodes on first use; other formats refuse
    crf_fasta_twobit."""
    recs = [rec_from_text(b"chr1", "ACGTNNNNacgtAC"), rec_from_text(b"chr2", "TTTT")]
    blob = twobit_bytes(recs)
    (tmp_path / "g.2bit").write_bytes(blob)
    with _cabi.Fasta(str(tmp_path / "g.2bit"), pinned=2) as fa:
        assert fa._bases is None and fa.names == ["chr1", "chr2"] and fa.offsets.tolist() == [0, 14, 18]
        tb = fa.twobit()
        assert tb.dna.tobytes() == blob[:tb.dna.size] and tb.dna.size == len(blob)
        assert [blob[b:b + 2] for b in tb.rec_byte.tolist()] == [recs[0].packed[:2], recs[1].packed[:2]]
        assert fa._bases is None
        assert fa.bases.tobytes() == b"ACGTNNNNacgtACTTTT"
    (tmp_path / "g.fa").write_bytes(b">chr1\nACGT\n")
    with _cabi.Fasta(str(tmp_path / "g.fa")) as fa:
        assert fa.format == "fasta"
        with pytest.raises(ValueError, match="not a .2bit file"):
            fa.twobit()


def test_existing_callers_read_the_decoded_text(tmp_path):
    """crf_fasta_packed and read_fasta work on a .2bit handle through its decoded text."""
    from crf_b200 import fasta
    from tests.fake_ctx import unpack_planes
    rng = random.Random(12)
    recs = alignment_recs(rng)
    (tmp_path / "g.2bit").write_bytes(twobit_bytes(recs))
    text, _, names, _ = expected(recs)
    with _cabi.Fasta(str(tmp_path / "g.2bit")) as fa:
        assert unpack_planes(fa.packed()).tobytes() == bytes(text).upper()
    got = fasta.read_fasta(str(tmp_path / "g.2bit"))
    assert [r.name.encode() for r in got] == names and b"".join(r.seq for r in got) == text


def test_twobit_harness_under_sanitizers(tmp_path):
    """tests/fuzz_twobit.cpp: random .2bit files (both byte orders and versions) read on 1 and 5 threads against a C++
    statement of twoBitToFa, headers with flipped bytes (every outcome an answer or CRF_ERR_ARG, never a fault), and
    crf_write_rows_twobit against crf_write_rows, without the CUDA runtime, under AddressSanitizer and UBSan."""
    if not shutil.which("g++"):
        pytest.skip("no g++")
    exe = str(tmp_path / "fuzz_twobit")
    built = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                            "-pthread", "-I", os.path.join(ROOT, "colab-repeat-finder_b200", "csrc"),
                            "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "fuzz_twobit.cpp"), "-o", exe,
                            "-lz"], capture_output=True, text=True)
    assert built.returncode == 0, built.stderr[-4000:]
    run = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=600,
                         env={**os.environ, "ASAN_OPTIONS": "detect_leaks=1"})
    assert run.returncode == 0 and run.stdout.startswith("ok "), (run.stdout[-2000:], run.stderr[-4000:])


# ---- CPU: the rows writer -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tsv", [False, True])
def test_rows_twobit_equals_rows_on_the_text(tmp_path, tsv):
    """150 000 rows (several formatting threads and waves): byte-identical to crf_write_rows on the decoded text."""
    rng = np.random.default_rng(8)
    recs = []
    for i in range(40):
        n = int(rng.integers(0, 30000))
        text = np.frombuffer(b"ACGTacgt", np.uint8)[rng.integers(0, 8, n)].tobytes().decode()
        recs.append(rec_from_text(b"chr%d" % i, text))
    path = tmp_path / "w.2bit"
    path.write_bytes(twobit_bytes(recs, order=list(range(39, -1, -1))))
    with _cabi.Fasta(str(path)) as fa:
        tb = fa.twobit()
        lengths = np.diff(fa.offsets.astype(np.int64))
        m = 150_000
        rec = np.sort(rng.choice(np.flatnonzero(lengths > 60), m))
        k = rng.integers(1, 51, m)
        start = (rng.random(m) * (lengths[rec] - k)).astype(np.int64)
        end = np.minimum(start + k * rng.integers(1, 4, m), lengths[rec])
        names = None if tsv else fa.names_blob
        a = _cabi.write_rows(str(tmp_path / "a"), names, fa.bases, fa.offsets, rec, start, end, k, tsv=tsv)
        b = _cabi.write_rows_twobit(str(tmp_path / "b"), names, tb.dna, tb.rec_byte, rec, start, end, k, tsv=tsv)
        a2 = _cabi.write_rows(str(tmp_path / "a"), names, fa.bases, fa.offsets, rec[:10], start[:10], end[:10], k[:10],
                              tsv=tsv, append=True)
        b2 = _cabi.write_rows_twobit(str(tmp_path / "b"), names, tb.dna, tb.rec_byte, rec[:10], start[:10], end[:10], k[:10],
                                     tsv=tsv, append=True)
    assert (a, a2) == (b, b2)
    assert (tmp_path / "a").read_bytes() == (tmp_path / "b").read_bytes() and a > 3_000_000


# ---- CPU: the command line with stand-ins -------------------------------------------------------------------------------

def _stand_in_load_2bit(self, source, max_motif_cap=50, on_device=False):
    """The .2bit load as a stand-in: decode the bytes (the Python statement above) and load the text."""
    if isinstance(source, _cabi.Fasta):
        source = source.twobit()
    dna = np.asarray(source.dna)
    texts = []
    for b, n in zip(source.rec_byte.tolist(), np.diff(source.offsets.astype(np.int64)).tolist()):
        p = dna[b:b + (n + 3) // 4]
        codes = np.stack([(p >> 6) & 3, (p >> 4) & 3, (p >> 2) & 3, p & 3], 1).reshape(-1)[:n]
        texts.append(np.frombuffer(b"TCAG", np.uint8)[codes])
    text = np.concatenate(texts + [np.zeros(0, np.uint8)])
    pos0 = int(source.offsets[0])
    for a, b in source.runs.tolist():
        a, b = max(a, pos0) - pos0, min(b, int(source.offsets[-1])) - pos0
        if a < b:
            text[a:b] = ord("N")
    TwoBitMaskContext.loads_2bit += 1
    return self.load(text, source.offsets - source.offsets[0], max_motif_cap)


class TwoBitMaskContext(MaskContext):
    loads_2bit = 0
    load_2bit = _stand_in_load_2bit


class TwoBitStopContext(StopContext):
    load_2bit = _stand_in_load_2bit


def _glue_records(rng):
    texts = [("chrA", random_seq(rng, 3000)), ("chrB", random_seq(rng, 50)), ("empty", ""),
             ("chrC", random_seq(rng, 7000)), ("chrD", ("acgt" * 30 + "AC" * 40) * 9), ("chrE", "N" * 30 + "ACAC" * 20 + "n" * 9)]
    texts += [(f"read{i}", random_seq(rng, rng.randint(0, 150))) for i in range(300)]
    # .2bit holds only ACGTN and case: other letters become N, as faToTwoBit writes them
    return [(n, "".join(c if c in "ACGTNacgtn" else ("n" if c.islower() else "N") for c in s)) for n, s in texts]


def _fasta_bytes(records):
    return b"".join(b">" + n.encode() + b"\n" + s.encode() + b"\n" for n, s in records)


def _run(capsys, argv):
    assert cli.main(argv) == 0
    return capsys.readouterr().out


def _write_pair(tmp_path, records, stem="g"):
    (tmp_path / f"{stem}.fa").write_bytes(_fasta_bytes(records))
    (tmp_path / f"{stem}.2bit").write_bytes(twobit_bytes([rec_from_text(n.encode(), s) for n, s in records], version=1))


def _single_copy_ok(text):
    try:
        oracle.detect_repeats(text.encode(), ns(min_motif_size=1, max_motif_size=8, min_repeats=1, min_span=4))
        return True
    except IndexError:
        return False


def test_cli_twobit_bed_equals_fasta_bed(tmp_path, monkeypatch, capsys):
    """BED and stdout of a .2bit file equal those of its FASTA: one load, several load groups, a record longer than a
    load (the decoded text's path), and --min-repeats 1."""
    rng = random.Random(21)
    records = _glue_records(rng)
    _write_pair(tmp_path, records)
    monkeypatch.setattr(api, "get_context", lambda device=None: TwoBitMaskContext())
    monkeypatch.setattr(api, "detect_repeats", lambda seq, fs, device=None: oracle.detect_repeats(seq, fs))
    monkeypatch.chdir(tmp_path)
    real_limit = _cabi.load_limit(12)
    for extra in (["-max", "12"], ["-max", "8", "--min-repeats", "1", "--min-span", "4"]):
        # (--min-repeats 1 as the reference runs it raises IndexError on some short or N-rich records: not those)
        recs = records if len(extra) == 2 else [r for r in records if _single_copy_ok(r[1])]
        _write_pair(tmp_path, recs)
        for limit in (real_limit, 7100, 3500, 1):
            monkeypatch.setattr(_cabi, "load_limit", lambda cap, limit=limit: limit)
            TwoBitMaskContext.loads_2bit = 0
            outs, beds = [], []
            for src in ("g.fa", "g.2bit"):
                outs.append(_run(capsys, [str(tmp_path / src), "-o", "out"] + extra))
                beds.append((tmp_path / "out.bed").read_bytes())
            assert beds[0] == beds[1] and len(beds[0]) > 1000, (extra, limit)
            assert outs[0] == outs[1]
            if len(extra) == 2:                    # the packed path (one load per group) unless a record exceeds a load
                assert TwoBitMaskContext.loads_2bit == 1 if limit == real_limit else (TwoBitMaskContext.loads_2bit > 1) == (limit == 7100)
            if len(extra) > 2:
                break


def test_cli_twobit_interval_and_intervals(tmp_path, monkeypatch, capsys, stand_ins):
    rng = random.Random(22)
    records = _glue_records(rng)
    _write_pair(tmp_path, records)
    monkeypatch.setattr(api, "get_context", lambda device=None: TwoBitStopContext())
    (tmp_path / "l.bed").write_text("chrA\t100\t2000\nread3\t0\t100\nchrD\t5\t400\nchrA\t0\t50\n")
    monkeypatch.chdir(tmp_path)
    for opt in (["-i", "chrA:100-2000"], ["-i", "chrD:0-400"], ["--intervals", str(tmp_path / "l.bed")]):
        outs, beds = [], []
        for src in ("g.fa", "g.2bit"):
            outs.append(_run(capsys, [str(tmp_path / src), "-max", "10", "-o", "o"] + opt))
            beds.append((tmp_path / "o.bed").read_bytes())
        assert beds[0] == beds[1] and len(beds[0]) > 50, opt
        assert outs[0] == outs[1]


@pytest.mark.parametrize("kind", ["soft", "hard"])
def test_cli_mask_on_twobit(tmp_path, monkeypatch, capsys, kind):
    """--mask on .2bit writes <prefix>.masked.fa from the decoded text: the same file its FASTA gives."""
    rng = random.Random(23)
    records = _glue_records(rng)
    _write_pair(tmp_path, records)
    monkeypatch.setattr(api, "get_context", lambda device=None: TwoBitMaskContext())
    monkeypatch.chdir(tmp_path)
    for limit in (None, 3500):
        if limit:
            monkeypatch.setattr(_cabi, "load_limit", lambda cap: limit)
        fa_out = _run(capsys, [str(tmp_path / "g.fa"), "-max", "12", "--mask", kind])
        fa_bed, fa_masked = (tmp_path / "g.bed").read_bytes(), (tmp_path / "g.masked.fa").read_bytes()
        tb_out = _run(capsys, [str(tmp_path / "g.2bit"), "-max", "12", "--mask", kind])
        assert (tmp_path / "g.bed").read_bytes() == fa_bed and tb_out == fa_out
        assert (tmp_path / "g.masked.fa").read_bytes() == fa_masked
        names = [n.encode() for n, _ in records]
        masks = mask_from_bed(fa_bed.decode(), [n for n, _ in records], [s.encode() for _, s in records])
        assert sum(int(m.sum()) for m in masks) > 500
        assert fa_masked == masked_fasta(names, [s.encode() for _, s in records], masks, kind == "hard")


def test_cli_default_prefix_for_twobit(tmp_path, monkeypatch, capsys):
    monkeypatch.setattr(api, "get_context", lambda device=None: TwoBitMaskContext())
    monkeypatch.chdir(tmp_path)
    (tmp_path / "in").mkdir()
    blob = twobit_bytes([rec_from_text(b"r1", "ACACACACACACAC")])
    for name, bed in (("hg38.2bit", "hg38.bed"), ("hs1.2bit", "hs1.bed"), ("x.2bit.bak", "x.2bit.bak.bed"),
                      ("genome", "genome.bed"), ("my.fa.2bit", "my.fa.bed")):
        (tmp_path / "in" / name).write_bytes(blob)
        out = _run(capsys, [str(tmp_path / "in" / name)])
        assert out.endswith(f"Wrote results to {bed}\n"), name
        assert (tmp_path / bed).read_text() == "r1\t0\t14\tAC\n"
        os.remove(tmp_path / bed)
    assert cli.default_prefix("a.fa.2bit", "2bit") == "a.fa" and cli.default_prefix("a.2bit", "fasta") == "a.2bit"


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


def _check_load(path, with_oracle=True, tensor=False):
    ctx = api.get_context()
    with _cabi.Fasta(str(path), pinned=2) as fa:
        tb = fa.twobit()
        if tensor:
            import torch
            tb = _cabi.TwoBitSource(torch.from_numpy(np.fromfile(str(path), np.uint8)).cuda(), tb.rec_byte, tb.offsets, tb.runs)
        with ctx.load_2bit(tb) as seq:
            got = _rows(seq)
        text = fa.bases.tobytes()
        with ctx.load(fa.bases, fa.offsets) as seq:
            want = _rows(seq)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    if with_oracle:
        for a, b in zip(got, _oracle_rows(text, fa.offsets)):
            assert np.array_equal(a.astype(np.int64), b)
    return len(got[0])


def _repeat_rich(rng, n):
    parts, at = [], 0
    while at < n:
        unit = "".join(rng.choice("ACGT") for _ in range(rng.randint(1, 12)))
        p = unit * rng.randint(1, 8) + "".join(rng.choice("ACGTacgt") for _ in range(rng.randint(0, 40)))
        parts.append(p)
        at += len(p)
    return "".join(parts)[:n]


@pytest.mark.gpu
def test_gpu_alignment_cases_equal_ascii_load_and_oracle(tmp_path):
    rng = random.Random(30)
    recs = []
    for i, n in enumerate(list(range(10)) + list(range(28, 37)) + list(range(60, 69)) + [500, 3000, 0, 7, 20000]):
        text = _repeat_rich(rng, n)
        r = rec_from_text(b"r%d" % i, text)
        if n > 20:
            r.nblocks += [(rng.randint(0, n - 5), rng.randint(0, 5)), (n - 1, 1)]
        recs.append(r)
    for swap, version in ((False, 0), (True, 1)):
        order = list(range(len(recs)))
        rng.shuffle(order)
        for o in (None, order):
            path = tmp_path / "a.2bit"
            path.write_bytes(twobit_bytes(recs, swap=swap, version=version, order=o))
            assert _check_load(path) > 200
    assert _check_load(path, tensor=True) > 200                    # the file's bytes as a CUDA tensor


@pytest.mark.gpu
def test_gpu_million_reads(tmp_path):
    """10^6 reads of 150 bp, some with N's."""
    rng = np.random.default_rng(31)
    n, rl = 10 ** 6, 150
    unit = rng.integers(0, 4, (n, 6))
    reads = np.frombuffer(b"TCAG", np.uint8)[np.where(rng.random((n, rl)) < 0.7, np.tile(unit, 25), rng.integers(0, 4, (n, rl)))]
    recs = []
    for i in range(n):
        row = reads[i].tobytes()
        nb = [(int(rng.integers(0, rl)), 1)] if i % 9 == 0 else []
        recs.append(Rec(b"q%d" % i, rl, pack_codes(row.decode()), nb, [(0, 10)] if i % 4 == 0 else []))
    path = tmp_path / "reads.2bit"
    path.write_bytes(twobit_bytes(recs))
    assert _check_load(path, with_oracle=False) > 300_000
    assert _check_load(path, with_oracle=False, tensor=True) > 300_000


@pytest.mark.gpu
def test_gpu_pipelined_upload(tmp_path):
    """A span of 1.2 G positions (300 MB of bytes: the chunked upload on the second stream), compared with the ASCII load;
    the oracle on one record."""
    rng = np.random.default_rng(32)
    recs = []
    for i in range(6):
        n = 200_000_001 + i
        codes = rng.integers(0, 4, n // 8 + 1).astype(np.uint8)
        c = np.repeat(codes, 8)[:n]
        pad = np.concatenate([c, np.zeros((-n) % 4, np.uint8)]).reshape(-1, 4)
        packed = ((pad[:, 0] << 6) | (pad[:, 1] << 4) | (pad[:, 2] << 2) | pad[:, 3]).astype(np.uint8).tobytes()
        recs.append(Rec(b"big%d" % i, n, packed, [(1000, 5000), (n - 77, 77)], [(0, 100_000)]))
    recs.append(rec_from_text(b"small", _repeat_rich(random.Random(3), 5000)))
    path = tmp_path / "big.2bit"
    path.write_bytes(twobit_bytes(recs))
    assert _check_load(path, with_oracle=False) > 10 ** 6
    with _cabi.Fasta(str(path)) as fa, api.get_context().load_2bit(fa.twobit().records(6, 7)) as seq:
        got = _rows(seq)
        text = fa.record(6).tobytes()
    for a, b in zip(got, _oracle_rows(text, [0, len(text)])):
        assert np.array_equal(a.astype(np.int64), b)


def s38_twobit(path):
    """S38 written as a .2bit file (S38 holds only ACGTN, soft mask and N runs: it converts exactly).  Packed on the GPU."""
    import torch
    from crf_b200 import synth
    bases, offsets, meta = synth.s38(device="cuda:0")
    lut = torch.zeros(256, dtype=torch.uint8, device=bases.device)
    for c, v in CODE.items():
        lut[ord(c)] = v
        lut[ord(c.lower())] = v
    recs = []
    for r in range(len(offsets) - 1):
        t = bases[int(offsets[r]):int(offsets[r + 1])]
        up = t & 0xDF
        assert bool((((up == 65) | (up == 67) | (up == 71) | (up == 84) | (up == 78))).all())
        c = lut[t.long()]
        n = t.numel()
        c = torch.cat([c, torch.zeros((-n) % 4, dtype=torch.uint8, device=c.device)]).view(-1, 4)
        packed = ((c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]).cpu().numpy().tobytes()
        isn = (up == 78).cpu().numpy()
        low = (t >= 97).cpu().numpy()
        recs.append(Rec(meta["names"][r].encode(), n, packed, runs_of(isn), runs_of(low)))
    with open(path, "wb") as f:
        f.write(twobit_bytes(recs))
    return bases, offsets, meta


@pytest.mark.gpu
def test_s38_as_twobit_gives_the_golden_rows_and_the_fasta_bed(tmp_path, monkeypatch, capsys):
    bases, offsets, meta = s38_twobit(tmp_path / "S38.2bit")
    with _cabi.Fasta(str(tmp_path / "S38.2bit"), pinned=2) as fa, api.get_context().load_2bit(fa) as seq:
        n = seq.scan(1, 50, 3, 9)
        rows = seq.fetch(n)
    sha = hashlib.sha256()
    for a in rows:
        sha.update(np.ascontiguousarray(a, dtype=np.uint32).tobytes())
    with open(os.path.join(ROOT, "tests", "golden", "workload_rows_sha256.json")) as f:
        assert json.load(f)["s38:1.0:1-50"] == sha.hexdigest()
    host = bases.cpu().numpy()
    with open(tmp_path / "S38.fa", "wb") as f:
        for r, name in enumerate(meta["names"]):
            f.write(b">" + name.encode() + b"\n")
            f.write(host[int(offsets[r]):int(offsets[r + 1])].tobytes())
            f.write(b"\n")
    del host, bases
    monkeypatch.chdir(tmp_path)
    import torch
    runs = [[]] + ([["--devices", "0-1"]] if torch.cuda.device_count() >= 2 else [])
    for extra in runs:
        outs, beds = [], []
        for src in ("S38.fa", "S38.2bit"):
            outs.append(_run(capsys, [str(tmp_path / src), "-o", "out"] + extra))
            bed = (tmp_path / "out.bed").read_bytes()
            beds.append((len(bed), hashlib.sha256(bed).hexdigest()))
            del bed
        assert outs[0] == outs[1]
        assert beds[0] == beds[1] and beds[0][0] > 100_000_000, extra
