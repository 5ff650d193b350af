"""FASTA input through the library's native reader (crf_fasta_open), standing in for pyfastx
(perfect_repeat_finder.py:117-137 uses only `.name` -- the first whitespace-delimited token of the header --
and `.seq`, the record's lines joined without line ends, case preserved).  Plain or gzip input.  A FASTQ file (first
byte that is not whitespace: '@') is read too: read names and sequences in the same layout, qualities on request.  So is a
UCSC .2bit file, whose text (what twoBitToFa writes) is decoded on first use of `bases`, and an unaligned BAM file (the
reads `samtools fastq -n` writes from it, kept as 4-bit codes until `bases` is first used)."""
import os

from . import _cabi


class FastaRecord:
    __slots__ = ("name", "seq")

    def __init__(self, name, seq):
        self.name = name      # str
        self.seq = seq        # uint8 view into the file's base buffer, one byte per base, case preserved


def open_fasta(path, pinned=False, qualities=False):
    """The whole file as a _cabi.Fasta (bases back to back + offsets + names; a FASTQ file's qualities in .quals when
    `qualities`)."""
    if not os.path.isfile(path):
        raise FileNotFoundError(path)
    return _cabi.Fasta(path, pinned=pinned, qualities=qualities)


def read_fasta(path):
    """All records of a FASTA or FASTQ file, in file order, as (name, bytes) records."""
    with open_fasta(path) as fa:
        return [FastaRecord(name, fa.record(i).tobytes()) for i, name in enumerate(fa.names)]
