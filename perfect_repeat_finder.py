"""Drop-in module for the reference's perfect_repeat_finder.py (same module name, same
detect_repeats() signature, same CLI).  The work is done by the B200 kernels in
colab-repeat-finder_b200/ (package crf_b200)."""
import os
import sys

_PKG_PARENT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "colab-repeat-finder_b200")
if _PKG_PARENT not in sys.path:
    sys.path.insert(0, _PKG_PARENT)

from crf_b200.api import detect_repeats  # noqa: E402,F401
from crf_b200.intervals import detect_repeats_intervals  # noqa: E402,F401
from crf_b200.batch import detect_repeats_batch, scan_batch  # noqa: E402,F401
from crf_b200.mask import repeat_mask  # noqa: E402,F401


def main(argv=None):
    from crf_b200.cli import main as _main
    return _main(argv)


if __name__ == "__main__":
    main()
