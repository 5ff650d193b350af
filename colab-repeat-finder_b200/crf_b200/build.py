"""Build libcrf.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(_HERE), "csrc")
OUT = os.path.join(_HERE, "libcrf.so")
SOURCES = ["crf_api.cu"]
HEADERS = ["crf_device.cuh", "crf_scan.cuh", "crf_scan_warp.cuh", "crf_aux.cuh", "crf_stop.cuh", "crf_xchg.cuh", "crf_fasta.h", "crf_codes.h", "crf_pack.h", "crf_inflate.h", "crf_rows.h", "crf_mask.cuh", "crf_fasta_out.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-cudart", "shared", "-Xcompiler", "-fPIC,-pthread"]   # cudart linked dynamically: the runtime's own
                                                                               # symbol table stays out of the shipped .so
LINK_FLAGS = ["-lz"]


TOOLS_OUT = os.path.join(_HERE, "libcrf_tools.so")   # bench-only helpers (INT32 peak micro-benchmark)
TOOLS_SOURCES = ["crf_tools.cu"]


def _stale(out, deps):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def _nvcc_path():
    return os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def have_nvcc():
    return os.path.exists(_nvcc_path())


def _nvcc(out, sources, verbose):
    nvcc = _nvcc_path()
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + \
          [os.path.join(CSRC, f) for f in sources] + LINK_FLAGS
    subprocess.check_call(cmd)


def build(force=False, verbose=False):
    """libcrf.so (the product) and libcrf_tools.so (bench helpers)."""
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(os.path.dirname(os.path.dirname(_HERE)), "include", "crf.h"))
    if force or _stale(OUT, deps):
        _nvcc(OUT, SOURCES, verbose)
    tdeps = [os.path.join(CSRC, f) for f in TOOLS_SOURCES]
    if force or _stale(TOOLS_OUT, tdeps):
        _nvcc(TOOLS_OUT, TOOLS_SOURCES, verbose)
    return OUT


if __name__ == "__main__":
    print(build(force=True, verbose=True))
