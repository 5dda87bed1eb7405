"""In-tree build of libvggp.so (sm_100a only; nvcc cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvggp.so")
SOURCES = ["vggp.cu"]
HEADERS = ["common.cuh", "gemm.cuh", "grid.cuh", "obs.cuh", "obs_binned.cuh", "binplan.hpp", "metrics.cuh", "b0scan.cuh", "svgpm.cuh", "meanopt.cuh", "covopt.cuh", "collapsed.cuh", "minibatch.cuh", "grid_b1.cuh", "grid_b1_fast.cuh", "collective.cuh", os.path.join("..", "..", "include", "vggp.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into libvggp.so next to this file.  Returns the library path."""
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libvggp.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
