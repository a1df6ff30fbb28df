"""Builds libneo360_b200.so in-tree with nvcc for sm_100a (no torch headers: the library is a plain C ABI)."""
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
HEADER = os.path.join(HERE, "..", "include", "neo360_b200.h")
LIB = os.path.join(HERE, "libneo360_b200.so")
STAMP = LIB + ".sha256"        # _source_hash() of the sources LIB was built from
SOURCES = ["scene.cu", "sampling.cu", "field_fp32.cu", "field_tc.cu", "render.cu", "vanilla.cu", "mip.cu", "gemm_tc.cu", "encoder.cu"]
FLAGS = ["-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
         "-std=c++17", "--threads", "4"]


def _source_hash() -> str:
    """sha256 of the flags, every file under csrc/ and the public header."""
    h = hashlib.sha256(" ".join(FLAGS + SOURCES).encode())
    for path in [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [HEADER]:
        with open(path, "rb") as f:
            h.update(os.path.basename(path).encode() + b"\0" + f.read())
    return h.hexdigest()


def _stale(digest: str) -> bool:
    # content, not mtimes: a copied or freshly checked-out tree keeps a library built from the same sources
    try:
        with open(STAMP) as f:
            return not os.path.exists(LIB) or f.read().strip() != digest
    except FileNotFoundError:
        return True


def build(force: bool = False, verbose: bool = False) -> str:
    """Returns the path of a library built from the current sources, compiling one if LIB is missing or stale.  A tree
    that is not writable is left untouched: the library is then compiled into a new temporary directory (load it with
    `_lib.load(path)`)."""
    digest = _source_hash()
    if not force and not _stale(digest):
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libneo360_b200.so must be prebuilt")
    out = LIB if os.access(HERE, os.W_OK) else os.path.join(tempfile.mkdtemp(prefix="neo360_b200-"), os.path.basename(LIB))
    tmp = f"{out}.{os.getpid()}.tmp"      # per process: ranks that decide to build at the same time do not write into each other's file
    cmd = [nvcc] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    os.replace(tmp, out)   # atomic: a concurrent reader never sees a half-written library
    if out == LIB:
        with open(tmp, "w") as f:
            f.write(digest)
        os.replace(tmp, STAMP)
    if verbose:
        print(res.stderr)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
