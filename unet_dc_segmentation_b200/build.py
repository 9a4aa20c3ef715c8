"""In-tree build of libunetdc_b200.so (nvcc, sm_100a only).

The shared library is the product's only compute path; it is built next to the sources so that it
travels with the repo snapshot to the GPU box (a JIT cache under ~/.cache would not).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "lib"
LIB_PATH = LIB_DIR / "libunetdc_b200.so"
SOURCES = ["api.cu", "conv_tc.cu", "morph.cu", "ccl.cu", "resize.cu", "density.cu", "generic.cu", "csv.cu", "png.cu"]
HEADERS = [CSRC / "common.cuh", CSRC / "upf_schedule.inc", CSRC / "csv_tables.inc", PKG.parent / "include" / "unetdc_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
]


def find_nvcc() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(cand).exists():
        raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc); the CUDA library cannot be built")
    return cand


HASH_PATH = LIB_DIR / "libunetdc_b200.so.srchash"


def source_hash() -> str:
    """Content hash of everything that goes into the library (file times do not survive a repo snapshot)."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for d in [CSRC / s for s in SOURCES] + HEADERS:
        h.update(d.name.encode())
        h.update(d.read_bytes())
    return h.hexdigest()


def is_stale() -> bool:
    if not LIB_PATH.exists() or not HASH_PATH.exists():
        return True
    return HASH_PATH.read_text().strip() != source_hash()


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every .cu of the package into lib/libunetdc_b200.so (separate objects, then link)."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = find_nvcc()
    LIB_DIR.mkdir(exist_ok=True)
    # several ranks may import the package at once (torchrun): one builds, the others wait and then find it fresh
    import fcntl
    lock = open(LIB_DIR / ".build.lock", "w")
    fcntl.flock(lock, fcntl.LOCK_EX)
    try:
        if not force and not is_stale():
            return LIB_PATH
        return _build_locked(nvcc, verbose)
    finally:
        fcntl.flock(lock, fcntl.LOCK_UN)
        lock.close()


def _build_locked(nvcc: str, verbose: bool) -> Path:
    obj_dir = PKG / "build" / f"obj_{os.getpid()}"
    obj_dir.mkdir(parents=True, exist_ok=True)
    procs = []
    objs = []
    for s in SOURCES:
        o = obj_dir / (s[:-3] + ".o")
        objs.append(str(o))
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / s), "-o", str(o)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
    tmp = LIB_PATH.with_suffix(".so.tmp")
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(tmp), *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB_PATH)
    HASH_PATH.write_text(source_hash() + "\n")
    shutil.rmtree(obj_dir, ignore_errors=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
