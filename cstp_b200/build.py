"""Builds libcstp_b200.so (hand-written sm_100a kernels + the C ABI of include/cstp_b200.h) in-tree with nvcc.

The shared library links the CUDA runtime statically and resolves the one driver symbol it needs
(cuTensorMapEncodeTiled) through cudaGetDriverEntryPoint, so it loads on a machine without a GPU driver.
"""
from __future__ import annotations

import fcntl
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "libcstp_b200.so"
OBJ_DIR = PKG_DIR / "_build"

SOURCES = ["common.cu", "conv_gemm.cu", "conv_halo.cu", "wgrad.cu", "wgrad_halo.cu", "elementwise.cu", "loss_optim.cu", "ntxent_tc.cu",
           "clip_pipeline.cu", "p2p_sync.cu", "video_eval.cu", "retrieval.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _digest() -> str:
    h = hashlib.sha256()
    for p in sorted(CSRC.glob("*")) + [PKG_DIR.parent / "include" / "cstp_b200.h"]:
        h.update(p.name.encode())
        h.update(p.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_stale() -> bool:
    """True when the library was built here from other sources than the ones in the tree (a library that arrived without
    its stamp -- a snapshot of built artefacts -- is taken as it is)."""
    stamp = OBJ_DIR / "stamp"
    return LIB_PATH.exists() and stamp.exists() and stamp.read_text() != _digest()


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every .cu for sm_100a and link libcstp_b200.so. Skips work when sources are unchanged.  Serialised over
    processes by a file lock (ranks of one torchrun launch), the library is moved into place atomically."""
    OBJ_DIR.mkdir(exist_ok=True)
    with open(OBJ_DIR / "lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force: bool, verbose: bool) -> Path:
    stamp = OBJ_DIR / "stamp"
    digest = _digest()
    if not force and LIB_PATH.exists() and stamp.exists() and stamp.read_text() == digest:
        return LIB_PATH
    nvcc = _nvcc()

    def compile_one(src: str) -> tuple[str, str]:
        obj = OBJ_DIR / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return str(obj), r.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    (OBJ_DIR / "ptxas.log").write_text("\n".join(log for _, log in results))
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    tmp = LIB_PATH.with_suffix(f".so.tmp{os.getpid()}")
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(tmp), *[o for o, _ in results]]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB_PATH)
    stamp.write_text(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
