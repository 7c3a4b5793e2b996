"""In-tree build of libemr2a.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m emr2a_b200.build [--force]

The shared library lands next to this file (git-ignored, but it travels to the
GPU box with the gpurun snapshot).
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
OUT = os.path.join(PKG, "libemr2a.so")
OBJ = os.path.join(PKG, "build")
SOURCES = ["api.cu", "normalize_fuse.cu", "simt_paths.cu", "merge_vote.cu", "topk_tc.cu", "topk_tc2.cu", "rescore.cu", "preprocess.cu", "late_fusion.cu",
           "components.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr",
]


def _stamp() -> str:
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)) + ["../../include/emr2a.h"]:
        with open(os.path.join(CSRC, name), "rb") as fh:
            h.update(name.encode())
            h.update(fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def _up_to_date(stamp_file: str, stamp: str) -> bool:
    if os.path.exists(OUT) and os.path.exists(stamp_file):
        with open(stamp_file) as fh:
            return fh.read().strip() == stamp
    return False


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile + link if a source changed since the library was linked.  Safe under ``torchrun``: the ranks of one
    node serialise on a file lock (the first one builds, the others find the stamp up to date), the library is linked
    under a temporary name and moved into place atomically, and the stamp is written last."""
    import fcntl
    stamp_file = os.path.join(OBJ, "stamp")
    stamp = _stamp()
    if not force and _up_to_date(stamp_file, stamp):
        return OUT
    os.makedirs(OBJ, exist_ok=True)
    with open(os.path.join(OBJ, "lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and _up_to_date(stamp_file, stamp):      # another rank built it while this one waited
                return OUT
            return _build_locked(stamp_file, stamp, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(stamp_file: str, stamp: str, verbose: bool) -> str:

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp_out = f"{OUT}.{os.getpid()}.tmp"
    r = subprocess.run([NVCC, "-shared", "-o", tmp_out, *objs, "-gencode", "arch=compute_100a,code=sm_100a"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp_out, OUT)                       # a process that dlopens concurrently sees the old or the new file, never half of one
    with open(stamp_file + ".tmp", "w") as fh:
        fh.write(stamp)
    os.replace(stamp_file + ".tmp", stamp_file)
    return OUT


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
