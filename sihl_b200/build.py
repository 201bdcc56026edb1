"""Build recipe for ``libsihl_b200.so`` (plain nvcc, in-tree, sm_100a only).

The library is a C-ABI shared object with no torch dependency
(``include/sihl_od.h``).  ``-fmad=false`` + IEEE division: every source operator
is one fp32 operation, which is what makes assignment indices bit-equal to
torch-CUDA eager (SURVEY.md §7.1).  ``-lineinfo`` so ncu's source page maps to
these files.
"""
from __future__ import annotations

import fcntl
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsihl_b200.so")
STAMP_PATH = os.path.join(LIB_DIR, "libsihl_b200.stamp")
SOURCES = ["od_api.cu", "od_anchors.cu", "od_assign.cu", "od_quad.cu", "od_loss.cu", "od_train.cu", "od_exchange.cu", "od_infer.cu", "od_nms.cu", "od_nms_wide.cu", "od_soft_nms.cu", "od_box_vote.cu", "od_map.cu", "od_mlp.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libsihl_b200.so cannot be built (there is no CPU fallback)")
    return exe


def _fingerprint() -> str:
    """Content hash of every source + the flags: file times do not survive being copied to another box."""
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    files.append(os.path.join(HERE, "..", "include", "sihl_od.h"))
    for path in files:
        h.update(os.path.basename(path).encode())
        with open(path, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def _fresh(fp: str) -> bool:
    try:
        with open(STAMP_PATH) as fh:
            return os.path.exists(LIB_PATH) and fh.read().strip() == fp
    except OSError:
        return False


def is_fresh() -> bool:
    """True when the library on disk was built from exactly the sources + flags now in the tree."""
    return _fresh(_fingerprint())


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every ``.cu`` for sm_100a and link ``sihl_b200/lib/libsihl_b200.so``.

    Safe under ``torchrun``: one process builds (file lock), the others wait; the library appears atomically."""
    fp = _fingerprint()
    if not force and _fresh(fp):
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and _fresh(fp):           # another rank built it while we waited
                return LIB_PATH
            _compile_and_link(fp, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


def _compile_and_link(fp: str, verbose: bool) -> None:
    nvcc = _nvcc()
    obj_dir = tempfile.mkdtemp(prefix="sihl_b200_build_")

    def compile_one(src: str) -> str:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-Xptxas", "-v" if verbose else "-warn-spills", "-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            sys.stderr.write(res.stderr)
        return obj

    try:
        with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
            objs = list(pool.map(compile_one, SOURCES))
        tmp_lib = os.path.join(obj_dir, "libsihl_b200.so")
        link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-o", tmp_lib, *objs,
                "-cudart", "shared"]
        res = subprocess.run(link, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
        staged = LIB_PATH + f".tmp{os.getpid()}"
        shutil.copyfile(tmp_lib, staged)
        os.chmod(staged, 0o755)
        os.replace(staged, LIB_PATH)               # atomic: a concurrent dlopen sees the old or the new file, never half
        with open(STAMP_PATH + f".tmp{os.getpid()}", "w") as fh:
            fh.write(fp + "\n")
        os.replace(STAMP_PATH + f".tmp{os.getpid()}", STAMP_PATH)
    finally:
        shutil.rmtree(obj_dir, ignore_errors=True)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
