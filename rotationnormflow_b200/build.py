"""Build librnf_b200.so in-tree with nvcc for sm_100a (the only target; no fallback, no multi-arch)."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librnf_b200.so")
STAMP = os.path.join(HERE, "csrc", ".build_stamp")
SOURCES = ["rnf_abi.cu", "flow_v1.cu", "flow_row.cu", "flow_t4.cu", "condition.cu", "dedup.cu", "healpix.cu", "fisher_sample.cu", "train_ops.cu", "flow_grad.cu", "modes.cu", "hgrid.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "--expt-relaxed-constexpr", "-Xptxas", "-v", "-lcuda",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: librnf_b200.so cannot be built (there is no CPU fallback)")


def _digest() -> str:
    h = hashlib.sha256()
    names = [n for n in sorted(os.listdir(CSRC)) if not n.startswith(".") and ".tmp" not in n] + ["../../include/rnf_abi.h"]
    for n in names:
        p = os.path.join(CSRC, n)
        if os.path.isfile(p):
            h.update(n.encode())
            with open(p, "rb") as f:
                h.update(f.read())
    h.update((" ".join(NVCC_FLAGS) + os.environ.get("RNF_NVCC_EXTRA", "")).encode())
    return h.hexdigest()


def up_to_date() -> bool:
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _digest()


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile in-tree.  Safe with one process per GPU: an inter-process file lock serialises the staleness check and the
    build, nvcc writes to a temporary path and the finished library is moved into place atomically, so no rank can dlopen a
    partly written file."""
    import fcntl
    lock_path = os.path.join(CSRC, ".build_lock")
    with open(lock_path, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and up_to_date():
                return LIB
            extra = os.environ.get("RNF_NVCC_EXTRA", "").split()      # e.g. -DRNF_TC_TRACE=1 for the phase-timeline debug build
            tmp = f"{LIB}.tmp.{os.getpid()}"
            cmd = [_nvcc()] + NVCC_FLAGS + extra + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", tmp]
            res = subprocess.run(cmd, capture_output=True, text=True)
            log = res.stdout + res.stderr
            with open(os.path.join(CSRC, ".build_log"), "w") as f:
                f.write(log)
            if res.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + log[-6000:])
            if verbose:
                print(log)
            os.replace(tmp, LIB)
            with open(STAMP + ".tmp", "w") as f:
                f.write(_digest())
            os.replace(STAMP + ".tmp", STAMP)
            return LIB
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


if __name__ == "__main__":
    build_library(force="--force" in sys.argv, verbose=True)
    print("built", LIB)
