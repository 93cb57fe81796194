"""Build librag_b200.so (sm_100a only) in-tree with nvcc.  `python -m rag_b200.build`."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librag_b200.so")
SOURCES = ["abi.cu", "cost_volume.cu", "disp_head.cu", "extras.cu", "cv_stem.cu", "cv_stem_train.cu", "last_conv.cu", "last_conv_bwd.cu", "trilinear.cu", "conv3d_cc.cu", "bn3d.cu", "conv3d_pw.cu", "grid_sample.cu"]
FLAGS = [
    "-O3", "-std=c++17", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-shared", "-cudart", "static",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; librag_b200.so cannot be built")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "rag_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile to a temporary file and rename it into place under a file lock: under torchrun every rank may find the library
    missing or stale at the same moment, and a rank must never dlopen a half-written .so (ADVICE r1)."""
    import fcntl
    import tempfile

    if not force and not needs_build():
        return LIB
    with open(LIB + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():          # another rank built it while we waited for the lock
                return LIB
            fd, tmp = tempfile.mkstemp(prefix="librag_b200.", suffix=".so.tmp", dir=HERE)
            os.close(fd)
            cmd = [nvcc()] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", tmp]
            res = subprocess.run(cmd, capture_output=True, text=True)
            if res.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
            os.chmod(tmp, 0o755)
            os.replace(tmp, LIB)                           # atomic on POSIX
            if verbose:
                print(res.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
