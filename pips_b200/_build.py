"""In-tree build of libpips_b200.so with nvcc for sm_100a (no torch headers, no libcuda link).

The shared object stays inside the package directory so that it travels with the repo snapshot to
the GPU box; it is git-ignored.  ``build()`` is idempotent (mtime check) and cheap to call.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "lib", "obj")
LIB = os.path.join(HERE, "lib", "libpips_b200.so")
SOURCES = ["abi.cu", "pyramid.cu", "corr_gather.cu", "mixer_simt.cu", "tokenmix_tc.cu", "gemm_tc.cu", "gemm_tc2.cu", "conv_tc.cu", "conv_rows.cu", "encoder_ops.cu", "heatmap.cu", "score_loss.cu", "peer.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


DIGEST = LIB + ".digest"


def source_digest() -> str:
    """SHA-256 over every source, header and the compiler flags: what the built library was made from.
    Robust to mtime churn (the repo snapshot pushed to the GPU box keeps contents, not necessarily times)."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    files.append(os.path.join(os.path.dirname(HERE), "include", "pips_b200.h"))
    for f in files:
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def is_stale() -> bool:
    """True when libpips_b200.so is missing or was built from other sources than the ones on disk."""
    if not os.path.exists(LIB) or not os.path.exists(DIGEST):
        return True
    with open(DIGEST) as f:
        return f.read().strip() != source_digest()


def have_nvcc() -> bool:
    import shutil
    return any(c and (os.path.exists(c) if os.path.isabs(c) else shutil.which(c)) for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"))


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _deps_mtime() -> float:
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "pips_b200.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def _compile(src: str, log: list) -> str:
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    spath = os.path.join(CSRC, src)
    if os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(spath), _deps_mtime()):
        return obj
    cmd = [_nvcc(), *NVCC_FLAGS, "-c", spath, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log.append((src, r.stderr))
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    return obj


def build(verbose: bool = False, force: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    log: list = []
    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(lambda s: _compile(s, log), SOURCES))
    if force or not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(DIGEST, "w") as f:
        f.write(source_digest() + "\n")
    if verbose:
        for src, err in log:
            print(f"--- {src}\n{err}", file=sys.stderr)
    return LIB


if __name__ == "__main__":
    print(build(verbose=True, force="--force" in sys.argv))
