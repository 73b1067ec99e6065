"""Build recipe for libbcosk.so (hand-written sm_100a kernels + C ABI), in-tree.

    python -m bcos_b200.build            # or  bcos_b200.build.build()

Plain nvcc, no torch headers: the library's interface is the C ABI in include/bcosk.h.
The .so is git-ignored but travels with the repo snapshot to the GPU box.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
ROOT = os.path.dirname(PKG)
LIB = os.path.join(PKG, "libbcosk.so")
STAMP = os.path.join(PKG, ".libbcosk.stamp")

SOURCES = ["bcosk_api.cu", "bcosk_igemm.cu", "bcosk_igemm_hp.cu", "bcosk_wgrad.cu", "bcosk_train.cu", "bcosk_elementwise.cu", "bcosk_layout.cu", "bcosk_tokens.cu",
           "bcosk_rgba.cu", "bcosk_norms.cu", "bcosk_vit.cu", "bcosk_vit_attn.cu", "bcosk_dense.cu", "bcosk_dense_train.cu", "bcosk_head.cu"]
HEADERS = ["bcosk_common.cuh", "bcosk_host.h", "bcosk_igemm_epi.cuh", os.path.join(ROOT, "include", "bcosk.h")]
OBJDIR = os.path.join(PKG, "build")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-DBCOSK_BUILD=1",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set $NVCC)")


def _digest() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        p = f if os.path.isabs(f) else os.path.join(CSRC, f)
        with open(p, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _file_digest(path: str, extra: str) -> str:
    h = hashlib.sha256()
    for f in [path] + HEADERS:
        p = f if os.path.isabs(f) else os.path.join(CSRC, f)
        with open(p, "rb") as fh:
            h.update(fh.read())
    h.update((" ".join(NVCC_FLAGS) + "|" + extra).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libbcosk.so if sources changed; returns the library path.  Every translation unit is compiled to its own
    object (in parallel, only those whose source or headers changed), then linked.
    $BCOSK_EXTRA_NVCC_FLAGS (experiments only) is appended to the nvcc command line."""
    from concurrent.futures import ThreadPoolExecutor
    extra = os.environ.get("BCOSK_EXTRA_NVCC_FLAGS", "").split()
    dig = _digest() + "|" + " ".join(extra)
    if not force and os.path.exists(LIB) and os.path.exists(STAMP):
        with open(STAMP) as fh:
            if fh.read().strip() == dig:
                return LIB
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str):
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        d = _file_digest(path, " ".join(extra))
        stamp = obj + ".stamp"
        if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read().strip() == d:
            return obj, None
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-I", os.path.join(ROOT, "include"), "-c", "-o", obj, path]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            return obj, RuntimeError(f"nvcc failed on {src}:\n{res.stdout}{res.stderr}")
        if verbose:
            sys.stderr.write(res.stdout + res.stderr)
        with open(stamp, "w") as fh:
            fh.write(d)
        return obj, None

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    for _, err in results:
        if err is not None:
            sys.stderr.write(str(err))
            raise RuntimeError("nvcc failed building libbcosk.so")
    res = subprocess.run([nvcc, "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB]
                         + [o for o, _ in results], capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking libbcosk.so")
    with open(STAMP, "w") as fh:
        fh.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
