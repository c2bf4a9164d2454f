"""In-tree build of the CUDA library: nvcc -> vision_transformer_detector_b200/libvitdet_b200.so.

The library is sm_100a only (tcgen05 / TMEM / TMA); nvcc cross-compiles it without a GPU.
`python -m vision_transformer_detector_b200.build` or `__graft_entry__.build()` runs this.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
LIB_PATH = os.path.join(PKG_DIR, "libvitdet_b200.so")
STAMP_PATH = os.path.join(PKG_DIR, ".libvitdet_b200.stamp")

SOURCES = ["engine.cu", "gemm_tc.cu", "gemm_tc2.cu", "gemm_simt.cu", "attention.cu", "attention_tc.cu", "attention_tcs.cu", "mlp_tail.cu", "rowops.cu", "metric.cu", "gather.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]



def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _source_hash() -> str:
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + [os.path.join(INCLUDE, "vitdet_b200.h")]
    for name in files:
        path = name if os.path.isabs(name) else os.path.join(CSRC, name)
        if not os.path.isfile(path):
            continue
        h.update(name.encode())
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


# Sources that define the dominant GEMM (gemm_tc2_kernel and what it includes): the ncu traffic capture quoted by bench.py's
# roofline.traffic is stamped with this hash, so that edits to unrelated kernels do not void it.
DOMINANT_KERNEL_SOURCES = ["gemm_tc2.cu", "common.cuh", "kernels.h", "launch.h"]


def kernel_hash(names=None) -> str:
    h = hashlib.sha256()
    for name in (names or DOMINANT_KERNEL_SOURCES):
        h.update(name.encode())
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current() -> bool:
    if not os.path.exists(LIB_PATH) or not os.path.exists(STAMP_PATH):
        return False
    with open(STAMP_PATH) as f:
        return f.read().strip() == _source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu of csrc/ into one shared library.  Objects are built in parallel."""
    if not force and is_current():
        return LIB_PATH
    nvcc = _nvcc()
    obj_dir = os.path.join(PKG_DIR, "build")
    os.makedirs(obj_dir, exist_ok=True)
    procs = []
    objs = []
    # A/B builds (scripts/gpu_ab_lib.sh): extra -D switches; such a build is never stamped as current
    extra = os.environ.get("VITDET_EXTRA_NVCC_FLAGS", "").split()
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-I", INCLUDE, "-I", CSRC, "-c", path, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = []
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            failed.append((src, out))
    if failed:
        msg = "\n".join(f"--- {s} ---\n{o}" for s, o in failed)
        raise RuntimeError(f"nvcc failed:\n{msg}")
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH, *objs, "-ldl"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    with open(STAMP_PATH, "w") as f:
        f.write(_source_hash() if not os.environ.get("VITDET_EXTRA_NVCC_FLAGS") else "ab-build")
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
