"""Build libb200unet.so (hand-written sm_100a CUDA behind the C ABI in include/b200unet.h) in-tree with nvcc.

No torch / pybind dependency: the library is plain `extern "C"` and is loaded with ctypes (see _lib.py).
"""
from __future__ import annotations

import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libb200unet.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["api.cu", "igemm.cu", "conv3_res.cu", "conv3_pair.cu", "first_layer.cu", "wgrad.cu", "elementwise.cu", "small.cu", "loss.cu", "optim.cu", "generic_f32.cu", "nvl_sync.cu", "edge.cu", "gate.cu", "dropout.cu", "head_many.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stamp() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for name in sorted(os.listdir(root)):
            with open(os.path.join(root, name), "rb") as f:
                h.update(name.encode())
                h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    stamp_file = os.path.join(OBJ_DIR, "stamp")
    stamp = _stamp()
    if not force and os.path.exists(OUT) and os.path.exists(stamp_file):
        with open(stamp_file) as f:
            if f.read().strip() == stamp:
                return OUT
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return OUT


def build_probe(force: bool = False) -> str:
    """tests/probe/libb200probe.so: the UMMA-descriptor hardware probe of tests/test_gpu_probe.py. A TEST-ONLY object (its
    entry point is not in include/b200unet.h and not in libb200unet.so); it reuses api.cu's host helpers."""
    root = os.path.join(HERE, "..", "tests", "probe")
    src, out = os.path.join(root, "probe_shift.cu"), os.path.join(root, "libb200probe.so")
    deps = [src, os.path.join(CSRC, "api.cu"), os.path.join(CSRC, "tc_common.cuh"), os.path.join(CSRC, "host_common.h")]
    if not force and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(d) for d in deps):
        return out
    cmd = [_nvcc(), *NVCC_FLAGS, "-shared", src, os.path.join(CSRC, "api.cu"), "-o", out, "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for the probe:\n{r.stdout}\n{r.stderr}")
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
