"""Build libdots_ocr_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m dots_ocr_b200.build [--force]

The library links cudart statically and resolves cuTensorMapEncodeTiled through
cudaGetDriverEntryPoint, so it has no link-time dependency on libcuda or on torch.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdots_ocr_b200.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["common.cu", "gemm_tcgen05.cu", "attn_fwd_mma.cu", "attn_fwd_tcgen05.cu", "attn_decode.cu", "decode_gemm.cu", "elementwise.cu", "sampling.cu", "partition.cu"]
# documented negative results (DESIGN.md section 8): compiled into the library only on request, never by default
EXPERIMENTS = ["experiments/attn_fwd_tcgen05_pair.cu", "experiments/decode_chain.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc"), "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _digest() -> str:
    h = hashlib.sha256()
    names = sorted(os.listdir(CSRC)) + ["../../include/dots_ocr_b200.h"]
    if os.environ.get("DOTS_BUILD_EXPERIMENTS") == "1":
        names += ["experiments/" + n for n in sorted(os.listdir(os.path.join(CSRC, "experiments")))]
        h.update(b"+experiments")
    for n in names:
        p = os.path.join(CSRC, n)
        if os.path.isfile(p):
            h.update(n.encode())
            with open(p, "rb") as f:
                h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    stamp = os.path.join(OBJ_DIR, "stamp")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()

    sources = SOURCES + (EXPERIMENTS if os.environ.get("DOTS_BUILD_EXPERIMENTS") == "1" else [])

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, os.path.basename(src).replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        objs = list(ex.map(compile_one, sources))
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
