"""In-tree build of libspeecht5_b200.so (hand-written sm_100a kernels behind a C ABI, no torch dependency).

nvcc cross-compiles without a GPU; the resulting .so travels with the source tree (git-ignored, not gpurun-ignored).
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib", "libspeecht5_b200.so")
SOURCES = ["api.cu", "gemm.cu", "elementwise.cu", "norm.cu", "layernorm.cu", "attention.cu", "attention_tc.cu", "attention_fused.cu", "attention_fused_bwd.cu", "attention_flash.cu",
           "optim.cu", "conv_frontend.cu", "ctc.cu", "ctc_prefix.cu", "criterion.cu"]
HEADERS = ["ptx.cuh", "gemm.cuh", "kernels.cuh", "tma_map.cuh", "vec8.cuh", os.path.join("..", "..", "include", "speecht5_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-cudart", "static",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stamp():
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu into objects (parallel) and link the shared library. Returns the library path."""
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    stamp_file = LIB + ".stamp"
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    objdir = os.path.join(HERE, "lib", "obj")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
        objs.append(obj)
    cmd = [_nvcc()] + NVCC_FLAGS + ["-shared"] + objs + ["-o", LIB]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    with open(stamp_file, "w") as fh:
        fh.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
