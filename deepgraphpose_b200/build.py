"""In-tree build of libdgp_b200.so (hand-written sm_100a CUDA, C ABI in include/dgp_b200.h).

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libdgp_b200.so")
SOURCES = ["capi.cu", "conv_gemm_sm100.cu", "wgrad_gemm_sm100.cu", "softargmax.cu", "aux_kernels.cu", "loss_kernels.cu", "param_kernels.cu", "bwd_kernels.cu", "train.cu", "feeder_kernels.cu", "boundary.cu", "variables.cu", "stream.cu", "flow_kernels.cu", "resize_kernels.cu", "augment_kernels.cu", "render_kernels.cu", "jpeg_kernels.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xcompiler", "-Wno-unused-function",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "dgp_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    objs = []
    build_dir = os.path.join(HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs + ["-lcudart", "-lpthread", "-ldl"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
