"""Builds rdfc_gan_b200/librdfc_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m rdfc_gan_b200.build [--force] [--verbose]
"""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "librdfc_b200.so")
SOURCES = ["api.cu", "dcn.cu", "nlspn.cu", "conv_simt.cu", "conv_umma.cu", "conv.cu", "norm.cu", "metrics.cu", "train.cu", "wgrad_umma.cu", "train_split.cu", "esanet.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         "-ccbin", "/usr/bin/g++"] + os.environ.get("RDFC_NVCC_FLAGS", "").split()   # e.g. -DRDFC_UMMA_TIMERS


def _deps_mtime():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "rdfc_b200.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    hdr_m = _deps_mtime()
    stamp = os.path.join(OBJ, ".flags")          # objects built with other flags (RDFC_NVCC_FLAGS) are stale
    if not os.path.exists(stamp) or open(stamp).read() != " ".join(FLAGS):
        force = True
    jobs = []
    for s in SOURCES:
        src, obj = os.path.join(CSRC, s), os.path.join(OBJ, s[:-3] + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_m):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append((s, cmd))
    with concurrent.futures.ThreadPoolExecutor(max_workers=8) as ex:
        futs = {s: ex.submit(subprocess.run, cmd, capture_output=True, text=True) for s, cmd in jobs}
    for s, f in futs.items():
        r = f.result()
        if verbose or r.returncode:
            sys.stderr.write(f"== {s}\n{r.stdout}{r.stderr}")
        if r.returncode:
            raise RuntimeError(f"nvcc failed on {s}")
    with open(stamp, "w") as f:
        f.write(" ".join(FLAGS))
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in SOURCES]
    if jobs or not os.path.exists(LIB):
        subprocess.check_call([NVCC, "-shared", "-o", LIB] + objs + ["-ccbin", "/usr/bin/g++", "-lcudart_static", "-ldl", "-lrt", "-lpthread"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
