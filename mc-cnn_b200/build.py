"""Build libadcensus_b200.so (the product: sm_100a kernels + C ABI) in-tree with nvcc.

Kept in-tree (mc-cnn_b200/libadcensus_b200.so) so the built library travels with
the repo snapshot to the GPU box; git-ignored so history stays source-only.
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libadcensus_b200.so")
SOURCES = ["common.cu", "stereo_join.cu", "stereo_join_tma.cu", "cross_cbca.cu", "cbca_tma.cu", "cbca_ws.cu", "sgm.cu", "post.cu", "adcensus_cost.cu", "scorer_head.cu", "feature_tower.cu", "pipeline.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ARCH + ["-O3", "-lineinfo", "-diag-suppress", "177", "-std=c++17", "--compiler-options", "-fPIC", "-I" + INCLUDE, "-I" + CSRC]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libadcensus_b200.so")
    return exe


def _newer(a, b):
    return (not os.path.exists(b)) or os.path.getmtime(a) > os.path.getmtime(b)


def _deps_mtime():
    hs = [os.path.join(INCLUDE, "adcensus_b200.h")] + [
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))
    ]
    return max(os.path.getmtime(h) for h in hs)


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library.  Returns its path."""
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()
    hdr_m = _deps_mtime()
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        if force or _newer(s, o) or os.path.getmtime(o) < hdr_m:
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (s, r.stdout, r.stderr))
        return r.stderr

    with concurrent.futures.ThreadPoolExecutor(max_workers=max(1, min(8, len(jobs)))) as ex:
        for log in ex.map(compile_one, jobs):
            if verbose and log:
                sys.stderr.write(log)
    objs = [os.path.join(OBJDIR, src.replace(".cu", ".o")) for src in SOURCES]
    if force or jobs or not os.path.exists(LIB):
        # --no-undefined: an internal reference without a definition fails here rather than at the first dlopen
        cmd = [nvcc] + ARCH + ["--shared", "-Xlinker", "--no-undefined", "-o", LIB] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
