"""Build libcosmomap2_b200.so for sm_100a with nvcc (in-tree, next to the sources)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["cabi.cu", "tod_pass.cu", "pixel_ops.cu", "noise_ops.cu", "deflation.cu", "vecops.cu", "p2p_allreduce.cu", "pcg_sharded.cu", "dense_z.cu", "toeplitz_fft.cu", "filter_runs.cu", "filter_poly.cu", "destripe.cu"]
LIB = os.path.join(HERE, "libcosmomap2_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _newest_source_mtime():
    files = [os.path.join(HERE, f) for f in SOURCES + ["cm2_common.cuh"]]
    files.append(os.path.join(HERE, "..", "..", "include", "cosmomap2_b200.h"))
    return max(os.path.getmtime(f) for f in files)


def build(force=False, verbose=False):
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_source_mtime():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(HERE, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("---- %s\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([nvcc, "-shared", "-o", LIB] + objs + ["-lcudart"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
