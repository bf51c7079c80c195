"""Build recipe for lib/libmeshclust2_b200.so: hand-written CUDA for sm_100a + the C ABI, in-tree.

nvcc cross-compiles without a GPU.  -fmad=false keeps the fp64 epilogue free of fused multiply-adds so it follows
the reference's expression order (the integer kernels are unaffected).  Every source is compiled to its own object
(in parallel, only when it or a header changed) and the objects are linked into the shared library.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
NAMES = ("mc2_api.cu", "kmer_count.cu", "pair_score.cu", "tile_sweep.cu", "mean_shift.cu", "text_ingest.cu", "strand.cu", "topk.cu",
         "host_encode.cpp")
SRC = [os.path.join(HERE, "csrc", f) for f in NAMES]
HDR = [os.path.join(HERE, "csrc", "mc2_internal.cuh"), os.path.join(HERE, "csrc", "pair_eval.cuh"),
       os.path.join(HERE, "..", "include", "meshclust2_b200.h")]
OUT = os.path.join(HERE, "lib", "libmeshclust2_b200.so")
OBJ_DIR = os.path.join(HERE, "lib", "obj")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CFLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-fmad=false", "-std=c++17",
          "-Xcompiler", "-fPIC,-fopenmp,-O2"]
LFLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC,-fopenmp", "-lgomp"]


def _obj(src):
    return os.path.join(OBJ_DIR, os.path.basename(src) + ".o")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(f) > t for f in deps)


def needs_build():
    return _stale(OUT, SRC + HDR + [os.path.abspath(__file__)])


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    os.makedirs(OBJ_DIR, exist_ok=True)
    todo = [s for s in SRC if force or _stale(_obj(s), [s] + HDR + [os.path.abspath(__file__)])]

    def compile_one(src):
        cmd = [NVCC] + CFLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", _obj(src), src]
        print("[meshclust2_b200.build]", " ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, r

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(todo)))) as ex:
        results = list(ex.map(compile_one, todo))
    for src, r in results:
        if verbose or r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise subprocess.CalledProcessError(r.returncode, "nvcc -c " + src)
    cmd = [NVCC] + LFLAGS + ["-o", OUT] + [_obj(s) for s in SRC]
    print("[meshclust2_b200.build]", " ".join(cmd), file=sys.stderr)
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
