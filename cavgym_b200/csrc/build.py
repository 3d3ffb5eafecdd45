"""Build libcavgym_sm100.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m cavgym_b200.csrc.build [--force] [--jobs N]

One translation unit per body count (small_mK.cu, record_mK.cu, until_mK.cu, params_mK.cu, regen_mK.cu) so the kernels compile in parallel.
-fmad=false keeps the fp64 arithmetic in the reference's operation order (no FMA contraction).
"""
import argparse
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
LIB = os.environ.get("CAVGYM_LIB_OUT") or os.path.join(PKG, "libcavgym_sm100.so")
OBJ_DIR = os.environ.get("CAVGYM_OBJ_DIR") or os.path.join(HERE, "build")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=" + os.environ.get("CAVGYM_FMAD", "false"), "-std=c++17",
         "-Xcompiler", "-fPIC,-O2", "--threads", "1"]


def sources():
    return sorted(f for f in os.listdir(HERE) if f.endswith(".cu"))


def headers_mtime():
    paths = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cuh", ".inc"))]
    paths.append(os.path.join(PKG, "..", "include", "cavgym.h"))
    return max(os.path.getmtime(p) for p in paths)


ONLY_M = [int(v) for v in os.environ.get("CAVGYM_ONLY_M", "").split(",") if v]   # development: compile these body counts only
EXTRA = os.environ.get("CAVGYM_NVCC_FLAGS", "").split()


def compile_one(src, force, verbose):
    stub = bool(ONLY_M) and src.startswith(("small_m", "record_m", "until_m", "params_m", "regen_m")) and int(src.split("_m")[1][:-3]) not in ONLY_M
    obj = os.path.join(OBJ_DIR, src[:-3] + (".stub.o" if stub else ".o"))
    src_path = os.path.join(HERE, src)
    if not force and not EXTRA and os.path.isfile(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(src_path), headers_mtime()):
        return obj, ""
    cmd = [NVCC] + FLAGS + EXTRA + (["-DCAV_STUB"] if stub else []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", src_path, "-o", obj]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{proc.stdout}\n{proc.stderr}")
    return obj, proc.stderr


def build(force=False, jobs=None, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    srcs = sources()
    jobs = jobs or min(len(srcs), os.cpu_count() or 4)
    logs = []
    with concurrent.futures.ThreadPoolExecutor(max_workers=jobs) as pool:
        results = list(pool.map(lambda s: compile_one(s, force, verbose), srcs))
    objs = [obj for obj, _ in results]
    logs = [log for _, log in results if log]
    if True:
        cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode != 0:
            raise RuntimeError(f"link failed:\n{proc.stdout}\n{proc.stderr}")
    if verbose:
        print("\n".join(logs))
    return LIB


if __name__ == "__main__":
    parser = argparse.ArgumentParser()
    parser.add_argument("--force", action="store_true")
    parser.add_argument("--jobs", type=int, default=None)
    parser.add_argument("--verbose", action="store_true")
    args = parser.parse_args()
    print(build(args.force, args.jobs, args.verbose))
