"""Builds pangenomix_b200/libpgx_b200.so (sm_100a only) in-tree with nvcc.

    python -m pangenomix_b200.build [--force] [--verbose]

The shared object is git-ignored but travels with the working tree to the GPU box.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpgx_b200.so")
SOURCES = ["pgx_api.cu", "pgx_rarefy.cu", "pgx_bernoulli.cu", "pgx_heaps.cu", "pgx_betabin.cu", "pgx_perm.cu", "pgx_shared.cu"]
HOST_SOURCES = ["pgx_rng.cpp", "pgx_plan.cpp", "pgx_inflate.cpp", "pgx_expand.cpp", "pgx_plan_build.cpp"]            # plain C++ (g++): AVX2 paths are selected at run time
HEADERS = [os.path.join(CSRC, "pgx_common.cuh"), os.path.join(REPO, "include", "pgx.h")]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    built = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HOST_SOURCES] + HEADERS
    return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False, debug=False):
    if not force and not needs_build():
        return LIB
    objects = []
    for src in HOST_SOURCES:
        obj = os.path.join(CSRC, os.path.splitext(src)[0] + ".o")
        subprocess.run([os.environ.get("CXX", "g++"), "-O3", "-std=c++17", "-fPIC", "-pthread",
                        "-I", os.path.join(REPO, "include"), "-c", os.path.join(CSRC, src), "-o", obj], check=True)
        objects.append(obj)
    cmd = [nvcc_path(), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
           "-lineinfo", "-Xcompiler", "-fPIC,-O3,-pthread", "-shared",
           "-I", os.path.join(REPO, "include"), "-I", CSRC, "-o", LIB]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    if debug:
        cmd += ["-DPGX_DEBUG_BOUNDS"]          # device-side index assertions (see pgx_common.cuh)
    cmd += [os.path.join(CSRC, s) for s in SOURCES] + objects
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv or "--debug" in sys.argv, verbose="--verbose" in sys.argv,
                debug="--debug" in sys.argv))
