"""Builds libcimbar_b200/lib/libcb200.so (the C-ABI shared library) with nvcc for sm_100a, in-tree.

    python -m libcimbar_b200.build [--force]

nvcc cross-compiles without a GPU; the built .so is git-ignored but travels to the GPU box with the repo snapshot.
Every .cu is compiled to its own object (in parallel, only when it or a header changed) and the objects are linked."""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "lib", "obj")
LIB = os.path.join(HERE, "lib", "libcb200.so")
SOURCES = ["api.cu", "k1_decode.cu", "k1x_flood.cu", "k2_rs.cu", "render.cu", "encode.cu", "host_sink.cu", "ccm.cu",
           "gather.cu", "deskew.cu", "scan.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]
NVCC_FLAGS += os.environ.get("CB200_NVCC_EXTRA", "").split()      # tuning only: -D switches of compile-time variants (A/B on the GPU box)


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(HERE, "..", "include", "cb200.h"))
    hs += [os.path.join(HERE, "host", f) for f in os.listdir(os.path.join(HERE, "host"))]
    return hs


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in _sources()] + _headers()
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = max(os.path.getmtime(h) for h in _headers())
    jobs = []
    for s in _sources():
        src, obj = os.path.join(CSRC, s), os.path.join(OBJ, s[:-3] + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_t):
            jobs.append([_nvcc()] + NVCC_FLAGS + ["-c", src, "-o", obj])
    if verbose:
        for j in jobs:
            print(" ".join(j))
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 4))) as ex:
        for rc in ex.map(lambda j: subprocess.call(j), jobs):
            if rc != 0:
                raise subprocess.CalledProcessError(rc, "nvcc")
    link = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + \
           [os.path.join(OBJ, s[:-3] + ".o") for s in _sources()] + ["-ldl"]
    if verbose:
        print(" ".join(link))
    subprocess.check_call(link)
    return LIB


FACADE_LIB = os.path.join(HERE, "lib", "libcimbard_b200.so")


def build_facade(force=False, verbose=False):
    """lib/libcimbard_b200.so: the reference's cimbard_* receive facade (include/cimbard_b200.h) over libcb200.so."""
    src = os.path.join(HERE, "host", "cimbard_b200.cpp")
    deps = [src, os.path.join(HERE, "..", "include", "cb200.h")]
    if not force and os.path.exists(FACADE_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(FACADE_LIB) for d in deps):
        return FACADE_LIB
    cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-o", FACADE_LIB, src, "-L" + os.path.dirname(LIB), "-lcb200",
           "-Wl,-rpath,$ORIGIN", "-ldl"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return FACADE_LIB


WIREHAIR_LIB = os.path.join(HERE, "lib", "libwirehair.so")
WIREHAIR_BUILT = os.path.join(HERE, "..", "oracle", "_ref", "libwirehair.so")


def build_wirehair(force=False, verbose=False):
    """wirehair -- the reference's third-party fountain codec (P15, stays on the rank-0 host) -- next to the product's libraries.
    Its sources are not part of this repository: `make -C oracle ref` compiles them unmodified from the reference checkout into
    oracle/_ref/libwirehair.so, and this installs that file as lib/libwirehair.so, where the facade and FountainSink look for it.
    The product binds it at run time (cb200_sink_create_wirehair), exactly as libcimbar links it."""
    if not os.path.exists(WIREHAIR_BUILT):
        return WIREHAIR_LIB if os.path.exists(WIREHAIR_LIB) else None
    if force or not os.path.exists(WIREHAIR_LIB) or os.path.getmtime(WIREHAIR_LIB) < os.path.getmtime(WIREHAIR_BUILT):
        os.makedirs(os.path.dirname(WIREHAIR_LIB), exist_ok=True)
        if verbose:
            print("install %s -> %s" % (WIREHAIR_BUILT, WIREHAIR_LIB))
        shutil.copy2(WIREHAIR_BUILT, WIREHAIR_LIB)
    return WIREHAIR_LIB


if __name__ == "__main__":
    print(build_wirehair(force="--force" in sys.argv, verbose=True))
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_facade(force="--force" in sys.argv, verbose=True))
