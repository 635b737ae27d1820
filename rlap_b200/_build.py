"""Builds rlap_b200/_lib/librlap_b200.so in-tree with nvcc for sm_100a (no torch headers needed:
the product boundary is a plain C ABI, include/rlap_b200.h)."""
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "librlap_b200.so")
SOURCES = ["api.cu", "schur.cu", "emit.cu", "ingest.cu"]
HEADERS = ["rlap_device.cuh", "schur.cuh", "scan.cuh", "star.cuh", "introsort.cuh", "ingest.cuh", os.path.join("..", "..", "include", "rlap_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]
OBJ_DIR = os.path.join(LIB_DIR, "obj")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    flags = list(NVCC_FLAGS)
    if os.environ.get("RLAP_DEBUG_BUILD"):   # profiling build: phase wait timers, RLAP_GROUPS / RLAP_DEBUG_SYNC knobs
        flags.append("-DRLAP_DEBUG")
    flags += os.environ.get("RLAP_NVCC_EXTRA", "").split()     # experiments: extra nvcc flags
    # one nvcc per translation unit, side by side (the elimination kernel is compiled once per mode: most of the time)
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs = [os.path.join(OBJ_DIR, s[:-3] + ".o") for s in SOURCES]

    def compile_one(src, obj):
        cmd = [nvcc] + flags + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        for f in [ex.submit(compile_one, s, o) for s, o in zip(SOURCES, objs)]:
            f.result()
    cmd = [nvcc] + flags + ["-shared", "-o", LIB_PATH] + objs
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
