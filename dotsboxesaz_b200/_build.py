"""In-tree nvcc build of the C-ABI library (sm_100a only; nvcc cross-compiles without a GPU)."""
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libdbaz_b200.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["dbaz_capi.cu", "dbaz_tower.cu", "dbaz_trunk.cu"]
HEADERS = ["dbaz_device.cuh", "dbaz_game_kernels.cuh", "dbaz_tree_kernels.cuh", "dbaz_nn_kernels.cuh", "dbaz_tower.cuh", "dbaz_tcgen05.cuh", "dbaz_trunk.cuh", "dbaz_loop.cuh", "dbaz_selfplay.cuh", "dbaz_solver.cuh", "dbaz_endgame.cuh"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-I" + INCLUDE]


def _deps():
    return [os.path.join(CSRC, f) for f in HEADERS] + [os.path.join(INCLUDE, "dbaz_b200.h")]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _stale():
    return _newer(LIB, [os.path.join(CSRC, s) for s in SOURCES] + _deps())


def build(force=False, verbose=False):
    """Compile dotsboxesaz_b200/libdbaz_b200.so if missing or older than its sources: one object per translation
    unit (in parallel, only the stale ones), then one link."""
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ_DIR, exist_ok=True)
    extra = ["-Xptxas", "-v"] if verbose else []

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        if force or _newer(obj, [os.path.join(CSRC, src)] + _deps()):
            subprocess.check_call([nvcc] + NVCC_FLAGS + extra + ["-c", "-o", obj, os.path.join(CSRC, src)], cwd=CSRC)
        return obj

    with ThreadPoolExecutor(len(SOURCES)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    subprocess.check_call([nvcc] + ARCH + ["-shared", "-o", LIB] + objs, cwd=CSRC)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
