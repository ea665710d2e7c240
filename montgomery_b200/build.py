"""In-tree build of the CUDA engine: nvcc -> montgomery_b200/libmontgomery_b200.so (sm_100a only).

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.  Rebuilds only when a
source is newer than the library.  `python -m montgomery_b200.build [--force]`.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmontgomery_b200.so")
OBJDIR = os.path.join(HERE, "build")
SOURCES = ["msm.cu", "tools.cu"]
HEADERS = ["ptx.cuh", "field.cuh", "ec.cuh", "coop.cuh", "warp.cuh", "onewarp.cuh", "engine.cuh", "constants_gen.cuh", os.path.join("..", "..", "include", "montgomery_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for f in SOURCES + HEADERS + ["../gen_constants.py"]:
        p = os.path.join(CSRC, f)
        if os.path.exists(p) and os.path.getmtime(p) > t:
            return True
    return False


def build(force=False, verbose=False, variant=None, extra_flags=()):
    """variant=None: the product library.  variant="name": an experiment build with extra_flags (e.g.
    ("-DMGB_COOP_WARP_MUL=1",)) -> libmontgomery_b200_<name>.so, loaded only when MGB_LIB points at it."""
    lib_path, objdir = LIB, OBJDIR
    if variant:
        lib_path = os.path.join(HERE, "libmontgomery_b200_%s.so" % variant)
        objdir = os.path.join(OBJDIR, variant)
        force = True
    if not force and not needs_build():
        return LIB
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        # MGB_NVCC_EXTRA: extra flags for experiments (e.g. -DMGB_MINB=5)
        cmd = [nvcc] + NVCC_FLAGS + os.environ.get("MGB_NVCC_EXTRA", "").split() + list(extra_flags) + ["-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(objdir, src + ".ptxas.log")
        with open(log, "w") as fh:
            fh.write(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, (res.stdout + res.stderr)[-4000:]))
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", lib_path] + objs + ["-lcudart"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    if verbose:
        print("built", lib_path)
    return lib_path


if __name__ == "__main__":
    # python -m montgomery_b200.build [--force] [--variant NAME -DFLAG ...]
    if "--variant" in sys.argv:
        i = sys.argv.index("--variant")
        build(verbose=True, variant=sys.argv[i + 1], extra_flags=[a for a in sys.argv[i + 2:] if a.startswith("-")])
    else:
        build(force="--force" in sys.argv, verbose=True)
