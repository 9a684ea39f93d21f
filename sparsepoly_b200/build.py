"""Builds sparsepoly_b200/libsparsepoly_b200.so from csrc/*.cu with nvcc for sm_100a.

    python -m sparsepoly_b200.build [--force]

-fmad=false: the reference (numba) never contracts a*b+c; parity at 1e-9 / identical support
sets is easier to argue with identical rounding of the scalar chains.
-cudart shared: the library must share the CUDA runtime instance (current device, primary
context) with PyTorch, which only holds the device tensors.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INC = os.path.join(HERE, "..", "include")
OUT = os.path.join(HERE, "libsparsepoly_b200.so")
OBJ = os.path.join(HERE, "csrc", "_obj")
SOURCES = ["errors.cu", "rows.cu", "plan.cu", "regcache.cu", "wplan.cu", "pcd.cu", "pcd_window.cu", "pbcd.cu", "pbcd_window.cu", "psgd.cu", "psgd_plan.cu", "objective.cu", "input.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
              "-fmad=false", "-Xcompiler", "-fPIC", "-I", INC, "-I", CSRC]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libsparsepoly_b200.so")
    return nvcc


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".inc"))]
    deps.append(os.path.join(INC, "sparsepoly_b200.h"))
    return any(os.path.getmtime(p) > t for p in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return OUT
    nvcc = _nvcc()
    os.makedirs(OBJ, exist_ok=True)
    extra = ["-DSP_WPROF=" + os.environ["SP_WPROF"]] if os.environ.get("SP_WPROF") else []     # debug: engine cycle accounting
    if os.environ.get("SP_DEFS"):                                     # debug: extra -D switches
        extra += ["-D" + x for x in os.environ["SP_DEFS"].split(",")]

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    link = [nvcc, "-shared", "-cudart", "shared", "-gencode", "arch=compute_100a,code=sm_100a",
            "-Xlinker", "-rpath,/usr/local/cuda/lib64", "-o", OUT] + objs
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
