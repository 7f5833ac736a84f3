"""Build visionworkbench_b200/libvwb200.so (sm_100a only) with nvcc, in-tree.

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(ROOT, "build", "obj")
SO = os.path.join(HERE, "libvwb200.so")
SOURCES = ["engine.cu", "k1_generic.cu", "k1_zone_int.cu", "k1_fast.cu", "k1_screen.cu", "k2_pyramid.cu", "k34_filters.cu", "k5_sgm.cu", "k5_sgm_paths.cu", "shard.cu", "k6_subpixel.cu", "k7_corr_eval.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"] + os.environ.get("VWB200_NVCC_EXTRA", "").split()


def nvcc():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found")
    return p


def _deps(src):
    hdr = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdr.append(os.path.join(ROOT, "include", "vwb200.h"))
    return [src] + hdr


def _compile(name, verbose):
    src = os.path.join(CSRC, name)
    obj = os.path.join(OBJ, name.replace(".cu", ".o"))
    if os.path.exists(obj) and all(os.path.getmtime(d) <= os.path.getmtime(obj) for d in _deps(src)):
        return obj, False
    cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {name}:\n{r.stdout}\n{r.stderr}")
    if verbose:
        sys.stderr.write(r.stderr)
    return obj, True


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    with concurrent.futures.ThreadPoolExecutor(max_workers=8) as ex:
        res = list(ex.map(lambda n: _compile(n, verbose), SOURCES))
    objs = [o for o, _ in res]
    if any(ch for _, ch in res) or not os.path.exists(SO):
        # exported symbols are the extern "C" ABI only (default visibility is set in the header macro below)
        cmd = [nvcc(), "-shared", "-o", SO] + objs + ["-Xcompiler", "-fPIC", "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
