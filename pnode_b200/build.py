"""In-tree build of the C-ABI CUDA library (sm_100a only).  `python -m pnode_b200.build [--force] [-v]`.

Every .cu is compiled to an object under csrc/_obj/ (in parallel, only when stale) and the objects are linked into
csrc/libpnode_b200.so, which travels with the tree (git-ignored, not gpurun-ignored)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
# (source, object, extra flags): conv_block.cu is the long pole, so its fp32 and fp64 instantiations compile as two objects
# and mlp_rk.cu compiles once per group of (dim, hidden) shapes (part 0 = the spiral shape + the C entry points)
UNITS = [("vecops.cu", "vecops.o", []), ("mlp_rk.cu", "mlp_rk.o", ["-DPNODE_MLP_PART=0"]),
         ("mlp_rk.cu", "mlp_rk_p1.o", ["-DPNODE_MLP_PART=1"]), ("mlp_rk.cu", "mlp_rk_p2.o", ["-DPNODE_MLP_PART=2"]),
         ("mlp_rk.cu", "mlp_rk_p3.o", ["-DPNODE_MLP_PART=3"]), ("cnf_rk.cu", "cnf_rk.o", []),
         ("bn_relu.cu", "bn_relu.o", []), ("umma_gemm.cu", "umma_gemm.o", []),
         ("dense_mlp.cu", "dense_mlp.o", []), ("cnf_net.cu", "cnf_net.o", []), ("conv_mma.cu", "conv_mma.o", []), ("conv_block.cu", "conv_block_f32.o", ["-DPNODE_CB_PART=1"]),
         ("conv_block.cu", "conv_block_f64.o", ["-DPNODE_CB_PART=2"])]
SOURCES = sorted({u[0] for u in UNITS})
HEADERS = ["common.cuh", "umma.cuh", "pdl.cuh", "f32x2.cuh", os.path.join("..", "..", "include", "pnode_b200.h")]
LIB = os.path.join(CSRC, "libpnode_b200.so")
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC"]


def _mtime(path):
    return os.path.getmtime(path) if os.path.exists(path) else 0.0


def _compile(nvcc, unit, verbose):
    src, objname, extra = unit
    obj = os.path.join(OBJ, objname)
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    proc = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), proc.stderr))
    if verbose:
        print(proc.stderr)
    return obj


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = max(_mtime(os.path.join(CSRC, h)) for h in HEADERS)
    objs, todo = [], []
    for unit in UNITS:
        obj = os.path.join(OBJ, unit[1])
        objs.append(obj)
        if force or _mtime(obj) < max(_mtime(os.path.join(CSRC, unit[0])), hdr_t):
            todo.append(unit)
    if todo:
        with ThreadPoolExecutor(max_workers=min(len(todo), os.cpu_count() or 1)) as ex:
            list(ex.map(lambda s: _compile(nvcc, s, verbose), todo))
    if todo or _mtime(LIB) < max(_mtime(o) for o in objs):
        cmd = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
        proc = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
        if proc.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (" ".join(cmd), proc.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
