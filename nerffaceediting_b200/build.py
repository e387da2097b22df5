"""Builds libnfe_b200.so in-tree with nvcc for sm_100a (no torch headers: the library is a plain C ABI).

    python -m nerffaceediting_b200.build [--force] [--verbose]

The .so is git-ignored but travels with the repo snapshot to the GPU box.  nvcc cross-compiles
without a GPU, so this also runs in the CPU-only build container.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "_obj")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libnfe_b200.so")
SOURCES = ["nfe_api.cu", "nfe_planes.cu", "nfe_rays.cu", "nfe_field.cu", "nfe_field_tc.cu", "nfe_field_pipe2.cu", "nfe_march.cu", "nfe_render.cu", "nfe_backward.cu", "nfe_field_bwd.cu", "nfe_diag.cu", "nfe_losses.cu", "nfe_stylegan_ops.cu", "nfe_modconv.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc():
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else "nvcc"


def _newest_dep():
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "nfe_b200.h"))
    return max(os.path.getmtime(d) for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library.  Returns the .so path.
    $NFE_NVCC_FLAGS adds flags (e.g. -DNFE_PIPE_PROFILE, the field kernel's role profiler) for experiments on the GPU box."""
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_dep():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    env = dict(os.environ)
    env.pop("CC", None)   # the image exports a gcc wrapper that nvcc must not pick up as host compiler
    env.pop("CXX", None)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + os.environ.get("NFE_NVCC_FLAGS", "").split() + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True, env=env)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    # the arch flag on the link line keeps nvcc's (empty) device-link stub at sm_100a too
    r = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-cudart", "static"],
                       capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
