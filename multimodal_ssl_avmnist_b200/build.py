"""Builds libavmnist_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m multimodal_ssl_avmnist_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libavmnist_b200.so")
SOURCES = ["core.cu", "loss.cu", "augment.cu", "encoder.cu", "linear.cu", "conv_tc.cu", "act8.cu", "gemm_tc.cu", "knn.cu", "dp.cu", "mix.cu", "probe.cu"]  # missing files are skipped
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(obj, src):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "avmnist_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ for sm_100a and link the shared library.  Returns the library path."""
    nvcc = _nvcc()
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    objs = []
    procs = []
    for name in SOURCES:
        src = os.path.join(CSRC, name)
        if not os.path.exists(src):
            continue
        obj = os.path.join(HERE, "build", name.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, src):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
            procs.append((name, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    relink = force or not os.path.exists(LIB) or bool(procs)
    for name, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {name}")
        with open(os.path.join(HERE, "build", name.replace(".cu", ".ptxas.log")), "w") as f:
            f.write(out)
    if relink or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-ldl"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
