"""Build libnvtb200.so in-tree with nvcc for sm_100a (no GPU needed to compile)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libnvtb200.so")
SOURCES = ["scan_kernels.cu", "hashagg.cu", "vocab.cu", "infer.cu", "comm.cu", "groupby.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libnvtb200.so")
    return exe


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "nvtb200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every .cu of the engine into nvtabular_b200/lib/libnvtb200.so."""
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIB_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out.decode()}")
        if verbose and out:
            print(out.decode())
    cmd = [nvcc, "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xcompiler", "-fPIC", "-lcudart", "-ldl"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout.decode()}")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
