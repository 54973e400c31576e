"""In-tree build of libdifflinker_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libdifflinker_b200.so")
SOURCES = ["dl_engine.cu", "output_stage.cu"]
HEADERS = ["common.cuh", "size_gnn.cuh", "kernels_simt.cuh", "kernels_tc.cuh", "kernels_node_tc.cuh", "kernels_edge_v3.cuh", "diffusion_loss.cuh", os.path.join("..", "..", "include", "difflinker_b200.h")]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    return None


def is_stale() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    for f in SOURCES + HEADERS:
        p = os.path.join(CSRC, f)
        if os.path.isfile(p) and os.path.getmtime(p) > t:
            return True
    return False


def build_native(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    nvcc = nvcc_path()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libdifflinker_b200.so")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-Xcompiler", "-fPIC", "-shared", "-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), file=sys.stderr)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed:\n{res.stdout}\n{res.stderr}")
    if verbose:
        print(res.stderr, file=sys.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose=True))
