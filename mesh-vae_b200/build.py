"""Build libmvb_sm100a.so in-tree with nvcc (sm_100a only; cross-compiles without a GPU)."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libmvb_sm100a.so")
SOURCES = ["mvb_api.cu", "mvb_spmm.cu", "mvb_contract.cu", "mvb_loss.cu", "mvb_optim.cu", "mvb_tc.cu", "mvb_dense.cu", "mvb_layer.cu", "mvb_mesh_tc.cu", "mvb_stream_tc.cu", "mvb_dp.cu", "mvb_opgrad.cu"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "mvb.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
           "-Xcompiler", "-fPIC,-O3", "-shared", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
           "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
