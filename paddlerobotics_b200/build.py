"""In-tree build of the sm_100a CUDA library (csrc/libb2q.so).  nvcc cross-compiles without a GPU."""
import os
import subprocess

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB = os.path.join(CSRC, "libb2q.so")
SOURCES = ["b2q_api.cu", "b2q_mlp.cu", "b2q_es.cu", "b2q_sac.cu", "b2q_rpm.cu"]
HEADERS = ["b2q_sim.cuh", "b2q_math.cuh", "b2q_host_common.h", "b2q_model_host.h", "b2q_tc.cuh", "b2q_philox.cuh", "../../include/b2q.h", "../../include/b2q_mlp.h", "../../include/b2q_es.h", "../../include/b2q_sac.h", "../../include/b2q_rpm.h", "b2q_mlp_internal.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for f in SOURCES + HEADERS:
        p = os.path.join(CSRC, f)
        if os.path.exists(p) and os.path.getmtime(p) > t:
            return True
    return False


def build(force=False, verbose=False):
    """Compiles every CUDA source for sm_100a into csrc/libb2q.so."""
    if not force and not _stale():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + srcs
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force=True, verbose="-v" in sys.argv))
