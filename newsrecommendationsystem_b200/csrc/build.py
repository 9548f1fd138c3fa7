"""Build libnrms_b200.so (sm_100a only) in-tree with nvcc.  Usage: python build.py [--force] [-v]"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
OUT = os.path.join(PKG, "libnrms_b200.so")
OBJ = os.path.join(HERE, "_obj")
SOURCES = ["encoder.cu", "misc.cu", "pack.cu", "tc_gemm.cu", "fused_host.cu", "tc_fused3.cu", "tc_fused7.cu", "k1g_table_attn.cu",
           "k1f_attn_pool.cu", "exp1.cu", "recommend.cu", "attn_mma.cu", "topk.cu",
           "attn_cross.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _deps():
    return [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cu", ".cuh"))] + \
           [os.path.join(PKG, "..", "include", "nrms_b200.h")]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    os.makedirs(OBJ, exist_ok=True)
    extra = ["-Xptxas", "-v"] if verbose else []
    if os.environ.get("NRMS_K1_TRACE"):
        extra.append("-DNRMS_K1_TRACE")
    for d in os.environ.get("NRMS_DEFINES", "").split():
        extra.append("-D" + d)

    def cc(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + extra + ["-c", os.path.join(HERE, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(cc, SOURCES))
    cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
