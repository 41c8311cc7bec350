"""Build libphotoverse_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m photoverse_b200.build [--force] [--verbose]

The shared object lands next to this file (photoverse_b200/libphotoverse_b200.so) so that it travels with the
source tree; object files go to photoverse_b200/csrc/build/ (git-ignored).
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(CSRC, "build")
LIB_PATH = os.path.join(HERE, "libphotoverse_b200.so")
SOURCES = ["pv_api.cu", "pv_gemm.cu", "pv_gemm3.cu", "pv_attn3.cu", "pv_attn4.cu", "pv_attn6.cu", "pv_simt.cu", "pv_pack.cu", "pv_adapter.cu", "pv_bwd.cu", "pv_bwd_mma.cu", "pv_bwd_tc.cu", "pv_lora_bwd.cu", "pv_loss.cu", "pv_sattn.cu", "pv_backbone.cu", "pv_convert.cu", "pv_ip_mask.cu"]
HEADERS = ["pv_common.cuh", "pv_softmax.cuh", "pv_outproj.cuh", "pv_host.h", os.path.join("..", "..", "include", "photoverse_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
if os.environ.get("PV_TRACE"):          # debug build: the persistent attention kernels record a device timeline;
    NVCC_FLAGS.append("-DPV_TRACE")     # separate objects and library (load it with PV_LIB_PATH=...)
    OBJ_DIR = os.path.join(CSRC, "build_trace")
    LIB_PATH = os.path.join(HERE, "libphotoverse_b200_trace.so")


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=...)")


def _newest_header_mtime() -> float:
    return max(os.path.getmtime(os.path.join(CSRC, h)) for h in HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_m = _newest_header_mtime()
    sources = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(src):
        srcp = os.path.join(CSRC, src)
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(srcp), hdr_m):
            return obj, ""
        cmd = [nvcc] + NVCC_FLAGS + ["-c", srcp, "-o", obj]
        r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        with open(obj + ".ptxas.log", "w") as f:
            f.write(r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        results = list(ex.map(compile_one, sources))
    objs = [o for o, _ in results]
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    need_link = force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(o) > os.path.getmtime(LIB_PATH) for o in objs)
    if need_link:
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
