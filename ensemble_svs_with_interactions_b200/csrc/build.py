"""Builds libsvsk.so in-tree with nvcc for sm_100a (cross-compiles on GPU-less machines).

    python -m ensemble_svs_with_interactions_b200.csrc.build [--force]
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["svsk_api.cu", "simt_f32.cu", "tma_util.cu", "diffnet_pack.cu", "diffnet_block3_sm100.cu", "diffnet_stack_sm100.cu", "diffnet_stack_duo_sm100.cu",
           "diffnet_step_sm100.cu", "diffnet_train_sm100.cu", "linear_sm100.cu", "usfgan_block_sm100.cu", "usfgan_block_fr_sm100.cu", "conv1d_sm100.cu", "usfgan_front.cu",
           "lstm_sm100.cu", "encoder_sm100.cu", "postproc.cu", "wavenet_f32.cu",
           "wavenet_ar_sm100.cu", "wavenet_train_sm100.cu", "lstm_train_sm100.cu", "encoder_train_sm100.cu"]
LIB = os.path.join(HERE, "libsvsk.so")
# micro-benchmarks behind tools/ubench_*.py: their own library, NOT part of the product libsvsk.so
TOOLS = os.path.join(HERE, "..", "..", "tools")
UBENCH_LIB = os.path.join(TOOLS, "libsvsk_ubench.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _deps_mtime():
    files = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cu", ".cuh"))]
    files.append(os.path.join(HERE, "..", "..", "include", "svsk.h"))
    return max(os.path.getmtime(f) for f in files)


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _deps_mtime():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(HERE, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose and r.stderr:
            print(r.stderr, file=sys.stderr)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


def build_ubench(force: bool = False) -> str:
    """tools/libsvsk_ubench.so: tools/ubench_sm100.cu + the error-string helpers of svsk_api.cu."""
    src = os.path.join(TOOLS, "ubench_sm100.cu")
    if not force and os.path.exists(UBENCH_LIB) and os.path.getmtime(UBENCH_LIB) >= max(_deps_mtime(), os.path.getmtime(src)):
        return UBENCH_LIB
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", HERE, "-shared", "-o", UBENCH_LIB, src, os.path.join(HERE, "svsk_api.cu"),
           "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for ubench:\n{r.stdout}\n{r.stderr}")
    return UBENCH_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    if "--ubench" in sys.argv:
        print(build_ubench(force="--force" in sys.argv))
