"""Builds libavh_b200.so (hand-written sm_100a CUDA + the C ABI of include/avh_b200.h) in-tree with nvcc.

`python -m multimodalvc_b200.build` or `multimodalvc_b200.build.build()`.  nvcc cross-compiles without a
GPU; the resulting .so sits next to this file so that it travels with the source tree.
"""
import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libavh_b200.so")
SOURCES = ["api.cu", "gemm_tcgen05.cu", "conv_window.cu", "conv_frame.cu", "stem_fused.cu", "attention.cu", "attention_tc.cu", "elementwise.cu", "train_ops.cu", "train_dropout.cu", "pretrain_ops.cu", "qformer.cu", "backward_ops.cu", "frontend_train.cu", "refresh.cu", "fbank.cu"]
NVCC_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
              "-I", os.path.join(ROOT, "include"), "-I", CSRC,
              # host packers round every fp32 operation on its own, as the device refresh kernels do (bit-identical
              # BatchNorm folds); x86-64 without -march has no FMA anyway, this keeps it so on hosts that do
              "-Xcompiler", "-ffp-contract=off"]
NVCC_FLAGS += os.environ.get("AVH_NVCC_EXTRA", "").split()      # e.g. -DAVH_STALL_ACC for tools/gemm_stall.py


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libavh_b200.so cannot be built")
    return exe


def _stamp():
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)) + ["../../include/avh_b200.h"]:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library.  Returns the library path."""
    os.makedirs(OBJ, exist_ok=True)
    stamp_file = os.path.join(OBJ, "stamp")
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
