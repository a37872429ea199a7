"""Builds libb200unet.so (the C-ABI CUDA library, include/b2u.h) in-tree with nvcc for sm_100a, and next to it
libb200unet_fp32.so, the fp32 VALIDATION build of the same ABI (csrc/validation_fp32.cu: NHWC fp32 tensors, CUDA-core
FMA contractions; loaded only by ops.set_validation_fp32 / B2U_FP32_VALIDATION=1, never on the product path).

Usage: python unet-pytorch_b200/build.py [--force]
The .so files are git-ignored but travel to the GPU box with the gpurun snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libb200unet.so")
OUT_FP32 = os.path.join(HERE, "libb200unet_fp32.so")
# the loss / metric / optimizer kernels compute in fp32 already and are shared; -DB2U_FP32_VALIDATION drops the bf16 head
SOURCES_FP32 = ["runtime.cu", "head_loss.cu", "hist.cu", "optim.cu", "dw_se.cu", "letterbox.cu", "render.cu",
                "validation_fp32.cu"]
SOURCES = ["runtime.cu", "conv_igemm.cu", "conv_wgrad.cu", "elementwise.cu", "head_loss.cu", "hist.cu", "optim.cu", "bn.cu", "resnet_ops.cu", "dw_se.cu",
           "letterbox.cu", "render.cu", "input_grad.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xptxas=-v",  # no --use_fast_math: precise math everywhere; -v prints registers/spills
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale():
    if not os.path.exists(OUT) or not os.path.exists(OUT_FP32):
        return True
    t = min(os.path.getmtime(OUT), os.path.getmtime(OUT_FP32))
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return OUT
    nvcc = _nvcc()
    objs = []
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        sp = os.path.join(CSRC, src)
        if not os.path.exists(sp):
            continue
        obj = os.path.join(bdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-I", CSRC, "-c", sp, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs32 = []
    for src in SOURCES_FP32:
        obj = os.path.join(bdir, src.replace(".cu", "_fp32.o"))
        objs32.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-DB2U_FP32_VALIDATION", "-I", CSRC, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src + " (fp32 validation)", subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    for out, oo in ((OUT, objs), (OUT_FP32, objs32)):
        cmd = [nvcc, "-shared", "-o", out, *oo, "-gencode", "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout)
            raise RuntimeError("link failed")
    with open(os.path.join(bdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
