"""Builds libb200edit.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python diffusion-image-editing_b200/b200edit/build.py [--force]
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "csrc")
OUT = os.path.join(HERE, "libb200edit.so")
OBJ = os.path.join(HERE, "_obj")
SOURCES = ["step_kernels.cu", "guidance_heads.cu", "mask_kernels.cu", "conv_igemm.cu", "flash_attn.cu", "attention.cu", "unet_kernels.cu", "resnet_kernels.cu", "lpips_kernels.cu", "unet.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC,-ffp-contract=off", "--expt-relaxed-constexpr",
         "-Xptxas", "-v"]


def _deps():
    out = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    out.append(os.path.join(os.path.dirname(os.path.dirname(HERE)), "include", "b200edit.h"))
    return out


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    os.makedirs(OBJ, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        with open(obj + ".ptxas.txt", "w") as f:
            f.write(r.stderr)
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [NVCC, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xcompiler", "-fPIC", "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
