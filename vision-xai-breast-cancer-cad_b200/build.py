"""Build libbcad.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python vision-xai-breast-cancer-cad_b200/build.py [--force] [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libbcad.so")
SOURCES = ["api.cu", "kernels_fp32.cu", "tensor_path.cu", "sm100_selftest.cu", "sm100_kernels.cu", "sm100_wide.cu", "sm100_tail.cu", "sm100_fused.cu", "sm100_fused2.cu", "kernels_train.cu", "sm100_train.cu", "api_train.cu", "refine.cu", "sm100_unet.cu", "saliency.cu"]
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _deps():
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    files.append(os.path.join(HERE, "..", "include", "bcad.h"))
    return files


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(f) > t for f in _deps())


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [nvcc, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
