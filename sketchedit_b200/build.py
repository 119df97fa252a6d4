"""Build libsketchedit_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

    python -m sketchedit_b200.build [--force]

nvcc cross-compiles without a GPU. The library links only cudart (the tensor-map encoder is
fetched from the driver at run time through cudaGetDriverEntryPoint), so it loads in a process
without libcuda -- it just cannot run anything there.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsketchedit_b200.so")
SOURCES = ["se_engine.cu", "se_conv_c8.cu", "se_cam.cu", "se_conv_direct.cu", "se_misc.cu", "se_split.cu", "se_gemm_split.cu", "se_resize.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]
# the resize coefficient tables must round exactly like Pillow's: no fused multiply-adds in their host code
SOURCE_FLAGS = {"se_resize.cu": ["-Xcompiler", "-ffp-contract=off"]}


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(HERE), "include", "sketchedit_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=True):
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")] + os.environ.get("SE_NVCC_EXTRA", "").split()   # A/B builds (-DSE_...)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + flags + SOURCE_FLAGS.get(src, []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s" % (" ".join(cmd), out))
        if verbose and out.strip():
            print(out)
    out_lib = os.environ.get("SE_LIB_OUT", LIB)   # A/B builds go next to the product library, selected with SE_B200_LIB at load time
    cmd = [nvcc, "-shared", "-o", out_lib] + objs + ["-lcudart"]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    return out_lib


if __name__ == "__main__":
    build(force="--force" in sys.argv)
    print(LIB)
