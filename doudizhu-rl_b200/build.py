"""Build libddz_b200.so (sm_100a only) in-tree with nvcc.  Cross-compiles without a GPU."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = [os.path.join(HERE, "csrc", f) for f in ("ddz_kernels.cu", "ddz_device.cuh", "ddz_flat.cuh", "ddz_ids.cuh",
                                                "ddz_action_ids.inc", "ddz_policy.cuh", "ddz_policy_linear.cuh")] + \
      [os.path.join(ROOT, "include", "ddz_b200.h")]
LIB = os.path.join(HERE, "libddz_b200.so")
LIB_FORM_B = os.path.join(HERE, "libddz_b200_formB.so")   # the other layout of the probability planes (-DDDZ_PROB_FORM_B)

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")
    return p


def build_native(force=False, verbose=False, form_b=False):
    lib = LIB_FORM_B if form_b else LIB
    if not force and os.path.exists(lib) and all(os.path.getmtime(lib) >= os.path.getmtime(s) for s in SRC):
        return lib
    cmd = [nvcc_path()] + NVCC_FLAGS + (["-DDDZ_PROB_FORM_B"] if form_b else []) + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", lib, SRC[0]]
    subprocess.check_call(cmd)
    return lib


def build_all(force=True):
    """both layouts of the library (default + -DDDZ_PROB_FORM_B), compiled side by side"""
    cmds = []
    for form_b, lib in ((False, LIB), (True, LIB_FORM_B)):
        if not force and os.path.exists(lib) and all(os.path.getmtime(lib) >= os.path.getmtime(s) for s in SRC):
            continue
        cmds.append(subprocess.Popen([nvcc_path()] + NVCC_FLAGS + (["-DDDZ_PROB_FORM_B"] if form_b else []) + ["-o", lib, SRC[0]]))
    for p in cmds:
        if p.wait() != 0:
            raise RuntimeError("nvcc failed (exit code %d)" % p.returncode)
    return LIB, LIB_FORM_B


if __name__ == "__main__":
    print(build_native(force=True, verbose=True))
