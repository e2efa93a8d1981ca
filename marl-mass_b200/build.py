"""Build the sm_100a shared library in-tree with nvcc (cross-compiles without a GPU).

    python -m marl_mass_b200.build        # or: python marl-mass_b200/build.py

Output: marl-mass_b200/_build/libmarl_mass_b200.so (git-ignored, travels to the GPU box with gpurun).
-fmad=false: the float64 reference never fuses a*b+c; keeping products and sums separately rounded is what
makes every threshold decision reproduce the reference (DESIGN.md "Numerics").
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libmarl_mass_b200.so")
SOURCES = ["merge_step.cu", "merge_step_occ4.cu", "merge_step_spec_mass.cu", "merge_step_spec_hss.cu", "merge_step_spec_mass4.cu", "merge_step_spec_hss4.cu", "merge_coop.cu", "merge_outputs.cu", "actor_sample.cu", "supervisor.cu", "learner.cu", "optim.cu", "eval_record.cu", "capi.cu"]
HEADERS = [os.path.join(CSRC, "mm_internal.h"), os.path.join(CSRC, "mm_device.cuh"), os.path.join(CSRC, "supervisor_core.h"),
           os.path.join(CSRC, "spawn_core.h"),
           os.path.join(HERE, "..", "include", "marl_mass_b200.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libmarl_mass_b200.so")
    os.makedirs(OUT_DIR, exist_ok=True)
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-I", os.path.join(HERE, "..", "include"), "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return LIB


def build_variant(name, defines, verbose=False):
    """Experiment build: _build/variants/lib_<name>.so with extra -D knobs (select it with MM_LIB_PATH)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out_dir = os.path.join(OUT_DIR, "variants")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, "lib_%s.so" % name)
    cmd = [nvcc] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + \
          ["-I", os.path.join(HERE, "..", "include"), "-o", out] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    if "--variant" in sys.argv:   # python build.py --variant NAME [KNOB=VALUE ...]
        k = sys.argv.index("--variant")
        print(build_variant(sys.argv[k + 1], [a for a in sys.argv[k + 2:] if "=" in a], verbose="-v" in sys.argv))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
