"""Builds csrc/lible_b200.so for sm_100a with nvcc (cross-compiles without a GPU).

    python learning_environments_b200/csrc/build.py [--force] [--verbose]

One object per translation unit, compiled in parallel; -lineinfo so ncu's source page maps to the .cu files.
"""
import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["le_api.cu", "le_general.cu", "le_td3.cu", "le_tc.cu", "le_inst_cp_tanh.cu", "le_inst_cp_leaky.cu", "le_inst_ac_tanh.cu", "le_inst_ac_leaky.cu"]
HEADERS = ["le_common.cuh", "le_lane.cuh", "le_envpack.cuh", "le_inner_loop.cuh", "le_instance.cuh", "le_cta_lane.cuh", "le_general.cuh", "le_tc.cuh", "le_general_api.h", "le_td3_api.h",
           os.path.join("..", "..", "include", "le_b200.h")]
OUT = os.path.join(HERE, os.environ.get("LE_LIB_NAME", "lible_b200.so"))
# a library built under another name (LE_LIB_NAME, e.g. an older build kept for an A/B run, selected by the same variable at run
# time) keeps its objects apart from the default build
OBJDIR = os.path.join(HERE, "build") if os.path.basename(OUT) == "lible_b200.so" else os.path.join(HERE, "build", os.path.basename(OUT) + ".d")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
EXTRA = os.environ.get("LE_NVCC_EXTRA", "").split()
FLAGS = EXTRA + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
         "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def _newest(paths):
    return max(os.path.getmtime(os.path.join(HERE, p)) for p in paths)


def _compile(src, verbose):
    obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
    cmd = [NVCC] + FLAGS + ["-c", os.path.join(HERE, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = r.stdout + r.stderr
    with open(obj + ".log", "w") as f:
        f.write(log)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (src, log[-6000:]))
    if verbose:
        print(log)
    return obj


def build(force=False, verbose=False):
    os.makedirs(OBJDIR, exist_ok=True)
    if not force and os.path.isfile(OUT) and os.path.getmtime(OUT) > _newest(SOURCES + HEADERS + ["build.py"]):
        return OUT
    with cf.ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
