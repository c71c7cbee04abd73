"""Build libldpcb200.so in-tree with nvcc for sm_100a (called by __graft_entry__.build()).

The persistent kernel is instantiated once per (memory mode, degree path) in its own translation
unit; the units are compiled in parallel and linked into one shared library."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
SRC_DIR = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
OBJ_DIR = os.path.join(os.path.dirname(HERE), "build", "obj")   # cached objects (git- and gpurun-ignored)
LIB = os.path.join(LIB_DIR, "libldpcb200.so")
SOURCES = (["ldpcb200.cu"] + ["bp_inst_m%d_b%d.cu" % (m, b) for m in (0, 1, 2) for b in (0, 1)]
           + ["bp_inst_m%d_b0_minsum.cu" % m for m in (0, 1, 2)] + ["bp_inst_m%d_b0_fast.cu" % m for m in (0, 1, 2)] + ["bp_inst_single.cu", "bp_inst_single_minsum.cu", "bp_inst_smem.cu", "bp_inst_smem_minsum.cu",
              "bp_inst_single_fast.cu", "bp_inst_smem_fast.cu"])
KERNEL_HEADERS = ["bp_math.cuh", "bp_kernel.cuh", "bp_smem.cuh", "bp_smem_inst.cuh", "bp_launch.h", "bp_launch_inst.cuh",
                  "bp_filter.cuh", "bp_single.h", "bp_single.cuh", "bp_single_inst.cuh", "../../include/ldpcb200.h"]
HEADERS = KERNEL_HEADERS + ["formats.cuh", "osd.cuh", "bpots.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",            # never contract a*b+c: every FP64 op of the parity path is rounded separately
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(SRC_DIR, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    pid = os.getpid()

    def compile_one(src):
        # objects are cached next to the library; a unit is recompiled when it or a header it includes changed
        obj = os.path.join(OBJ_DIR, "%s.o" % src[:-3])
        deps = [os.path.join(SRC_DIR, f) for f in [src] + (HEADERS if src == "ldpcb200.cu" else KERNEL_HEADERS)]
        deps.append(os.path.abspath(__file__))
        if not force and os.path.exists(obj) and all(os.path.getmtime(d) <= os.path.getmtime(obj) for d in deps):
            return src, obj, "(cached) " + obj, 0, ""
        tmp_obj = obj + ".tmp.%d" % pid
        cmd = [nvcc] + NVCC_FLAGS + ["-c", "-o", tmp_obj, os.path.join(SRC_DIR, src)]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode == 0:
            os.replace(tmp_obj, obj)
        elif os.path.exists(tmp_obj):
            os.remove(tmp_obj)
        return src, obj, " ".join(cmd), res.returncode, res.stdout

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    log = []
    ok = True
    for src, obj, cmd, rc, out in results:
        log.append(cmd + "\n" + out)
        ok &= rc == 0
    tmp = LIB + ".tmp.%d" % pid
    if ok:
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + [r[1] for r in results]
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        log.append(" ".join(cmd) + "\n" + res.stdout)
        ok &= res.returncode == 0
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose or not ok:
        sys.stderr.write("\n".join(log)[-8000:])
    if not ok:
        raise RuntimeError("nvcc failed (see %s)" % os.path.join(LIB_DIR, "build.log"))
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
