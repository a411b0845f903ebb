"""Builds libcodenet_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcodenet_b200.so")
SOURCES = ["engine.cu", "pw_gemm.cu", "heads_fused.cu", "unit_fused.cu", "unit_s2_fused.cu", "unit_fused_ws.cu", "dw.cu", "dw_tma.cu", "deform_tile.cu", "stem.cu", "prepost.cu", "decode.cu", "deform_f32.cu", "f32_net.cu", "pw_tf32.cu", "merge.cu", "jpeg.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-Xptxas", "-v", "-Xcudafe", "--diag_suppress=177"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))] + [os.path.join(HERE, "..", "include", "codenet_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    extra = os.environ.get("CDN_NVCC_EXTRA", "").split()      # experiments only (e.g. -DPW_EPI_WARPS=8)
    from concurrent.futures import ThreadPoolExecutor

    def compile_one(src):
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
               [os.path.join(CSRC, src), os.path.join(HERE, "..", "include", "codenet_b200.h")]
        if not force and not extra and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(d) for d in deps):
            return obj, ""                           # up to date
        cmd = [NVCC] + FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed on %s" % src)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        res = list(ex.map(compile_one, SOURCES))
    objs = [r[0] for r in res]
    logs = [r[1] for r in res]
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    if verbose:
        sys.stderr.write("\n".join(logs))
    with open(os.path.join(CSRC, "ptxas.log"), "w") as f:
        f.write("\n".join(logs))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
