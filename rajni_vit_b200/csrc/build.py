"""Build librajni_b200.so (the model) and librajni_jpeg.so (the GPU JPEG decoder) in-tree with nvcc for sm_100a
(cross-compiles without a GPU).  runtime.cu (error string, launch plumbing) is linked into both."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "librajni_b200.so")
JPEG_LIB = os.path.join(HERE, "librajni_jpeg.so")
LIBS = {
    LIB: ["runtime.cu", "capi.cu", "score_select.cu", "rowops.cu", "resize.cu", "gemm_tcgen05.cu", "attention.cu",
          "attention_pipe.cu", "attention_tc.cu", "attention_long.cu"],
    JPEG_LIB: ["runtime.cu", "jpeg.cu"],
}
SOURCES = list(dict.fromkeys(s for srcs in LIBS.values() for s in srcs))
HEADERS = ["common.cuh", os.path.join(ROOT, "include", "rajni_b200.h"), os.path.join(ROOT, "include", "rajni_jpeg.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else "nvcc"


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    hdrs = [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
    jobs = []
    for src in SOURCES:
        s = os.path.join(HERE, src)
        o = os.path.join(HERE, src[:-3] + ".o")
        if force or _stale(o, [s] + hdrs):
            cmd = [_nvcc(), *NVCC_FLAGS, "-c", s, "-o", o]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        for out in ex.map(run, jobs):
            if verbose and out:
                print(out, file=sys.stderr)
    for lib, srcs in LIBS.items():
        objs = [os.path.join(HERE, src[:-3] + ".o") for src in srcs]
        if force or jobs or _stale(lib, objs):
            run([_nvcc(), "-shared", "-o", lib, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
