"""Build libasis_b200.so in-tree for sm_100a (and nothing else).

    python -m adaptersis_b200.build            # incremental
    python -m adaptersis_b200.build --force

nvcc cross-compiles without a GPU; the resulting .so sits next to the package so that it
travels to the GPU box and shows up as a loaded in-tree library.
"""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libasis_b200.so")
BUILD = os.path.join(CSRC, "build")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC",
         "-Xptxas", "-v"]
if os.environ.get("ASIS_TRACE"):      # debug build with in-kernel event stamps (tools/attn_trace8.py, tools/gemm_trace.py):
    FLAGS = FLAGS + ["-DASIS_TRACE"]  # a separate library, loaded with ASIS_LIB=<path>; the product library is untouched
    OUT = os.path.join(HERE, "libasis_b200_trace.so")
    BUILD = os.path.join(CSRC, "build_trace")
SOURCES = ["api.cu", "msda.cu", "norm.cu", "gemm_f32.cu", "attention_f32.cu", "misc.cu", "conv.cu", "gemm_tc.cu", "attention_tc.cu"]


def _deps_mtime():
    m = 0.0
    for d in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(d):
            if f.endswith((".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(d, f)))
    return m


def _compile(src, force, hdr_m):
    obj = os.path.join(BUILD, src[:-3] + ".o")
    spath = os.path.join(CSRC, src)
    if (not force and os.path.exists(obj) and os.path.getmtime(obj) > os.path.getmtime(spath)
            and os.path.getmtime(obj) > hdr_m):
        return src, None
    cmd = [NVCC] + FLAGS + ARCH + ["-c", spath, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(os.path.join(BUILD, src[:-3] + ".ptxas.log"), "w") as f:
        f.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    return src, obj


def build(force=False, verbose=True):
    os.makedirs(BUILD, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    missing = [s for s in SOURCES if s not in srcs]
    if missing:
        raise RuntimeError(f"missing CUDA sources: {missing}")
    hdr_m = _deps_mtime()
    rebuilt = False
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        for src, obj in ex.map(lambda s: _compile(s, force, hdr_m), srcs):
            if obj is not None:
                rebuilt = True
                if verbose:
                    print(f"[build] compiled {src}", file=sys.stderr)
    objs = [os.path.join(BUILD, s[:-3] + ".o") for s in srcs]
    if rebuilt or not os.path.exists(OUT):
        cmd = [NVCC] + ARCH + ["-shared", "-o", OUT] + objs + ["-lcudart_static", "-ldl", "-lpthread", "-lrt"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(f"[build] linked {OUT}", file=sys.stderr)
    return OUT


if __name__ == "__main__":
    build(force="--force" in sys.argv)
