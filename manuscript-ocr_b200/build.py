"""Build libmanuscript_b200.so (the sm_100a kernels + the C ABI of include/manuscript_b200.h) in-tree.

    python manuscript-ocr_b200/build.py [--force] [--verbose]

nvcc cross-compiles for sm_100a without a GPU.  --fmad=false is part of the contract: the reference's
numpy / numba arithmetic never contracts a*b+c, and keep / suppress decisions must be bit-identical.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
OUT = os.path.join(HERE, "manuscript_b200", "libmanuscript_b200.so")
SOURCES = ["api.cu", "decode.cu", "sort.cu", "lanms.cu", "boxes.cu", "reading_order.cu", "crop.cu",
           "quadcrop.cu", "tps.cu", "np_sum_test.cu", "jpeg.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "--fmad=false", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static"]
OBJ_DIR = os.path.join(HERE, "build")


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
           [os.path.join(INCLUDE, "manuscript_b200.h"), __file__]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "manuscript_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None, obj_dir=None):
    """One object per .cu (compiled in parallel, rebuilt only when the source or a header is newer), then one link.
    `defines` / `out` / `obj_dir` build an experiment variant (extra -D flags) next to the product library."""
    global OUT, OBJ_DIR
    if out is not None:
        OUT, OBJ_DIR, force = out, obj_dir or (out + ".obj"), True
    if not force and not needs_build():
        return OUT
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_t = max(os.path.getmtime(h) for h in _headers())
    jobs, objs = [], []
    for src in SOURCES:
        s, o = os.path.join(CSRC, src), os.path.join(OBJ_DIR, src[:-3] + ".o")
        objs.append(o)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr_t):
            cmd = [_nvcc(), *NVCC_FLAGS, *[f"-D{d}" for d in defines], "-I", INCLUDE, "-c", "-o", o, s]
            if verbose:
                cmd[1:1] = ["-Xptxas", "-v"]
                print(" ".join(cmd))
            jobs.append((src, subprocess.Popen(cmd)))
    failed = [src for src, p in jobs if p.wait() != 0]
    if failed:
        raise subprocess.CalledProcessError(1, f"nvcc -c {failed}")
    subprocess.run([_nvcc(), *LINK_FLAGS, "-o", OUT, *objs], check=True)
    return OUT


if __name__ == "__main__":
    # python build.py [--force] [--verbose] [--variant NAME -DFOO=1 ...]  (variant -> manuscript_b200/libvariant_NAME.so)
    args = sys.argv[1:]
    if "--variant" in args:
        name = args[args.index("--variant") + 1]
        defs = [a[2:] for a in args if a.startswith("-D")]
        print(build(defines=defs, out=os.path.join(HERE, "manuscript_b200", f"libvariant_{name}.so"),
                    obj_dir=os.path.join(HERE, "build", f"variant_{name}")))
    else:
        print(build(force="--force" in args, verbose="--verbose" in args))
