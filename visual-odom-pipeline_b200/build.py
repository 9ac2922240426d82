"""Builds libklt_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

    python visual-odom-pipeline_b200/build.py [--force] [--verbose] [--variant NAME --extra "-DFOO ..."]

Every .cu is compiled to its own object (in parallel, rebuilt only when it or a header changed) and the objects are
linked into lib/libklt_b200.so.  `--variant NAME` builds lib/libklt_b200_NAME.so with extra nvcc flags (e.g.
`--variant phases --extra -DKLT_LK_PHASES`, the diagnostics build that scripts/gpu_lk_phases.sh loads through
KLT_LIB_PATH).
"""
import concurrent.futures
import hashlib
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIB_DIR, "libklt_b200.so")
SOURCES = ["klt_pyramid.cu", "klt_lk.cu", "klt_lk_fast.cu", "klt_filter.cu", "klt_corners.cu", "klt_grid.cu", "klt_bilateral.cu", "klt_subpix.cu", "klt_clahe.cu", "klt_capi.cu"]
HEADERS = [os.path.join(CSRC, "klt_common.cuh"), os.path.join(CSRC, "klt_lk_point.cuh"), os.path.join(ROOT, "include", "klt_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",   # B200 only; no PTX for other archs, no fallback
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",            # OpenCV's x86 build rounds every float op once (SURVEY.md A.7)
    "-prec-div=true", "-prec-sqrt=true",
    "-Xcompiler", "-fPIC,-O2,-Wall",
]


def nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def lib_path(variant=None):
    return LIB if not variant else os.path.join(LIB_DIR, "libklt_b200_%s.so" % variant)


def needs_build(variant=None):
    lib = lib_path(variant)
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    deps = [os.path.join(CSRC, s) for s in _sources()] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, variant=None, extra=None):
    lib = lib_path(variant)
    extra = list(extra or []) + os.environ.get("KLT_NVCC_EXTRA", "").split()
    if not force and not needs_build(variant):
        return lib
    os.makedirs(LIB_DIR, exist_ok=True)
    tag = hashlib.sha1(" ".join(NVCC_FLAGS + extra).encode()).hexdigest()[:10]
    obj_dir = os.path.join(LIB_DIR, "obj", (variant or "default") + "-" + tag)
    os.makedirs(obj_dir, exist_ok=True)
    hdr_t = max(os.path.getmtime(p) for p in HEADERS + [os.path.abspath(__file__)])
    base = [nvcc()] + NVCC_FLAGS + extra + ["-I", os.path.join(ROOT, "include"), "-I", CSRC]
    if verbose:
        base += ["-Xptxas", "-v"]

    def compile_one(src):
        path = os.path.join(CSRC, src)
        obj = os.path.join(obj_dir, src[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(path), hdr_t):
            return obj, 0, ""
        res = subprocess.run(base + ["-c", path, "-o", obj], capture_output=True, text=True)
        return obj, res.returncode, res.stdout + res.stderr

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 2)) as pool:
        results = list(pool.map(compile_one, _sources()))
    for obj, rc, log in results:
        if verbose or rc != 0:
            sys.stderr.write(log)
        if rc != 0:
            raise RuntimeError("nvcc failed compiling for %s" % os.path.basename(obj))
    res = subprocess.run([nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", lib] + [r[0] for r in results],
                         capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking %s" % os.path.basename(lib))
    return lib


if __name__ == "__main__":
    variant, extra = None, []
    if "--variant" in sys.argv:
        variant = sys.argv[sys.argv.index("--variant") + 1]
    if "--extra" in sys.argv:
        extra = sys.argv[sys.argv.index("--extra") + 1].split()
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, variant=variant, extra=extra))
