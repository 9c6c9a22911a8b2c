"""Build libwmf_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension:
the C-ABI library has no torch types in it). `python -m recmodel_b200.build` or
`__graft_entry__.build()`."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libwmf_b200.so")
SOURCES = ["api.cu", "csr.cu", "ease.cu", "eval_topn.cu", "knn.cu", "exchange.cu", "gram.cu", "half_step_api.cu", "half_step_simt.cu", "half_step_tc.cu", "half_step_tc256.cu", "half_step_dual.cu", "whiten.cu", "loss.cu", "score.cu", "score_tc.cu",
           "topn_metrics.cu", "unweighted.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return "nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, variant=None, extra_flags=()):
    """``variant``: suffix of a development build kept beside the product library (objects and .so get the
    suffix), e.g. build(variant="wd", extra_flags=["-DWMF_WATCHDOG"])."""
    headers = [os.path.join(CSRC, h) for h in os.listdir(CSRC) if h.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "wmf_b200.h"))
    flags = list(NVCC_FLAGS)
    flags += os.environ.get("WMF_NVCC_EXTRA", "").split()   # e.g. -DWMF_WATCHDOG, -DWMF_TC_PROFILE_BUILD (development)
    flags += list(extra_flags)
    sfx = f"_{variant}" if variant else ""
    lib_path = LIB.replace(".so", sfx + ".so")
    if verbose:
        flags += ["-Xptxas", "-v"]
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src.replace(".cu", sfx + ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            jobs.append([_nvcc(), *flags, "-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if verbose and (r.stdout or r.stderr):
            print(r.stdout + r.stderr)

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            list(ex.map(run, jobs))
    if jobs or force or _stale(lib_path, objs):
        run([_nvcc(), "-shared", "-o", lib_path, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static",
             "-lcuda"])
    return lib_path


if __name__ == "__main__":
    if "--watchdog" in sys.argv:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, variant="wd", extra_flags=["-DWMF_WATCHDOG"]))
    elif "--profile" in sys.argv:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, variant="prof", extra_flags=["-DWMF_TC_PROFILE_BUILD"]))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
