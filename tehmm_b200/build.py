"""Build libtehmm_b200.so in-tree with nvcc for sm_100a (no GPU needed).

    python -m tehmm_b200.build          # or tehmm_b200.build.build()

Each translation unit is compiled to an object in parallel and linked into
tehmm_b200/libtehmm_b200.so.  strict.cu is compiled with -fmad=false so the
float64 operation order of the reference is kept (no contraction).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libtehmm_b200.so")
UNITS = ["api", "strict", "emission", "forward", "backward", "viterbi", "stats", "tile", "host", "umma", "fallback", "tracks", "ratios", "supervised", "window"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
          "-Xptxas", "-v"]
EXTRA = {"strict": ["-fmad=false"], "supervised": ["-fmad=false"]}


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "tehmm_b200.h"))
    nvcc = _nvcc()

    def compile_one(unit):
        src = os.path.join(CSRC, unit + ".cu")
        obj = os.path.join(OBJ, unit + ".o")
        if not force and not _stale(obj, [src] + headers):
            return unit, ""
        cmd = [nvcc] + ARCH + COMMON + EXTRA.get(unit, []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (unit, r.stdout, r.stderr))
        with open(os.path.join(OBJ, unit + ".ptxas.log"), "w") as f:
            f.write(r.stderr)
        return unit, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, len(UNITS))) as ex:
        logs = list(ex.map(compile_one, UNITS))
    objs = [os.path.join(OBJ, u + ".o") for u in UNITS]
    if force or _stale(LIB, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    if verbose:
        for unit, log in logs:
            if log:
                print("==== %s\n%s" % (unit, log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
