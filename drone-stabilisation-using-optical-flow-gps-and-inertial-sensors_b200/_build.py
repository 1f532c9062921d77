"""In-tree build of libofb200.so (sm_100a only). Used by __graft_entry__.build() and by hand:

    python -m ofb200._build            (through the ofb200 alias at the repo root)

Objects go to csrc/build/, the library next to this file so that it travels with the source tree.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libofb200.so")
SOURCES = ["api.cu", "pyramid.cu", "features.cu", "pyrlk.cu", "velocity.cu", "montecarlo.cu", "pairs.cu", "tracker.cu", "camera.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, debug=False):
    """debug=True: libofb200_dbg.so with -DOFB_DEBUG_BOUNDS=1 (device-side index assertions, see csrc/common.cuh);
    select it with OFB200_LIB=<path> when running the tests."""
    bdir = os.path.join(CSRC, "build_dbg" if debug else "build")
    os.makedirs(bdir, exist_ok=True)
    out = OUT.replace("libofb200.so", "libofb200_dbg.so") if debug else OUT
    flags = FLAGS + (["-DOFB_DEBUG_BOUNDS=1"] if debug else [])
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "ofb200.h"))
    jobs = []
    objs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(bdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + headers):
            cmd = [NVCC] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        return cmd, r

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for cmd, r in ex.map(run, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for " + cmd[-3])
    if force or jobs or _stale(out, objs):
        cmd = [NVCC, "-shared", "-o", out] + objs + ["-cudart", "static", "-Xlinker", "--exclude-libs,ALL"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug="--debug" in sys.argv))
