"""Build csrc/libgalerkin_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Each .cu is compiled to an object under csrc/build/ (in parallel, only when stale) and the objects are linked
into the shared library; a header change recompiles everything."""
import glob
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
OUT = os.environ.get("GB200_LIB", os.path.join(CSRC, "libgalerkin_b200.so"))
OBJ_DIR = os.path.join(CSRC, "build")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _headers():
    return glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "..", "..", "include", "*.h"))


def is_stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in sources() + _headers())


def build(force=False, verbose=False):
    if not force and not is_stale():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    extra = os.environ.get("GB200_NVCC_EXTRA", "").split()      # extra nvcc flags for experiments: e.g. -Xptxas -warn-spills
    os.makedirs(OBJ_DIR, exist_ok=True)
    tag = os.path.join(OBJ_DIR, ".flags")
    flags_now = " ".join(NVCC_FLAGS + extra)
    if not os.path.exists(tag) or open(tag).read() != flags_now:
        force = True
    hdr_time = max([os.path.getmtime(h) for h in _headers()] + [0.0])
    jobs = []
    for src in sources():
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_time):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        return src, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as pool:
        for src, res in pool.map(compile_one, jobs):
            if res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
                raise RuntimeError(f"nvcc failed compiling {os.path.basename(src)}")
            if verbose:
                print(res.stderr)
    objs = [os.path.join(OBJ_DIR, os.path.basename(s)[:-3] + ".o") for s in sources()]
    res = subprocess.run([nvcc, "-shared", "-o", OUT] + objs, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking libgalerkin_b200.so")
    with open(tag, "w") as f:
        f.write(flags_now)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
