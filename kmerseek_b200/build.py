"""Build libkmerseek_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libkmerseek_b200.so")
SOURCES = ["api.cu", "sketch.cu", "index_build.cu", "dense.cu", "search.cu", "append.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
EXTRA = os.environ.get("KS_NVCC_EXTRA", "").split()  # experiments: -DKS_...=...
FLAGS = EXTRA + ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function", "--expt-relaxed-constexpr"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".hpp"))]
    headers.append(os.path.join(HERE, "..", "include", "kmerseek_b200.h"))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    jobs = []
    for s in SOURCES:
        src, obj = os.path.join(CSRC, s), os.path.join(objdir, s + ".o")
        if force or _stale(obj, [src] + headers):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append(cmd)
    with concurrent.futures.ThreadPoolExecutor(max_workers=4) as ex:
        for cmd, res in zip(jobs, ex.map(lambda c: subprocess.run(c, capture_output=True, text=True), jobs)):
            if verbose or res.returncode:
                sys.stderr.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
            if res.returncode:
                raise RuntimeError("nvcc failed: " + " ".join(cmd))
    objs = [os.path.join(objdir, s + ".o") for s in SOURCES]
    if force or jobs or _stale(OUT, objs):
        cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-lz", "-ldl", "-cudart", "static"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("link failed")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
