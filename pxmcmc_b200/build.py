"""In-tree nvcc build of libpxmcmc_b200.so for sm_100a (no JIT cache: the .so
travels with the repository snapshot to the GPU box)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.environ.get("PXM_LIB_OUT", os.path.join(HERE, "libpxmcmc_b200.so"))
SOURCES = ["pxm_plan.cu", "pxm_tables.cu", "pxm_legendre.cu", "pxm_fft.cu", "pxm_healpix.cu", "pxm_elem.cu", "pxm_paths.cu", "pxm_stats.cu",
           "pxm_rank.cu", "pxm_credible.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xptxas", "-v"] + os.environ.get("PXM_EXTRA_NVCC_FLAGS", "").split()
# the elementwise file must not contract a*b+c into FMAs: the reference's numpy
# expressions round every product (bit-level agreement of the prox support)
# (the running moments of pxm_stats.cu likewise: the same Welford updates on every path, whatever the compiler fuses)
PER_FILE = {"pxm_elem.cu": ["-fmad=false"], "pxm_stats.cu": ["-fmad=false"]}


def _stale(obj, src):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(HERE, "..", "include", "pxmcmc_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    objs = []
    logs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(bdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, src):
            cmd = [nvcc, *ARCH, *COMMON, *PER_FILE.get(s, []), "-c", src, "-o", obj]
            r = subprocess.run(cmd, capture_output=True, text=True)
            logs.append(f"$ {' '.join(cmd)}\n{r.stdout}{r.stderr}")
            if r.returncode != 0:
                sys.stderr.write(logs[-1])
                raise RuntimeError(f"nvcc failed on {s}")
    if force or not os.path.exists(OUT) or any(os.path.getmtime(o) > os.path.getmtime(OUT) for o in objs):
        cmd = [nvcc, *ARCH, "-shared", "-o", OUT, *objs, "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        logs.append(f"$ {' '.join(cmd)}\n{r.stdout}{r.stderr}")
        if r.returncode != 0:
            sys.stderr.write(logs[-1])
            raise RuntimeError("link failed")
    if logs:
        with open(os.path.join(bdir, "build.log"), "w") as f:
            f.write("\n".join(logs))
        if verbose:
            print("\n".join(logs))
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
