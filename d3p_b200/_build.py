"""In-tree build of libd3p_b200.so (sm_100a only) with nvcc.

``python -m d3p_b200._build`` or ``__graft_entry__.build()``.  Objects are compiled in parallel
and cached by source mtime; the shared library lands in ``d3p_b200/_lib/`` so that it travels
with the source tree (it is git-ignored, not gpurun-ignored).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "_lib")
LIBNAME = "libd3p_b200.so"
SOURCES = ["rng.cu", "samplers.cu", "clip.cu", "finalize.cu", "meanfield_step.cu", "meanfield_step_vec.cu",
           "tc_gemm.cu", "vae.cu", "gmm_step.cu", "evaluate.cu", "epoch.cu", "comm.cu", "jrandom.cu", "gmm_dist.cu",
           "autodiag.cu"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def lib_path():
    return os.path.join(LIBDIR, LIBNAME)


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _deps_mtime():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "d3p_b200.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def _defines():
    """Development builds only (e.g. D3P_NVCC_DEFINES=D3P_GEMM_TRACE python -m d3p_b200._build): extra -D flags; the
    object cache is invalidated whenever the set changes, so the next plain build is the product library again."""
    return [d for d in os.environ.get("D3P_NVCC_DEFINES", "").split(",") if d]


def _compile(src, verbose):
    obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
    srcp = os.path.join(CSRC, src)
    if os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(srcp), _deps_mtime()):
        return obj, ""
    cmd = ([_nvcc()] + NVCC_FLAGS + ["-D" + d for d in _defines()] + (["-Xptxas", "-v"] if verbose else [])
           + ["-c", srcp, "-o", obj])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    return obj, r.stderr


def build(verbose=False, force=False):
    os.makedirs(LIBDIR, exist_ok=True)
    flags_file = os.path.join(LIBDIR, ".defines")
    want = ",".join(_defines())
    have = open(flags_file).read() if os.path.exists(flags_file) else ""
    if want != have:
        force = True
        with open(flags_file, "w") as f:
            f.write(want)
    if force:
        for f in os.listdir(LIBDIR):
            if f.endswith((".o", ".so")):
                os.remove(os.path.join(LIBDIR, f))
    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        results = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    objs = [o for o, _ in results]
    log = "".join(l for _, l in results)
    out = lib_path()
    if (not os.path.exists(out)) or any(os.path.getmtime(o) > os.path.getmtime(out) for o in objs):
        cmd = [_nvcc(), "-shared", "-o", out] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print(log)
    return out


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
