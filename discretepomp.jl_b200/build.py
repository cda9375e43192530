"""In-tree build of libdpomp.so for sm_100a with nvcc (no JIT cache, no setuptools): the .so travels with the repo
snapshot to the GPU box.  Translation units are compiled in parallel and linked into discretepomp.jl_b200/lib/."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
SOURCES = ["capi.cu", "pf_kernels.cu", "pf_sim_f32.cu", "pf_sim_f64.cu", "pf_sim_count_f32.cu", "pf_sim_count_f64.cu", "mbp.cu",
           "comm.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr", "-ftz=true",
] + os.environ.get("DPOMP_NVCC_EXTRA", "").split()


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _host_cxx_args() -> list:
    # nvcc needs a g++ it supports; prefer the system one
    for cand in ("/usr/bin/g++",):
        if os.path.exists(cand):
            return ["-ccbin", cand]
    return []


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build_variant(name: str, extra_flags) -> str:
    """Build lib/variants/libdpomp_<name>.so with extra nvcc flags (kernel A/B measurements; select it at run time
    with DPOMP_LIB_PATH).  Not used by the product path."""
    vdir = os.path.join(LIBDIR, "variants")
    odir = os.path.join(vdir, "obj_" + name)
    os.makedirs(odir, exist_ok=True)
    out = os.path.join(vdir, f"libdpomp_{name}.so")
    nvcc, ccbin = _nvcc(), _host_cxx_args()

    def one(src: str) -> str:
        obj = os.path.join(odir, src.replace(".cu", ".o"))
        res = subprocess.run([nvcc, *NVCC_FLAGS, *extra_flags, *ccbin, "-c", os.path.join(CSRC, src), "-o", obj],
                             capture_output=True, text=True)
        with open(obj.replace(".o", ".ptxas.log"), "w") as f:
            f.write(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{res.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(one, SOURCES))
    res = subprocess.run([nvcc, "-shared", *ccbin, "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, *objs, "-lcudart", "-ldl"],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stderr}")
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    out = os.path.join(LIBDIR, "libdpomp.so")
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "dpomp.h")]
    stamp = os.path.join(LIBDIR, "build.stamp")
    digest = _digest(deps)
    if not force and os.path.exists(out) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return out
    nvcc = _nvcc()
    ccbin = _host_cxx_args()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *ccbin, "-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(OBJDIR, src.replace(".cu", ".ptxas.log"))
        with open(log, "w") as f:
            f.write(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            sys.stderr.write(res.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    link = [nvcc, "-shared", *ccbin, "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, *objs, "-lcudart", "-ldl"]
    res = subprocess.run(link, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return out


def build_bounds_variant() -> str:
    """lib/variants/libdpomp_bounds.so: the same library with -DDPOMP_BOUNDS_CHECK (every shared / global index of the
    resample phase, the warp work queue and the MBP windows trapped when out of range).  Used by tests/test_gpu_bounds.py
    as the stand-in for compute-sanitizer; never loaded by the product path."""
    out = os.path.join(LIBDIR, "variants", "libdpomp_bounds.so")
    stamp = out + ".stamp"
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "dpomp.h")]
    digest = _digest(deps)
    if os.path.exists(out) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return out
    build_variant("bounds", ["-DDPOMP_BOUNDS_CHECK"])
    with open(stamp, "w") as f:
        f.write(digest)
    return out


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--variant":
        print(build_variant(sys.argv[2], sys.argv[3:]))
        sys.exit(0)
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
