"""Builds liblto_b200.so (hand-written sm_100a CUDA + the C ABI) in-tree with nvcc.

    python -m lowthrustopt_b200.build [--force] [--verbose]

The shared object lands next to this file so that it travels with a repo snapshot.
There is deliberately no other backend: if nvcc or the sources are missing this raises.
build_experiments() builds the variant library of tools/experiments/ the same way.
"""
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INC = os.path.join(HERE, "..", "include")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "liblto_b200.so")
EXPERIMENTS = os.path.normpath(os.path.join(HERE, "..", "tools", "experiments"))
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
              "-Xptxas", "-v", "-ccbin", "/usr/bin/g++"] + os.environ.get("LTO_NVCC_EXTRA", "").split()   # (development: -D switches)


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: liblto_b200.so cannot be built (there is no non-CUDA backend)")
    return nvcc


def _sources(extra=()):
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu")) + [os.path.abspath(f) for f in extra]


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hs.append(os.path.join(INC, "lto_b200.h"))
    return hs


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_lib(force=False, verbose=False, lib=LIB, obj_dir=OBJ, extra_sources=(), extra_flags=()):
    nvcc = _nvcc()
    os.makedirs(obj_dir, exist_ok=True)
    hdrs = _headers()
    srcs = _sources(extra_sources)
    jobs = []
    for src in srcs:
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc] + ARCH + NVCC_FLAGS + list(extra_flags) + ["-I", INC, "-I", CSRC, "-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".ptxas.log")
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stdout + r.stderr))
        return r.stderr

    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for out in ex.map(compile_one, jobs):
                if verbose:
                    sys.stderr.write(out)
    objs = [os.path.join(obj_dir, os.path.basename(s)[:-3] + ".o") for s in srcs]
    if force or jobs or _stale(lib, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", lib] + objs + ["-ccbin", "/usr/bin/g++"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return lib


def build_experiments(name="k3x", flags=(), force=False, verbose=False):
    """tools/experiments/lib/liblto_<name>.so: the product library PLUS the measured-and-not-adopted layouts of the 12-dim STM kernel
    (tools/experiments/lto_indirect_{hc,wl,hc2}.cu), selected at run time with LTO_K3=hc|wl|hc2 and loaded with LTO_B200_LIB.  The
    parity test of those layouts runs liblto_k3x.so; the product library never contains them."""
    out = os.path.join(EXPERIMENTS, "lib")
    srcs = [os.path.join(EXPERIMENTS, f) for f in ("lto_indirect_hc.cu", "lto_indirect_wl.cu", "lto_indirect_hc2.cu")]
    return build_lib(force, verbose, lib=os.path.join(out, "liblto_%s.so" % name), obj_dir=os.path.join(out, "_build_" + name),
                     extra_sources=srcs, extra_flags=["-DLTO_K3_EXPERIMENTS"] + list(flags))


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
