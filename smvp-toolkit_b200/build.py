"""Build libsmvp_cuda.so (CUDA kernels + C ABI, sm_100a) and the host C side in-tree.

    python smvp-toolkit_b200/build.py [--force]

nvcc cross-compiles without a GPU.  Outputs land in smvp-toolkit_b200/lib/ (git-ignored, but they
travel to the GPU box with the gpurun snapshot).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIB = os.path.join(HERE, "lib")
OBJ = os.path.join(LIB, "obj")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "-DSMVP_BUILDING_LIB"]
CUDA_SO = os.path.join(LIB, "libsmvp_cuda.so")
HOST_SO = os.path.join(LIB, "libsmvp_host.so")
CLI = os.path.join(LIB, "smvp-toolkit-cli")


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("command failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
    return r.stdout + r.stderr


def build_cuda(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers += [os.path.join(REPO, "include", f) for f in os.listdir(os.path.join(REPO, "include"))]
    srcs = sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))
    jobs = []
    objs = []
    for f in srcs:
        src = os.path.join(CSRC, f)
        obj = os.path.join(OBJ, f[:-3] + ".o")
        objs.append(obj)
        if force or _newer(obj, [src] + headers):
            jobs.append([NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj])
    with ThreadPoolExecutor(max_workers=8) as ex:
        outs = list(ex.map(_run, jobs))
    if verbose:
        for o in outs:
            print(o)
    if jobs or force or _newer(CUDA_SO, objs):
        _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", CUDA_SO] + objs)
    return CUDA_SO


def build_host(force=False):
    """The C host side (loader, report writer, CLI) -- plain gcc, links against libsmvp_cuda."""
    if not os.path.isdir(HOST):
        return None
    os.makedirs(LIB, exist_ok=True)
    csrcs = sorted(os.path.join(HOST, f) for f in os.listdir(HOST) if f.endswith(".c"))
    hdrs = [os.path.join(HOST, f) for f in os.listdir(HOST) if f.endswith(".h")]
    hdrs += [os.path.join(REPO, "include", f) for f in os.listdir(os.path.join(REPO, "include"))]
    if not csrcs:
        return None
    lib_srcs = [s for s in csrcs if os.path.basename(s) != "main-cli.c"]
    common = ["gcc", "-O2", "-std=gnu11", "-Wall", "-Wextra", "-D_XOPEN_SOURCE=700", "-I" + os.path.join(REPO, "include"),
              "-I" + HOST]
    if force or _newer(HOST_SO, lib_srcs + hdrs):
        _run(common + ["-fPIC", "-shared", "-o", HOST_SO] + lib_srcs + ["-lm", "-lpthread"])
    main = os.path.join(HOST, "main-cli.c")
    if os.path.exists(main) and (force or _newer(CLI, csrcs + hdrs + [CUDA_SO])):
        _run(common + ["-o", CLI] + csrcs + ["-L" + LIB, "-lsmvp_cuda", "-Wl,-rpath,$ORIGIN", "-lm", "-lpthread"])
    return HOST_SO


def build_all(force=False, verbose=False):
    so = build_cuda(force=force, verbose=verbose)
    build_host(force=force)
    return so


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose="-v" in sys.argv))
