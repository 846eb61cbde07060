"""Build the in-tree native artefacts with nvcc for sm_100a (no torch JIT cache, so the .so travels with the tree).

  is3d_b200/libis3d_b200.so   CUDA kernels + C ABI + C++ host layer
  is3d_b200/is3d_b200_run     drop-in executable (the RuniS3D.cpp equivalent for operation = 1)

`python -m is3d_b200.build [--force] [--verbose]`
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libis3d_b200.so")
EXE = os.path.join(HERE, "is3d_b200_run")
OBJ = os.path.join(HERE, "build")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math"]

# (source, extra flags).  cf_prepare.cu keeps separate multiply/add so the per-cell set-up rounds like the reference.
SOURCES = [
    ("cf_kernels.cu", []),
    ("cf_factored.cu", []),
    ("cf_prepare.cu", ["-fmad=false"]),
    ("cf_decays.cu", ["-fmad=false"]),
    ("cf_strict.cu", ["-fmad=false"]),
    ("cf_shift.cu", []),
    ("cf_polzn.cu", []),
    ("cf_polzn_xi.cu", []),
    ("cf_polzn_she.cu", []),
    ("cf_spin_density.cu", []),
    ("cf_hbt.cu", []),
    ("cf_hbtq.cu", []),
    ("cf_api.cu", []),
    ("host_math.cpp", []),
    ("host_io.cpp", []),
    ("host_run.cpp", []),
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "is3d_b200.h"))
    objs = []
    procs = []
    for src, extra in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(OBJ, src.rsplit(".", 1)[0] + ".o")
        objs.append(obj)
        if force or _newer(obj, [path] + headers):
            cmd = [nvcc] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
            if verbose:
                print(" ".join(cmd), flush=True)
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed for %s:\n%s\n" % (src, out))
        elif verbose and out:
            print(out)
    if failed:
        raise RuntimeError("is3d_b200 native build failed")
    if force or procs or _newer(LIB, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart"]
        subprocess.check_call(cmd)
    main_src = os.path.join(CSRC, "main.cpp")
    if os.path.exists(main_src) and (force or _newer(EXE, [main_src, LIB])):
        cmd = [nvcc, "-O2", "-std=c++17", main_src, "-o", EXE, "-L" + HERE, "-lis3d_b200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print("built", LIB)
