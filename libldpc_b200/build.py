"""Builds libldpc_b200/libldpc.so (C ABI + CUDA kernels, sm_100a) and the ldpcsim CLI with nvcc.

In-tree, explicit nvcc invocation (no JIT cache): the built files travel with the repo snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libldpc.so")
CLI = os.path.join(HERE, "ldpcsim")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function,-fvisibility=hidden"]
TILE_SOURCES = ["tile_%s_%s_l%d.cu" % (a, t, l) for a in ("bp", "ms") for t in ("f64", "f32") for l in (1, 2, 4)]  # slowest first
SOURCES = TILE_SOURCES + ["layered.cu", "engine.cu", "code.cpp", "sim_driver.cpp", "shim.cpp"]
HEADERS = ["exports.map", "engine.hpp", "code.hpp", "kernels.cuh", "tile4.cuh", "tile_launch.cuh", "bec_kernel.cuh", "bec_slice.cuh", "layered.cuh", "report.cuh", "../../include/ldpc_b200.h"]
OBJDIR = os.path.join(HERE, "build")
if os.environ.get("B200_PHASE_TIMING"):  # debug: per-warp phase cycle counts printed by CTA 0
    COMMON = COMMON + ["-DB200_PHASE_TIMING=1"]
if os.environ.get("B200_TILE_MAX_THREADS"):  # tuning experiments only; the default lives in csrc/tile4.cuh
    COMMON = COMMON + ["-DB200_TILE_MAX_THREADS=" + os.environ["B200_TILE_MAX_THREADS"]]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    global LIB, OBJDIR, COMMON
    if os.environ.get("B200_VARIANT"):  # experiment builds: B200_VARIANT=name B200_DEFS="-DX=1 ..." -> libldpc_<name>.so (A/B runs via LDPC_B200_LIB)
        LIB = os.path.join(HERE, "libldpc_%s.so" % os.environ["B200_VARIANT"])
        OBJDIR = os.path.join("/tmp", "b200_build_%s" % os.environ["B200_VARIANT"])  # outside the tree: the gpurun snapshot stays small
        COMMON = COMMON + os.environ.get("B200_DEFS", "").split()
    if os.environ.get("B200_PHASE_TIMING"):  # the debug build lives beside the product library (LDPC_B200_LIB selects it at load time)
        LIB = os.path.join(HERE, "libldpc_pt.so")
        OBJDIR = os.path.join("/tmp", "b200_build_pt")
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    if force or _stale(LIB, deps):
        from concurrent.futures import ThreadPoolExecutor
        os.makedirs(OBJDIR, exist_ok=True)
        hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]

        def compile_one(src):
            obj = os.path.join(OBJDIR, os.path.basename(src) + ".o")
            if force or _stale(obj, [src] + hdrs):
                cmd = [NVCC] + ARCH + COMMON + ["-c", "-o", obj, src]
                if verbose:
                    cmd += ["-Xptxas", "-v"]
                r = subprocess.run(cmd, capture_output=True, text=True)
                if verbose or r.returncode != 0:
                    sys.stderr.write(r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError("nvcc failed for " + src)
            return obj

        with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
            objs = list(ex.map(compile_one, srcs))
        # exported: exactly the functions include/ldpc_b200.h declares (LDPC_B200_API); the static CUDA runtime stays internal
        subprocess.run([NVCC] + ARCH + ["-shared", "-cudart", "static", "-ccbin", "/usr/bin/g++", "-Xlinker", "--exclude-libs,ALL", "-Xlinker", "--version-script=" + os.path.join(CSRC, "exports.map"), "-o", LIB] + objs, check=True)
    cli_src = os.path.join(CSRC, "cli_main.cpp")
    if not os.environ.get("B200_PHASE_TIMING") and not os.environ.get("B200_VARIANT") and (force or _stale(CLI, [cli_src, LIB])):
        cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-pthread", "-o", CLI, cli_src, LIB, "-Wl,-rpath,$ORIGIN"]  # a plain C-ABI client
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
