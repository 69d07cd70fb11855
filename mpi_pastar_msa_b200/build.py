"""Build libpastar_gpu.so (CUDA kernels + C ABI) and the pastar CLI, in-tree, for sm_100a only.

    python -m mpi_pastar_msa_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The outputs are git-ignored but travel to the GPU box.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
PHASE = bool(os.environ.get("PG_PHASE_TIMING"))  # instrumented variant: per-phase cycle counters in the expand kernel
# experiment variants: PG_VARIANT=name PG_EXTRA_NVCC="-DX=1 ..." builds lib/libpastar_gpu_<name>.so (load it with PASTAR_GPU_LIB)
VARIANT = "phase" if PHASE else os.environ.get("PG_VARIANT", "")
OBJ = os.path.join(HERE, "build_" + VARIANT if VARIANT else "build")
LIB = os.path.join(HERE, "lib", "libpastar_gpu_%s.so" % VARIANT if VARIANT else "libpastar_gpu.so")
BIN = os.path.join(HERE, "bin", "pastar")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CXX = os.environ.get("CXX", "g++")

CU_SOURCES = ["pg_api.cu", "pg_pairdp.cu", "pg_expand.cu", "pg_primer.cu", "pg_search.cu", "pg_drivers.cu", "pg_layered.cu"]
HOST_SOURCES = ["host/pg_host_weights.cpp"]
CLI_SOURCES = ["host/pastar_main.cpp"]
NVCC_FLAGS = (["-DPG_PHASE_TIMING"] if PHASE else []) + os.environ.get("PG_EXTRA_NVCC", "").split() + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
              "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC]
# -ffp-contract=off: the host weight routine must not fuse multiply-adds (float-order exact vs the reference)
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC]


def _newer(src_list, out):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(s) > t for s in src_list)


def _headers():
    hs = [os.path.join(ROOT, "include", "pastar_gpu.h")]
    for d, _, fs in os.walk(CSRC):
        hs += [os.path.join(d, f) for f in fs if f.endswith((".cuh", ".h", ".hpp"))]
    return hs


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0:
        sys.stderr.write(r.stdout.decode())
        raise RuntimeError("build step failed: " + " ".join(cmd[:3]) + " ...")
    if verbose and r.stdout:
        print(r.stdout.decode())


def build(force=False, verbose=False, ptxas_info=False):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    os.makedirs(os.path.dirname(BIN), exist_ok=True)
    hdrs = _headers()
    jobs, objs = [], []
    for s in CU_SOURCES:
        src = os.path.join(CSRC, s)
        o = os.path.join(OBJ, s.replace("/", "_") + ".o")
        objs.append(o)
        if force or _newer([src] + hdrs, o):
            jobs.append([NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if ptxas_info else []) + ["-c", src, "-o", o])
    for s in HOST_SOURCES:
        src = os.path.join(CSRC, s)
        o = os.path.join(OBJ, s.replace("/", "_") + ".o")
        objs.append(o)
        if force or _newer([src] + hdrs, o):
            jobs.append([CXX] + CXX_FLAGS + ["-c", src, "-o", o])
    with ThreadPoolExecutor(max_workers=max(1, min(8, len(jobs)))) as ex:
        list(ex.map(lambda c: _run(c, verbose or ptxas_info), jobs))
    if jobs or force or not os.path.exists(LIB):
        _run([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-lpthread"], verbose)
    cli = [os.path.join(CSRC, s) for s in CLI_SOURCES if os.path.exists(os.path.join(CSRC, s))]
    if cli and not VARIANT and (force or _newer(cli + hdrs + [LIB], BIN)):
        _run([CXX] + CXX_FLAGS + cli + ["-o", BIN, "-L" + os.path.dirname(LIB), "-lpastar_gpu", "-Wl,-rpath,$ORIGIN/../lib", "-pthread"],
             verbose)
    # the C++ boundary test program (tests/cpp/boundary_test.cpp): binds the host mirror's Node / Coord / HeuristicHPair
    tsrc = os.path.join(ROOT, "tests", "cpp", "boundary_test.cpp")
    tbin = os.path.join(HERE, "bin", "boundary_test")
    if os.path.exists(tsrc) and not VARIANT and (force or _newer([tsrc] + hdrs + [LIB], tbin)):
        _run([CXX] + CXX_FLAGS + [tsrc, "-o", tbin, "-L" + os.path.dirname(LIB), "-lpastar_gpu", "-Wl,-rpath,$ORIGIN/../lib", "-pthread"], verbose)
    # CPU-only check program of the host mirror (FASTA reader, similarity / alignment printer): the CLI's translation unit
    # with its main renamed, plus tests/cpp/host_cpu_test.cpp
    hsrc = os.path.join(ROOT, "tests", "cpp", "host_cpu_test.cpp")
    hbin = os.path.join(HERE, "bin", "host_cpu_test")
    if os.path.exists(hsrc) and cli and not VARIANT and (force or _newer([hsrc] + cli + hdrs + [LIB], hbin)):
        cobj = os.path.join(OBJ, "pastar_main_nomain.o")
        _run([CXX] + CXX_FLAGS + ["-Dmain=pastar_cli_main", "-c", cli[0], "-o", cobj], verbose)
        _run([CXX] + CXX_FLAGS + [hsrc, cobj, "-o", hbin, "-L" + os.path.dirname(LIB), "-lpastar_gpu", "-Wl,-rpath,$ORIGIN/../lib", "-pthread"], verbose)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, ptxas_info="--ptxas" in sys.argv)
    print(LIB)
