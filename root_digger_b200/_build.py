"""Build recipes (nvcc / g++) for the native libraries, all in-tree.

  lib/librdk_b200.so   CUDA kernels + C ABI (include/rdk.h), sm_100a only
  lib/librd_host.so    C++ host: traversal scheduler + model_t mirror, linked
                       against librdk_b200.so
  lib/liblbfgsb.so     L-BFGS-B 3.0 (setulb), from lbfgsb/lbfgsb.c

The oracle (test infrastructure) has its own recipes, oracle/Makefile and
oracle/oracle_build.py; nothing in the product builds, links or loads it.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "root_digger_b200"
LIBDIR = PKG / "lib"
CSRC = PKG / "csrc"
HOST = PKG / "host"
INCLUDE = ROOT / "include"
LBFGSB = PKG / "lbfgsb"

NVCC_ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _cxx() -> str:
    return "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def _cc() -> str:
    return "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"


def _nvcc() -> str:
    for cand in ("/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA engine cannot be built (there is no CPU fallback)")


def _newer(target: Path, sources) -> bool:
    if not target.exists():
        return False
    t = target.stat().st_mtime
    return all(Path(s).stat().st_mtime <= t for s in sources)


def _run(cmd, **kw):
    res = subprocess.run([str(c) for c in cmd], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, **kw)
    if res.returncode != 0:
        raise RuntimeError("build failed: %s\n%s" % (" ".join(str(c) for c in cmd), res.stdout))
    return res.stdout


PROGRAM_KS = (1, 2, 4, 8, 16, 32)  # rate-category counts the program kernel is instantiated for


def build_engine(force: bool = False, verbose: bool = False) -> Path:
    """nvcc -> lib/librdk_b200.so (sm_100a, -lineinfo).  The ABI, the host math and one
    translation unit per rate-category count (rdk_program_inst.cu, -DRDK_INST_K=K) are compiled
    in parallel and linked into one shared library."""
    from concurrent.futures import ThreadPoolExecutor

    LIBDIR.mkdir(exist_ok=True)
    out = LIBDIR / "librdk_b200.so"
    srcs = [CSRC / "rdk_abi.cu", CSRC / "rdk_host_math.cpp", CSRC / "rdk_lower_debug.cpp", CSRC / "rdk_program_inst.cu",
            CSRC / "rdk_support.cu"]
    deps = srcs + [CSRC / "rdk_kernels.cuh", CSRC / "rdk_lower.hpp", CSRC / "rdk_support.cuh", INCLUDE / "rdk.h"]
    if not force and _newer(out, deps):
        return out
    objdir = LIBDIR / "obj_librdk_b200"
    objdir.mkdir(exist_ok=True)
    base = [_nvcc(), *NVCC_ARCH, "-lineinfo", "-O3", "-std=c++17", "--fmad=false", "-ccbin", _cxx(),
            "-Xcompiler", "-fPIC,-ffp-contract=off,-Wall", "-I", INCLUDE]
    if verbose:
        base.insert(1, "-Xptxas=-v")
    jobs = [(base + ["-c", CSRC / "rdk_abi.cu", "-o", objdir / "rdk_abi.o"]),
            (base + ["-c", CSRC / "rdk_host_math.cpp", "-o", objdir / "rdk_host_math.o"]),
            (base + ["-c", CSRC / "rdk_lower_debug.cpp", "-o", objdir / "rdk_lower_debug.o"]),
            (base + ["-c", CSRC / "rdk_support.cu", "-o", objdir / "rdk_support.o"])]
    for k in PROGRAM_KS:
        jobs.append(base + ["-DRDK_INST_K=%d" % k, "-c", CSRC / "rdk_program_inst.cu", "-o", objdir / ("rdk_program_k%d.o" % k)])
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
        logs = list(pool.map(_run, jobs))
    objs = [j[-1] for j in jobs]
    logs.append(_run([_nvcc(), *NVCC_ARCH, "-shared", "-o", out, *objs, "-ldl"]))
    if verbose:
        print("\n".join(logs))
    return out


def lbfgsb_source_dir() -> Path:
    """where the L-BFGS-B 3.0 C sources are: $RDK_LBFGSB_SRC (e.g. RootDigger's own lib/lbfgsb, to run
    against the C translation it vendors), else this package's lbfgsb/"""
    cand = os.environ.get("RDK_LBFGSB_SRC")
    if cand and Path(cand).is_dir() and list(Path(cand).glob("*.c")):
        return Path(cand)
    return LBFGSB


def build_lbfgsb(force: bool = False) -> Path:
    """lib/liblbfgsb.so (setulb, the optimiser model_t::bfgs_params drives, reference
    src/model.cpp:1430-1522), built from lbfgsb_source_dir()."""
    LIBDIR.mkdir(exist_ok=True)
    out = LIBDIR / "liblbfgsb.so"
    src_dir = lbfgsb_source_dir()
    srcs = sorted(src_dir.glob("*.c"))
    if not force and _newer(out, srcs):
        return out
    _run([_cc(), "-O2", "-fPIC", "-shared", "-w", "-ffp-contract=off", "-I", src_dir, "-o", out, *srcs, "-lm"])
    return out


def host_sources():
    return [HOST / "tree.cpp", HOST / "tree_capi.cpp", HOST / "msa.cpp", HOST / "partition_file.cpp", HOST / "checkpoint.cpp",
            HOST / "checkpoint_capi.cpp", HOST / "model.cpp",
            HOST / "lbfgsb_driver.cpp", HOST / "model_capi.cpp", HOST / "optim_capi.cpp"]


def build_host(force: bool = False) -> Path:
    """g++ -> lib/librd_host.so (scheduler + model_t mirror on the CUDA engine)."""
    engine = build_engine()
    build_lbfgsb()
    out = LIBDIR / "librd_host.so"
    srcs = [s for s in host_sources() if s.exists()]
    deps = srcs + list(HOST.glob("*.hpp")) + [INCLUDE / "rdk.h", engine]
    if not force and _newer(out, deps):
        return out
    _run([_cxx(), "-std=c++17", "-O2", "-fPIC", "-fopenmp", "-Wall", "-ffp-contract=off", "-I", INCLUDE, "-shared",
          "-o", out, *srcs, "-L", LIBDIR, "-lrdk_b200", "-ldl", "-Wl,-rpath,$ORIGIN", "-Wl,-Bsymbolic"])
    return out


def build_all(verbose: bool = False):
    """the product: engine + L-BFGS-B + host library (the oracle has its own recipe, oracle/oracle_build.py)"""
    build_engine(verbose=verbose)
    build_lbfgsb()
    build_host()
