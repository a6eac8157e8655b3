"""TEST INFRASTRUCTURE -- build recipes of the CPU oracle and of the host sources compiled
against it.  Only tests/, __graft_entry__ (build / smoke) and bench.py's CPU-baseline leg use
this; the product package (root_digger_b200/) never imports it.

  oracle/librd_oracle.so             oracle/Makefile
  oracle/alpha_oracle.py             (pure Python, nothing to build) the reference's search for the root
                                     position on a branch, restated over any function on [0, 1]
  oracle/bfgs_oracle.py              (pure Python) the reference's L-BFGS-B driver bfgs_params, restated
                                     around the same setulb (lib/liblbfgsb.so) over any objective
  tests/_build/librd_host_oracle.so  root_digger_b200/host/*.cpp compiled against the oracle
                                     through tests/oracle_shim/rdk.h (-DRD_BACKEND_ORACLE)
  oracle/_ref/librd_reference_on_{oracle,engine}.so
                                     RootDigger's own src/*.cpp, compiled unmodified from a RootDigger
                                     checkout ($ROOTDIGGER_SRC) against root_digger_b200/compat/corax/corax.h
                                     (built only where such a checkout is given)
"""
from __future__ import annotations

import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from root_digger_b200._build import HOST, _cxx, _newer, _run, build_lbfgsb, host_sources  # noqa: E402

ORACLE = ROOT / "oracle"


def build_oracle(force: bool = False) -> Path:
    """TEST INFRASTRUCTURE: oracle/librd_oracle.so via oracle/Makefile."""
    out = ORACLE / "librd_oracle.so"
    deps = [ORACLE / "rd_oracle.c", ORACLE / "rd_oracle.h", ORACLE / "Makefile"]
    if not force and _newer(out, deps):
        return out
    _run(["make", "-C", ORACLE, "-B" if force else "-s"])
    return out


def build_host_on_oracle(force: bool = False) -> Path:
    """TEST INFRASTRUCTURE: the same host sources compiled against the oracle
    through tests/oracle_shim/rdk.h -> tests/_build/librd_host_oracle.so."""
    oracle = build_oracle()
    build_lbfgsb()
    outdir = ROOT / "tests" / "_build"
    outdir.mkdir(exist_ok=True)
    out = outdir / "librd_host_oracle.so"
    srcs = [s for s in host_sources() if s.exists()]
    shim = ROOT / "tests" / "oracle_shim"
    deps = srcs + list(HOST.glob("*.hpp")) + [shim / "rdk.h", oracle]
    if not force and _newer(out, deps):
        return out
    _run([_cxx(), "-std=c++17", "-O2", "-fPIC", "-fopenmp", "-Wall", "-ffp-contract=off", "-DRD_BACKEND_ORACLE",
          "-I", shim, "-I", ORACLE, "-shared", "-o", out, *srcs, "-L", ORACLE, "-lrd_oracle", "-ldl",
          "-Wl,-rpath," + str(ORACLE), "-Wl,-Bsymbolic"])
    return out


REFERENCE = Path(os.environ["ROOTDIGGER_SRC"]) if os.environ.get("ROOTDIGGER_SRC") else None
REF_SOURCES = ("model.cpp", "tree.cpp", "msa.cpp", "checkpoint.cpp", "util.cpp")


def build_reference_sources(backend: str = "oracle", force: bool = False):
    """TEST INFRASTRUCTURE: RootDigger's OWN src/{model,tree,msa,checkpoint,util}.cpp, unmodified and
    compiled from where they lie in the RootDigger checkout $ROOTDIGGER_SRC, against root_digger_b200/compat/corax/corax.h
    -- i.e. against the engine's C ABI (backend "engine": include/rdk.h + librdk_b200.so) or against
    the oracle behind the same ABI (backend "oracle": tests/oracle_shim/rdk.h + librd_oracle.so) --
    plus tests/ref_build/ref_capi.cpp (ctypes wrappers) -> oracle/_ref/librd_reference_on_<backend>.so
    (git-ignored: no reference source is copied).  Returns None when no checkout is given and no
    library was built earlier."""
    from root_digger_b200._build import INCLUDE, LIBDIR, PKG
    outdir = ORACLE / "_ref"
    out = outdir / ("librd_reference_on_%s.so" % backend)
    if REFERENCE is None or not (REFERENCE / "src" / "model.cpp").exists():
        return out if out.exists() else None
    ref_src = REFERENCE / "src"
    outdir.mkdir(exist_ok=True)
    lbfgsb = build_lbfgsb()
    compat = PKG / "compat"
    ours = [compat / "corax_compat.cpp", HOST / "tree.cpp"]
    theirs = [ref_src / f for f in REF_SOURCES] + [ROOT / "tests" / "ref_build" / "ref_capi.cpp"]
    if backend == "oracle":
        abi_inc = ["-I", ROOT / "tests" / "oracle_shim", "-I", ORACLE]
        link = ["-L", ORACLE, "-lrd_oracle", "-Wl,-rpath," + str(ORACLE)]
        deps_lib = build_oracle()
    else:
        abi_inc = ["-I", INCLUDE]
        link = ["-L", LIBDIR, "-lrdk_b200", "-Wl,-rpath," + str(LIBDIR)]
        deps_lib = LIBDIR / "librdk_b200.so"
    deps = ours + theirs + [compat / "corax" / "corax.h", deps_lib, lbfgsb] + list(HOST.glob("tree.hpp"))
    if not force and _newer(out, deps):
        return out
    objdir = outdir / ("obj_reference_on_%s" % backend)
    objdir.mkdir(exist_ok=True)
    base = [_cxx(), "-std=c++17", "-O2", "-fPIC", "-fopenmp", "-w", "-ffp-contract=off", "-I", compat, *abi_inc]
    objs = []
    # the engine host's utree module next to RootDigger's own rooted_tree_t: its classes are renamed
    for src in ours:
        obj = objdir / (src.stem + ".o")
        _run(base + ["-Drooted_tree_t=rdh_compat_rooted_tree_t", "-Droot_location_t=rdh_compat_root_location_t",
                     "-I", HOST, "-c", src, "-o", obj])
        objs.append(obj)
    for src in theirs:
        obj = objdir / ("ref_" + src.stem + ".o")
        _run(base + ["-I", ref_src, "-I", REFERENCE / "lib" / "lbfgsb", "-c", src, "-o", obj])
        objs.append(obj)
    _run([_cxx(), "-shared", "-fopenmp", "-o", out, *objs, *link, "-L", LIBDIR, "-llbfgsb",
          "-Wl,-rpath," + str(LIBDIR), "-ldl", "-Wl,-Bsymbolic"])
    return out


def build_all():
    build_oracle()
    build_host_on_oracle()
    build_reference_sources("oracle")
    build_reference_sources("engine")
