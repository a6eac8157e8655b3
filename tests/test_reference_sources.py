"""The drop-in boundary proven with the reference's OWN callers.

RootDigger's src/model.cpp, src/tree.cpp, src/msa.cpp, src/checkpoint.cpp and src/util.cpp are
compiled UNCHANGED -- from where they lie in a RootDigger checkout ($ROOTDIGGER_SRC), never copied --
against root_digger_b200/compat/corax/corax.h, the header that serves the coraxlib calls they make
(src/model.cpp:159-168 ... 466, src/tree.cpp:12-620, src/msa.cpp:18-88) from the engine's C ABI
(oracle/oracle_build.py build_reference_sources).  Through tests/ref_build/ref_capi.cpp they run the
call sequence of src/main.cpp:513-640 on the bundled fixtures; the engine host's model_t mirror
(root_digger_b200/host) must return the same bits: chosen root branch, root position, final
log-likelihood, every per-branch likelihood, LWR ranking.

Without a checkout (and without a library built from one earlier) the reference's side is a record of
what those sources returned on the same calls, tests/golden/reference_sources_v1.json, written by
tests/golden/make_reference_golden.py from such a build; with none of the three the tests skip.  Which
one a run compared against is reported as a warning.

Here (no GPU) both sides run on the oracle behind the same ABI; tests/test_gpu_model.py repeats the
search on the CUDA engine."""
import ctypes as C
import json
import os
import tempfile
import warnings
from pathlib import Path

import numpy as np
import pytest

import fixtures
import oracle_build
import oracle_capi
from root_digger_b200 import capi

_dp = C.POINTER(C.c_double)
_up = C.POINTER(C.c_uint)


# the calls compared (fixture, rate categories, seed[, search strategy]); the record holds these
SEARCHES = [("10.fasta", 1, 7, 1), ("10.fasta", 2, 7, 0), ("10.fasta", 4, 7, 2), ("10.fasta", 3, 7, 0)]
EVERY_ROOT = [("101.phy", 4, 11), ("10.fasta", 2, 5)]
EXHAUSTIVE = [("10.fasta", 4, 3)]
GOLDEN = Path(__file__).resolve().parent / "golden" / "reference_sources_v1.json"


class ReferenceBuild:
    """ctypes face of tests/ref_build/ref_capi.cpp"""

    def __init__(self, path):
        self.path = path
        self.L = C.CDLL(str(path))
        L = self.L
        L.rdref_last_error.restype = C.c_char_p
        L.rdref_create.restype = C.c_void_p
        L.rdref_create.argtypes = [C.c_char_p, C.c_char_p, C.c_uint, C.c_ulonglong, C.c_int, C.c_char_p]
        L.rdref_destroy.argtypes = [C.c_void_p]
        L.rdref_root_count.argtypes = [C.c_void_p]
        L.rdref_root_count.restype = C.c_uint
        L.rdref_search.argtypes = [C.c_void_p, C.c_uint, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_int, _up, _dp, _dp]
        L.rdref_exhaustive.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double, _up, _dp, _dp,
                                       C.c_uint, _up, _up, _dp]
        L.rdref_all_root_lh.argtypes = [C.c_void_p, _dp, C.c_uint]

    def model(self, fx_name: str, rate_cats: int, seed: int, early_stop: bool, tmp, alignment=None):
        a, t = fixtures.FILES[fx_name]
        h = self.L.rdref_create(str(fixtures.FX / t).encode(), str(alignment or fixtures.FX / a).encode(), rate_cats,
                                seed, 1 if early_stop else 0, os.path.join(tmp, "ref").encode())
        if not h:
            raise RuntimeError(self.L.rdref_last_error().decode())
        return C.c_void_p(h)

    def check(self, rc):
        if not rc:
            raise RuntimeError(self.L.rdref_last_error().decode())

    def search(self, fx_name, K, seed, strategy):
        """-> (root count, root id, alpha, log-likelihood) of model_t::search"""
        with tempfile.TemporaryDirectory() as tmp:
            h = self.model(fx_name, K, seed, True, tmp)
            rid, alpha, lh = C.c_uint(), C.c_double(), C.c_double()
            self.check(self.L.rdref_search(h, 2, 0.05, 1e-3, 1e-3, 1e-4, 1e12, strategy, C.byref(rid), C.byref(alpha),
                                           C.byref(lh)))
            n_roots = self.L.rdref_root_count(h)
            self.L.rdref_destroy(h)
        return n_roots, rid.value, alpha.value, lh.value

    def exhaustive(self, fx_name, K, seed):
        """-> (root ids, log-likelihoods, alphas) of exhaustive_search, ordered by root id"""
        with tempfile.TemporaryDirectory() as tmp:
            h = self.model(fx_name, K, seed, False, tmp)
            n = self.L.rdref_root_count(h)
            ids, llh, alpha = np.zeros(n, dtype=np.uint32), np.zeros(n), np.zeros(n)
            got_n, best_id, best_lh = C.c_uint(), C.c_uint(), C.c_double()
            self.check(self.L.rdref_exhaustive(h, 1e-2, 1e-2, 1e-3, 1e13, ids.ctypes.data_as(_up),
                                               llh.ctypes.data_as(_dp), alpha.ctypes.data_as(_dp), n, C.byref(got_n),
                                               C.byref(best_id), C.byref(best_lh)))
            self.L.rdref_destroy(h)
        assert got_n.value == n
        assert int(ids[np.argmax(llh)]) == best_id.value
        order = np.argsort(ids)
        return ids[order], llh[order], alpha[order]

    def all_root_lh(self, fx_name, K, seed, alignment=None):
        """-> compute_all_root_lh (early stop on), from the fixture's alignment or the file `alignment`"""
        with tempfile.TemporaryDirectory() as tmp:
            h = self.model(fx_name, K, seed, True, tmp, alignment)
            n = self.L.rdref_root_count(h)
            out = np.zeros(n)
            self.check(self.L.rdref_all_root_lh(h, out.ctypes.data_as(_dp), n))
            self.L.rdref_destroy(h)
        return out


class RecordedReference:
    """the reference's results on the calls above, from tests/golden/reference_sources_v1.json (the
    alignment files of tests/test_msa.py are not read: every form must give the fixture's record)"""

    def __init__(self):
        self.rec = json.loads(GOLDEN.read_text())

    @staticmethod
    def _f(values):
        return np.array([float.fromhex(v) for v in values])

    def _find(self, kind, **key):
        hits = [r for r in self.rec[kind] if all(r[k] == v for k, v in key.items())]
        assert len(hits) == 1, (kind, key)
        return hits[0]

    def search(self, fx_name, K, seed, strategy):
        r = self._find("search", fixture=fx_name, rate_cats=K, seed=seed, strategy=strategy)
        return r["root_count"], r["root_id"], float.fromhex(r["alpha"]), float.fromhex(r["llh"])

    def exhaustive(self, fx_name, K, seed):
        r = self._find("exhaustive", fixture=fx_name, rate_cats=K, seed=seed)
        return np.array(r["root_ids"], dtype=np.uint32), self._f(r["llh"]), self._f(r["alpha"])

    def all_root_lh(self, fx_name, K, seed, alignment=None):
        # every on-disk form of the fixture's alignment is the same alignment (tests/test_msa.py)
        return self._f(self._find("every_root", fixture=fx_name, rate_cats=K, seed=seed)["llh"])


def reference(backend: str):
    """RootDigger's sources built against `backend` when a checkout (or a library built from one) is
    here, else the record of what they returned; skips without either"""
    path = oracle_build.build_reference_sources(backend)
    if path is not None and path.exists():
        origin = ("built now from $ROOTDIGGER_SRC = %s" % oracle_build.REFERENCE if oracle_build.REFERENCE
                  else "a library built earlier, not rebuilt against the current host sources")
        warnings.warn("comparing with RootDigger's own sources: %s (%s)" % (path, origin))
        return ReferenceBuild(path)
    if GOLDEN.exists():
        warnings.warn("comparing with the recorded results of RootDigger's own sources: %s" % GOLDEN)
        return RecordedReference()
    pytest.skip("RootDigger's sources are not here: set $ROOTDIGGER_SRC to a RootDigger checkout "
                "(tests/golden/make_reference_golden.py records its results)")


@pytest.fixture(scope="module")
def ref():
    oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
    return reference("oracle")


@pytest.fixture(scope="module")
def mirror_lib():
    oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
    return capi.load_tree_lib(oracle_build.build_host_on_oracle())


def mirror_model(lib, fx_name, rate_cats, seed, early_stop):
    a, t = fixtures.FILES[fx_name]
    tree = capi.RootedTree(path=str(fixtures.FX / t), lib=lib)
    m = capi.Model.from_files(tree, fixtures.FX / a, None, rate_cats, seed=seed, early_stop=early_stop)
    try:
        m.initialize_partitions(uniform_freqs=False)
    except RuntimeError:
        m.initialize_partitions(uniform_freqs=True)
    m.L.rdh_model_initialize(m.h) if hasattr(m.L, "rdh_model_initialize") else None
    return m


def same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def check_search(ref, mirror_lib, fx_name, K, strategy):
    n_roots, rid, alpha, lh = ref.search(fx_name, K, 7, strategy)
    m = mirror_model(mirror_lib, fx_name, K, 7, True)
    assert m.root_count == n_roots
    got = m.search(2, 0.05, 1e-3, 1e-3, 1e-4, 1e12, strategy=["random", "midpoint", "modified_mad"][strategy])
    m.close()
    assert got[0] == rid
    assert same([got[1], got[2]], [alpha, lh]), (got, rid, alpha, lh)


def check_exhaustive(ref, mirror_lib, K):
    ids, llh, alpha = ref.exhaustive("10.fasta", K, 3)
    m = mirror_model(mirror_lib, "10.fasta", K, 3, False)
    mids, mllh, malpha = m.exhaustive_search(1e-2, 1e-2, 1e-3, 1e13)
    order_m = np.argsort(mids)
    assert np.array_equal(ids, mids[order_m])
    assert same(llh, mllh[order_m]) and same(alpha, malpha[order_m])
    assert int(mids[np.argmax(mllh)]) == int(ids[np.argmax(llh)])
    assert same(m.lwr(mllh[order_m]), m.lwr(llh))
    m.close()


def check_every_root(ref, mirror_lib):
    out = ref.all_root_lh("101.phy", 4, 11)
    m = mirror_model(mirror_lib, "101.phy", 4, 11, True)
    want = m.compute_all_root_lh()
    m.close()
    assert same(out, want)


# ---- the CPU suite keeps the light cases (both sides on the oracle); tests/test_gpu_reference_sources.py
# ---- runs the heavy ones (4 categories, exhaustive mode) on the CUDA engine
@pytest.mark.parametrize("K,strategy", [(1, 1), (2, 0)])
def test_search_with_the_reference_sources_equals_the_mirror(ref, mirror_lib, K, strategy):
    """model_t::search (src/model.cpp:1008-1138) from the reference's own file: same root, same
    position on the branch, same log-likelihood, bit for bit"""
    check_search(ref, mirror_lib, "10.fasta", K, strategy)


def test_every_root_with_the_reference_sources_equals_the_mirror(ref, mirror_lib):
    """compute_all_root_lh (src/model.cpp:1737-1746): move_root + compute_lh per root through the
    reference's own tree.cpp schedules and the compat tree module"""
    check_every_root(ref, mirror_lib)
