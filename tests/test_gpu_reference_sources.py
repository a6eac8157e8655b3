"""tests/test_reference_sources.py on the CUDA engine: RootDigger's own src/model.cpp, src/tree.cpp,
src/msa.cpp (unchanged, compiled against root_digger_b200/compat/corax/corax.h + librdk_b200.so) next
to the engine host's model_t mirror (librd_host.so), both on cuda:0 through include/rdk.h: search with
4 and 3 rate categories, exhaustive mode with its LWR inputs, every root of 101.phy -- bit for bit.
Without a RootDigger checkout the reference's side is its recorded results (t.RecordedReference)."""
import pytest

import test_reference_sources as t
from root_digger_b200 import capi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    return t.reference("engine")


@pytest.fixture(scope="module")
def mirror_lib():
    return capi.load_tree_lib()


@pytest.mark.parametrize("K,strategy", [(4, 2), (3, 0), (1, 1)])
def test_search_with_the_reference_sources_on_the_engine(ref, mirror_lib, K, strategy):
    t.check_search(ref, mirror_lib, "10.fasta", K, strategy)


def test_exhaustive_mode_with_the_reference_sources_on_the_engine(ref, mirror_lib):
    """exhaustive_search + the LWR inputs (src/model.cpp:1140-1258): per-branch log-likelihoods and
    root positions identical, hence the LWR ranking"""
    t.check_exhaustive(ref, mirror_lib, 4)


def test_every_root_with_the_reference_sources_on_the_engine(ref, mirror_lib):
    t.check_every_root(ref, mirror_lib)
