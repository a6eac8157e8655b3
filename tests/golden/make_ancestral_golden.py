"""Writes tests/golden/ancestral_small{.state,.fasta} and ancestral_small_parts{.state,.fasta}: the .state
tables and root sequences capi.write_state_file writes for the 6-taxon case of
tests/test_ancestral_cpu.py on the oracle-backed host (every node; two partitions, root only).
tests/test_ancestral_cpu.py::test_the_state_file_is_the_golden_one compares with them byte for byte.

    python tests/golden/make_ancestral_golden.py
"""
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent.parent / "oracle"))

import oracle_build  # noqa: E402
import oracle_capi  # noqa: E402
import test_ancestral_cpu as t  # noqa: E402
from root_digger_b200 import capi  # noqa: E402


def main():
    oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
    lib = capi.load_tree_lib(oracle_build.build_host_on_oracle())
    for name, parts, full in (("ancestral_small", None, "all"), ("ancestral_small_parts", t.SMALL_PARTS, "root")):
        m = t.small_model(lib, 4, parts)
        res = m.ancestral_states(t.GOLDEN_ROOT, 0.3, full_nodes=full)
        capi.write_state_file(res, HERE / (name + ".state"))


if __name__ == "__main__":
    main()
