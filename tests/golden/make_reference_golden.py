"""Writes tests/golden/reference_sources_v1.json: what RootDigger's own src/model.cpp, tree.cpp and
msa.cpp return for the calls tests/test_reference_sources.py, tests/test_gpu_reference_sources.py and
tests/test_msa.py make on the bundled fixtures, so that those tests compare with the reference without
a RootDigger checkout.  Doubles are stored as hex strings (bit exact).

The values come from RootDigger's sources themselves, compiled against the oracle behind the engine's
ABI (oracle/oracle_build.py build_reference_sources, engine arithmetic) and linked with RootDigger's
own L-BFGS-B (its lib/lbfgsb); nothing of this repository's model_t mirror is run.  Without a checkout
the script refuses to run.

usage: ROOTDIGGER_SRC=/path/to/root_digger python tests/golden/make_reference_golden.py
"""
import json
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "oracle"))

import oracle_build  # noqa: E402
import oracle_capi  # noqa: E402
from root_digger_b200 import _build  # noqa: E402
from test_reference_sources import EVERY_ROOT, EXHAUSTIVE, SEARCHES, ReferenceBuild  # noqa: E402


def hx(values):
    return [float(v).hex() for v in np.atleast_1d(values)]


def main():
    if oracle_build.REFERENCE is None or not (oracle_build.REFERENCE / "src" / "model.cpp").exists():
        raise SystemExit("set ROOTDIGGER_SRC to a RootDigger checkout: the record holds what ITS sources return")
    lbfgsb_src = oracle_build.REFERENCE / "lib" / "lbfgsb"
    if not list(lbfgsb_src.glob("*.c")):
        raise SystemExit("%s holds no L-BFGS-B sources" % lbfgsb_src)
    os.environ["RDK_LBFGSB_SRC"] = str(lbfgsb_src)
    try:
        _build.build_lbfgsb(force=True)
        ref = ReferenceBuild(oracle_build.build_reference_sources("oracle", force=True))
        oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
        out = {"version": 1, "search": [], "every_root": [], "exhaustive": []}
        for fx_name, K, seed, strategy in SEARCHES:
            n_roots, rid, alpha, lh = ref.search(fx_name, K, seed, strategy)
            out["search"].append({"fixture": fx_name, "rate_cats": K, "seed": seed, "strategy": strategy,
                                  "root_count": int(n_roots), "root_id": int(rid), "alpha": hx(alpha)[0],
                                  "llh": hx(lh)[0]})
        for fx_name, K, seed in EVERY_ROOT:
            out["every_root"].append({"fixture": fx_name, "rate_cats": K, "seed": seed,
                                      "llh": hx(ref.all_root_lh(fx_name, K, seed))})
        for fx_name, K, seed in EXHAUSTIVE:
            ids, llh, alpha = ref.exhaustive(fx_name, K, seed)
            out["exhaustive"].append({"fixture": fx_name, "rate_cats": K, "seed": seed,
                                      "root_ids": [int(i) for i in ids], "llh": hx(llh), "alpha": hx(alpha)})
    finally:  # the product's lib/liblbfgsb.so is this repository's again
        del os.environ["RDK_LBFGSB_SRC"]
        _build.build_lbfgsb(force=True)
    path = Path(__file__).with_name("reference_sources_v1.json")
    path.write_text(json.dumps(out, indent=1) + "\n")
    print("wrote", path)


if __name__ == "__main__":
    main()
