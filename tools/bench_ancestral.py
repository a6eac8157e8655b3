#!/usr/bin/env python3
"""Times rdk_marginal_ancestral_states (Model.ancestral_states; DESIGN.md section 11) at the cfg2 shape:
500 taxa x 100 000 patterns, Gamma 4, one GPU.  Reports the device time of the pass, the bytes it
moves by its own accounting (per node: the two child CLVs or tip rows, o_v, o_c1 / o_c2, the outputs)
against the HBM peak bench.py uses, and the device memory the call allocates.  Prints one JSON line;
writes nothing unless --out is given.

    python tools/bench_ancestral.py [--taxa 500] [--sites 100000] [--repeats 5] [--out FILE]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from root_digger_b200 import capi, synth  # noqa: E402


def hbm_peak():
    """the HBM bandwidth bench.py divides by: MEASURED_PEAKS.json hbm_gbs when present"""
    import bench
    return bench.peaks()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--taxa", type=int, default=500)
    ap.add_argument("--sites", type=int, default=100000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    top = synth.random_tree(a.taxa, 17, 0.05)
    tree = capi.RootedTree(synth.to_newick(top))
    aln = synth.iid_alignment(synth.tip_labels(top), a.sites, 19)
    m = capi.Model(tree, aln, rate_cats=4, compress=False, seed=3)
    m.initialize_partitions()
    m.compute_lh(7, 0.5)
    m.ancestral_states(7, 0.5)  # warm-up: module load, first allocations
    times = []
    for _ in range(a.repeats):
        r = m.ancestral_states(7, 0.5)
        times.append(r["ms"][0])
    S, K, n = m.sites(0), 4, len(r["nodes"])
    clv = S * K * 4 * 8
    inner_children = sum(1 for o in r["ops"] for c in (o[2], o[5]) if c >= a.taxa)
    tip_children = 2 * n - inner_children
    moved = (inner_children * clv          # child CLVs read
             + tip_children * S            # tip codes read
             + (n - 1) * clv               # o_v read (the root's is pi)
             + inner_children * clv        # o_c written
             + n * S * (1 + 8 + 8)         # map_state, map_prob, log_norm
             + S * 32)                     # the root's posterior
    peak, peak_src = hbm_peak()
    ms = float(np.median(times))
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        gpu = "unknown"
    res = {"taxa": a.taxa, "patterns": S, "K": K, "nodes": n, "ms_median": ms, "ms_all": times,
           "bytes_moved": moved, "gb_per_s": moved / ms / 1e6, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
           "share_of_hbm_peak": moved / ms / 1e6 / peak, "device_bytes": r["device_bytes"][0], "gpu": gpu}
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
