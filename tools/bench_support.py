#!/usr/bin/env python3
"""Times root placement support (Model.placement_support, DESIGN.md section 10) at the cfg2 shape:
a synthetic 500-taxon x 100 000-site alignment, 4 Gamma categories, a checkpoint holding all 2n-3
placements (written record by record with Checkpoint.write, no search), B = 1 000 and 10 000.

Prints one JSON line: per B the median over --reps calls (after one warm-up call) of the capture
(host wall time of the 2n-3 full evaluations that store the rows), and of the counts, accumulation
and statistics kernels (CUDA events inside the engine), the accumulation's term rate
(B x patterns x records / accumulation time), the device memory the resampling allocated, and the
card's name and power limit read in the same run.

With --au-scales (e.g. 0.5,0.6,...,1.4, or "default" for capi.AU_SCALES) every call also runs the
AU test's multiscale bootstrap and the expected likelihood weights, and the line adds their phases:
multiscale counts, multiscale accumulation, and statistics + ELW.

With --branches it times branch support instead (Model.branch_support, DESIGN.md section 10, items
9-10): the checkpoint holds ONE record, as after a search-mode run, and every call scores all 2n-3
branches at that record's parameters.  Per B the line gives the median of positions_ms (the 2n-3
position searches), capture_ms (the one placement sweep that stores the rows) and the resampling
phases, and, next to them, the capture_ms of placement_support on the equivalent 2n-3-record
checkpoint (the record-by-record capture this mode replaces), measured once at the first B.

    python tools/bench_support.py [--taxa 500] [--sites 100000] [--replicates 1000,10000] [--reps 3]
                                  [--au-scales default] [--branches] [--atol 1e-14]
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402


def card():
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_support.py needs a CUDA device")
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in out.split(",")]
    except Exception as exc:  # the number is still reported, without its card settings
        info["power_limit"] = "unavailable: %s" % exc
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--taxa", type=int, default=500)
    ap.add_argument("--sites", type=int, default=100000)
    ap.add_argument("--cats", type=int, default=4)
    ap.add_argument("--replicates", default="1000,10000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0x5EED0002)
    ap.add_argument("--au-scales", default=None, help='comma-separated scales, or "default" (capi.AU_SCALES)')
    ap.add_argument("--branches", action="store_true", help="time branch_support from a one-record checkpoint")
    ap.add_argument("--atol", type=float, default=1e-14, help="--branches: tolerance of the position searches")
    args = ap.parse_args()

    from root_digger_b200 import capi, synth
    au = None
    if args.au_scales:
        au = capi.AU_SCALES if args.au_scales == "default" else [float(v) for v in args.au_scales.split(",")]
    device = card()
    top = synth.random_tree(args.taxa, args.seed)
    rates, freqs = synth.random_params(args.seed + 1)
    aln = synth.simulate_alignment(top, args.sites, args.seed + 2, rates, freqs, capi.gamma_cats(1.0, args.cats))
    m = capi.Model(capi.RootedTree(synth.to_newick(top)), aln, rate_cats=args.cats, seed=1)
    m.initialize_partitions(uniform_freqs=False)
    R, P = m.root_count, m.sites(0)
    r12, f4, _ = m.get_params()
    rng = np.random.default_rng(args.seed + 3)
    if args.branches:
        return branches(args, m, au, device, r12, f4, rng)
    with tempfile.TemporaryDirectory() as tmp:
        prefix = str(Path(tmp) / "support")
        ckp = capi.Checkpoint(prefix)
        ckp.save_options(prefix=prefix)
        for rid in range(R):
            params = [{"rates": r12, "freqs": f4, "alpha": float(rng.uniform(0.5, 2.0)),
                       "weights": np.full(args.cats, 1.0 / args.cats)}]
            ckp.write(rid, 0.0, float(rng.uniform(0.0, 1.0)), params, K=args.cats)
        ckp.close()
        results = {}
        for B in [int(b) for b in args.replicates.split(",")]:
            m.placement_support(prefix, replicates=B, seed=1, au_scales=au)  # warm-up: module load, allocations
            runs = [m.placement_support(prefix, replicates=B, seed=1 + i, au_scales=au) for i in range(args.reps)]
            keys = ["capture_ms", "counts_ms", "accumulate_ms", "statistics_ms", "resample_ms"]
            if au:
                keys += ["au_counts_ms", "au_accumulate_ms", "au_statistics_ms"]
            med = {k: statistics.median(r[k] for r in runs) for k in keys}
            med["accumulate_terms_per_s"] = B * P * R / (med["accumulate_ms"] / 1e3)
            med["device_bytes"] = max(r["device_bytes"] for r in runs)
            med["bp_sum"] = int(runs[0]["bp_count"].sum())
            if au:
                extra = len(au) - (1 if 1.0 in au else 0)  # scales resampled beyond the unit scale
                med["au_terms_per_s"] = B * P * R * extra / (med["au_accumulate_ms"] / 1e3)
                med["au_extra_scales"] = extra
                med["elw_sum"] = float(runs[0]["elw"].sum())
            results[str(B)] = med
    line = {"tool": "bench_support", "taxa": args.taxa, "patterns": P, "records": R, "cats": args.cats,
            "reps": args.reps, "card": device, "results": results}
    if au:
        line["au_scales"] = list(au)
    print(json.dumps(line))


def branches(args, m, au, device, r12, f4, rng):
    from root_digger_b200 import capi
    R, P = m.root_count, m.sites(0)
    params = [{"rates": r12, "freqs": f4, "alpha": float(rng.uniform(0.5, 2.0)),
               "weights": np.full(args.cats, 1.0 / args.cats)}]
    results = {}
    with tempfile.TemporaryDirectory() as tmp:
        one = str(Path(tmp) / "search")
        ckp = capi.Checkpoint(one)
        ckp.save_options(prefix=one)
        ckp.write(R // 2, 0.0, 0.5, params, K=args.cats)
        ckp.close()
        Bs = [int(b) for b in args.replicates.split(",")]
        kw = dict(atol=args.atol, au_scales=au)
        first = m.branch_support(one, replicates=Bs[0], seed=1, **kw)  # warm-up: module load, allocations
        # the record-by-record capture of the same 2n-3 placements, for comparison
        eq = str(Path(tmp) / "equivalent")
        ckp = capi.Checkpoint(eq)
        ckp.save_options(prefix=eq)
        for q in range(R):
            ckp.write(q, 0.0, float(first["alpha"][q]), params, K=args.cats)
        ckp.close()
        checkpoint_capture_ms = m.placement_support(eq, replicates=Bs[0], seed=1, au_scales=au)["capture_ms"]
        for B in Bs:
            runs = [m.branch_support(one, replicates=B, seed=1 + i, **kw) for i in range(args.reps)]
            keys = ["positions_ms", "capture_ms", "counts_ms", "accumulate_ms", "statistics_ms", "resample_ms"]
            if au:
                keys += ["au_counts_ms", "au_accumulate_ms", "au_statistics_ms"]
            med = {k: statistics.median(r[k] for r in runs) for k in keys}
            med["device_bytes"] = max(r["device_bytes"] for r in runs)
            med["bp_sum"] = int(runs[0]["bp_count"].sum())
            med["same_positions"] = all(np.array_equal(r["alpha"], first["alpha"]) for r in runs)
            results[str(B)] = med
    line = {"tool": "bench_support", "mode": "branches", "taxa": args.taxa, "patterns": P, "records": R,
            "cats": args.cats, "reps": args.reps, "atol": args.atol, "card": device,
            "checkpoint_capture_ms": checkpoint_capture_ms, "row_bytes": 8 * P * R, "results": results}
    if au:
        line["au_scales"] = list(au)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
