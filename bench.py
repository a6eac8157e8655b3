#!/usr/bin/env python
"""bench.py -- root placements evaluated per second + CLV-update GB/s (BASELINE.json metric).

Workload (BASELINE.json configs[1]): synthetic 500-taxon x 100 000-site DNA alignment, UNREST
model, 4 Gamma categories, search mode.  One STEP is what one outer iteration of
model_t::search needs from the likelihood engine to score every candidate root
(reference src/model.cpp:1051-1057 -> optimize_root_location :796 -> suggest_roots_lh :865-889):

    1 full evaluation           model_t::compute_lh        (n-1 CLV operations + root logL)
  + 1 placement sweep           model_t::suggest_roots_lh  (for each of the 2n-3 candidate
                                root branches: move_root + compute_lh_root)

value   = (2n-3) placements x K steps / device time, schedules and alignment already
          resident (host arrays pre-built, tips in HBM); CUDA events on the engine's stream.
e2e     = the same step through the host model_t mirror (librd_host.so: C++ traversal
          scheduler generates the op lists each step, programs go host->device, the 2n-3
          log-likelihoods come back device->host), wall clock around the public calls.
roofline= the dominant kernel (clv_program_kernel): algorithmic bytes (SURVEY 8d table, counted
          per launch by the engine) / its device time (CUDA events bracketing each launch).

N > 1 (strong scaling: the global problem is fixed), one process per GPU, N = G_s x G_r
(root_digger_b200.sharding.plan_grid, SURVEY 8e).  Default G_s = N: the alignment's sites are
split into N contiguous, 256-aligned shards, CLVs resident per GPU, ONE NCCL all-reduce of the
per-shard tree nodes per evaluation batch (the north-star layout).  --shard roots keeps a replica
per GPU and splits the 2n-3 candidate placements of the sweep into N contiguous chunks instead
(the rule exhaustive mode uses for ranks, reference src/model.cpp:1899-1907; no data-path
collective, one all-gather of the log-likelihoods per step) -- but every rank then repeats the
full evaluation, and measured on B200 (profiles/r01_bench_e4_n{4,8}_{sites,roots}.json) the site
shards win from N = 4 up: 296.5 k vs 228.2 k placements/s at N = 8, 187.8 k vs 183.9 k at N = 4.

--impl reference: the CPU oracle restatement of the same step (the reference's coraxlib is an
absent submodule: it cannot be built, SURVEY 8c), all host threads, on a bounded site sample.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import numpy as np  # noqa: E402

METRIC = "root_placements_per_sec"
UNIT = "placements/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--taxa", type=int, default=500)
    ap.add_argument("--sites", type=int, default=100000)
    ap.add_argument("--cats", type=int, default=4)
    ap.add_argument("--data", default="evolved", choices=["evolved", "iid"])
    ap.add_argument("--seed", type=int, default=0x5EED0002)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--exhaustive-branches", type=int, default=1,
                    help="also time exhaustive mode (one placement = one fully optimised branch, SURVEY 8d) on "
                         "this many branches of the e2e model (0 = skip; each branch is thousands of evaluations)")
    ap.add_argument("--north-star", default="auto",
                    help="the BASELINE configs beyond the headline, appended to the line as `north_star`: a comma "
                         "list of cfg3,cfg4,cfg5, `all`, `off`, or `auto` (= all when --gpus 8, else off)")
    ap.add_argument("--ns-scale", type=float, default=1.0,
                    help="shrink the north-star configs (taxa and sites) by this factor: functional runs on small boxes")
    ap.add_argument("--ns-exhaustive-branches", type=int, default=1)
    ap.add_argument("--ns-exhaustive-iterations", type=int, default=2,
                    help="cap on the outer iterations per branch of the cfg3 exhaustive sample (0 = to convergence: "
                         "~9e4 full evaluations, 7 minutes per branch on 8 GPUs)")
    ap.add_argument("--launch-config", default="", help="ctas_per_sm,threads,elems (0 = engine default)")
    ap.add_argument("--tail-mode", type=int, default=0, help="0 engine rule, 1 always skip idle slots, 2 never")
    ap.add_argument("--sweep", default="directed", choices=["directed", "path"],
                    help="how our arm scores the 2n-3 placements: one pre-order pass over directed CLVs "
                         "(default) or the reference-shaped move_root path per placement; identical values")
    ap.add_argument("--chunks", type=int, default=0,
                    help="independent chunks of the directed sweep (0 = the engine's hint for the shard size)")
    ap.add_argument("--shard", default="sites", choices=["auto", "sites", "roots"],
                    help="N > 1: sites = one site shard per GPU (the north-star layout: one all-reduce per "
                         "evaluation batch); roots = a replica per GPU, root placements in chunks; auto = fewest "
                         "site shards that fit HBM, rest over root placements (exhaustive mode's rule)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed to DIR/<name>.npy (float64): logl_root0 (the "
                         "full evaluation at root 0) and placement_logl (all 2n-3 placements, in root-id order); "
                         "the inputs are seeded, so two builds run with the same arguments can be compared")
    return ap.parse_args()


def dump_outputs(out_dir: str, **arrays):
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / (name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpus):
        self.gpus = gpus
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", ",".join(str(g) for g in self.gpus)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_first(self, timeout=3.0):
        """block until nvidia-smi has delivered its first sample: its start-up (NVML initialisation takes
        driver locks for 0.1-0.3 s) is then over and does not fall into a timed region of a few tens of ms"""
        t0 = time.time()
        while self.proc and not self.lines and time.time() - t0 < timeout and self.proc.poll() is None:
            time.sleep(0.01)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def build_case(args):
    from cases import Case
    from root_digger_b200.capi import gamma_cats
    return Case(args.taxa, args.sites, args.cats, seed=args.seed, data=args.data, alpha=1.0, gamma_cats=gamma_cats)


def step_bytes_formula(n, S, K):
    """SURVEY 8d: bytes of one full evaluation, per site count S (unfused accounting)"""
    return S * ((n - 1) * (64 * K + 8) + n)


# ---------------------------------------------------------------------------------------------
# reference arm: CPU oracle, all host threads, bounded site sample
# ---------------------------------------------------------------------------------------------
def oracle_step(o, case, full_arr, full_pm, full_br, sw, sw_ops_arrs, threads):
    """one step on the oracle: compute_lh(root 0) + the sweep, as the three reference calls"""
    o.update_prob_matrices(full_pm, full_br)
    o.L.rdo_update_clvs_mt(o.p, full_arr, len(full_arr), threads)
    lh0 = o.root_loglikelihood_mt(case.root_clv, case.root_scaler, threads)
    pm_off, mi, bl, op_off, _ = sw
    out = np.zeros(len(pm_off) - 1)
    for q in range(len(pm_off) - 1):
        a, b = pm_off[q], pm_off[q + 1]
        if b > a:
            o.update_prob_matrices(mi[a:b], bl[a:b])
        arr, cnt = sw_ops_arrs[q]
        if cnt:
            o.L.rdo_update_clvs_mt(o.p, arr, cnt, threads)
        out[q] = o.root_loglikelihood_mt(case.root_clv, case.root_scaler, threads)
    return lh0, out


def cpu_reference_run(args, case, steps, warmup, threads, target_step_s=1.5, quiet=False):
    """times the oracle on a site sample; returns (placements/s scaled to the full site count, info)"""
    from oracle_capi import OraclePartition
    from root_digger_b200.capi import ops_array
    n, S, K = case.n, case.S, case.K
    full_ops, full_pm, full_br = case.full_schedule(0, 0.5)
    full_arr = ops_array(full_ops)
    roots = list(range(case.tree.root_count))
    sw = case.sweep_schedule(roots, 0.5)
    pm_off, mi, bl, op_off, ops = sw
    sw_ops_arrs = []
    for q in range(len(roots)):
        sub = ops[op_off[q]:op_off[q + 1]]
        sw_ops_arrs.append((ops_array(sub), len(sub)))

    def make(sample):
        o = OraclePartition(n, sample, K)
        case.setup(o, slice(0, sample))
        return o

    # calibrate the sample so that one step costs about target_step_s
    probe = min(S, 1024)
    o = make(probe)
    oracle_step(o, case, full_arr, full_pm, full_br, sw, sw_ops_arrs, threads)  # first touch, thread start-up
    t0 = time.perf_counter()
    oracle_step(o, case, full_arr, full_pm, full_br, sw, sw_ops_arrs, threads)
    t_probe = time.perf_counter() - t0
    o.close()
    sample = int(min(S, max(probe, probe * target_step_s / max(t_probe, 1e-6))))
    sample = max(256, (sample // 256) * 256) if sample < S else S
    o = make(sample)
    for _ in range(warmup):
        oracle_step(o, case, full_arr, full_pm, full_br, sw, sw_ops_arrs, threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle_step(o, case, full_arr, full_pm, full_br, sw, sw_ops_arrs, threads)
    dt = time.perf_counter() - t0
    o.close()
    ms_step_sample = dt / steps * 1e3
    ms_step_full = ms_step_sample * S / sample
    value = len(roots) / (ms_step_full * 1e-3)
    info = {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "oracle/rd_oracle.c (CPU restatement; coraxlib is an absent submodule), OpenMP site-parallel, "
                      "%d of %d sites of the same alignment, all %d placements, %d steps; scaled by sites"
                      % (sample, S, len(roots), steps),
            "ms_per_step_full_size": ms_step_full, "ms_per_step_sample": ms_step_sample, "timed_seconds": dt,
            "sample_sites": sample}
    return value, info, ms_step_full


def cpu_single_thread(args, case):
    """what the reference itself would do on this single-partition workload: it threads over
    partitions only (SURVEY F5), i.e. ONE thread; short bounded sample, scaled by sites"""
    v, info, ms = cpu_reference_run(args, case, steps=1, warmup=0, threads=1, target_step_s=1.0)
    return {"value": v, "unit": UNIT, "cores": 1, "ms_per_step_full_size": ms, "sample": info["sample"]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from root_digger_b200.sharding import plan_grid
    threads = os.cpu_count() or 1
    case = build_case_cpu(args)
    value, info, ms_full = cpu_reference_run(args, case, args.steps, args.warmup, threads)
    info["single_thread"] = cpu_single_thread(args, case)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_full, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, case.tree.root_count,
                                  plan_grid(args.gpus, case.n, case.S, case.K, force=args.shard)),
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "native_libraries_mapped": sorted({l.split("/")[-1].strip() for l in open("/proc/self/maps")
                                           if "/root_digger_b200/lib/" in l or "/tests/_build/" in l or "/oracle/" in l}),
    }
    print(json.dumps(line), flush=True)


def build_case_cpu(args):
    """the reference arm must not map the CUDA libraries: gamma categories from the oracle, traversal
    schedules from the host sources compiled against the oracle (tests/_build/librd_host_oracle.so)"""
    sys.path.insert(0, str(ROOT / "oracle"))
    import oracle_build
    from cases import Case
    from root_digger_b200 import capi
    lib = capi.load_tree_lib(oracle_build.build_host_on_oracle())
    return Case(args.taxa, args.sites, args.cats, seed=args.seed, data=args.data, alpha=1.0, tree_lib=lib)


def workload_config(args, placements, grid=None):
    return {"workload": "cfg2: synthetic %d-taxon x %d-site DNA, UNREST+G%d, search-mode step = 1 full "
                        "evaluation (compute_lh) + 1 sweep of all %d candidate root placements "
                        "(suggest_roots_lh: move_root + compute_lh_root each)"
                        % (args.taxa, args.sites, args.cats, placements),
            "taxa": args.taxa, "sites": args.sites, "rate_cats": args.cats, "placements_per_step": placements,
            "alignment": args.data,
            "sharding": "sites/%d x root-placements/%d" % (grid if grid else (args.gpus, 1)),
            "l2_policy": "inputs larger than L2 (inner CLVs %.1f GB per GPU vs 126 MB L2)"
                         % ((args.taxa - 1) * 32.0 * args.cats * args.sites / (grid[0] if grid else args.gpus) / 1e9)}


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_gpus = world

    from cases import compute_lh
    from root_digger_b200 import capi
    from root_digger_b200.capi import Model, Partition, RootedTree, ops_array
    from root_digger_b200.sharding import plan_grid, plan_root_shards, plan_site_shards

    case = build_case(args)
    n, S, K = case.n, case.S, case.K
    # N = G_s site shards x G_r root-placement chunks; rank r: site shard r % G_s, chunk r // G_s
    G_s, G_r = plan_grid(world, n, S, K, force=args.shard)
    site_rank, root_group = rank % G_s, rank // G_s
    shards = plan_site_shards(S, G_s)
    off, cnt = shards[site_rank]
    sl = slice(off, off + cnt)

    def fresh_comm_id():
        """a new 128-byte NCCL unique id per site group (one per communicator), made by the group's
        first rank and shipped with torch.distributed"""
        if G_s == 1:
            return None
        mine = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if site_rank == 0:
            mine = torch.tensor(list(capi.comm_unique_id()), dtype=torch.uint8, device="cuda")
        ids = torch.zeros(world * 128, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(ids, mine)
        leader = root_group * G_s
        return bytes(ids[leader * 128:(leader + 1) * 128].cpu().tolist())

    comm_id = fresh_comm_id()

    # reference buffer counts + the spare buffers of the directed sweep, once per independent chunk of
    # placements (a small shard fills the device only when several chunks are walked side by side)
    # (site-sharded: the all-reduce adds the ranks' values slot by slot, so every rank must cut the
    # sweep the same way -- the count comes from the LARGEST shard, not from this rank's own)
    n_chunks = args.chunks if args.chunks > 0 else capi.sweep_chunk_hint(max(c for _, c in plan_site_shards(S, G_s)), K)
    lay = case.tree.sweep_layout(n_chunks)
    g = Partition(n, cnt, K, device=local, clv_buffers=lay["clv_buffers"], scale_buffers=lay["scale_buffers"],
                  prob_matrices=lay["prob_matrices"])
    g.set_stream(torch.cuda.current_stream().cuda_stream)
    case.setup(g, sl)
    if G_s > 1:
        g.set_shard(off, S)
        g.attach_comm(G_s, site_rank, comm_id)
    if args.launch_config:
        g.set_launch_config(*[int(x) for x in args.launch_config.split(",")])
    if args.tail_mode:
        g.set_tail_mode(args.tail_mode)

    full_ops, full_pm, full_br = case.full_schedule(0, 0.5)
    full_arr = ops_array(full_ops)
    placements = case.tree.root_count
    chunks = plan_root_shards(range(placements), G_r)
    roots = chunks[root_group]  # this rank's contiguous chunk of root ids
    if args.sweep == "directed":
        # the tree is rooted at root 0 (full_schedule above): directed-CLV pass over this rank's chunk
        pm_off, mi, bl, op_off, ops, pos, chunk_off = case.tree.generate_chunked_sweep_operations(
            roots[0], roots[-1] + 1, layout=lay)
        pos = pos - roots[0]
        sweep_flags = capi.RDK_SWEEP_KEEP_ROOT | capi.RDK_SWEEP_DISCARD
    else:
        pm_off, mi, bl, op_off, ops = case.sweep_schedule(roots, 0.5)
        pos = np.arange(len(roots))
        sweep_flags = 0
        chunk_off = None
    sw_arr = ops_array(ops)
    chunk_max = max(len(c) for c in chunks)
    gather_in = torch.zeros(chunk_max, dtype=torch.float64, device="cuda")
    gather_out = torch.zeros(world * chunk_max, dtype=torch.float64, device="cuda")
    pinned = torch.zeros(chunk_max, dtype=torch.float64).pin_memory()

    def gather_placements(mine):
        """every rank ends with all 2n-3 log-likelihoods (exhaustive mode's final gather)"""
        if G_r == 1:
            return mine
        pinned[:len(mine)] = torch.from_numpy(mine)
        gather_in.copy_(pinned, non_blocking=True)
        dist.all_gather_into_tensor(gather_out, gather_in)
        allv = gather_out.cpu().numpy().reshape(world, chunk_max)
        return np.concatenate([allv[q * G_s, :len(chunks[q])] for q in range(G_r)])

    # the device arm's driver: the C ABI called with pointers bound once (schedules resident on the host in
    # the ABI's own layout; what is timed is the engine, not numpy -> ctypes marshalling)
    import ctypes as C
    up, dp = C.POINTER(C.c_uint), C.POINTER(C.c_double)
    keep = [np.ascontiguousarray(full_pm, dtype=np.uint32), np.ascontiguousarray(full_br, dtype=np.float64),
            np.ascontiguousarray(pm_off, dtype=np.uint32), np.ascontiguousarray(mi, dtype=np.uint32),
            np.ascontiguousarray(bl, dtype=np.float64), np.ascontiguousarray(op_off, dtype=np.uint32),
            np.ascontiguousarray(chunk_off if chunk_off is not None else [0, len(pm_off) - 1], dtype=np.uint32),
            np.zeros(len(pm_off) - 1)]
    p_fpm, p_fbr, p_pmo, p_mi, p_bl, p_opo, p_co = [a.ctypes.data_as(dp if a.dtype == np.float64 else up) for a in keep[:7]]
    sw_out = keep[7]
    p_out = sw_out.ctypes.data_as(dp)
    n_full_pm, n_full_ops, n_pl, n_co = len(keep[0]), len(full_ops), len(pm_off) - 1, len(keep[6]) - 1
    L, zeros = g.L, g._zeros
    root_clv, root_scaler = case.root_clv, case.root_scaler

    def step():
        if L.rdk_update_prob_matrices(g.p, zeros, p_fpm, p_fbr, n_full_pm) != capi.RDK_SUCCESS:
            raise RuntimeError("rdk_update_prob_matrices failed")
        L.rdk_update_clvs(g.p, full_arr, n_full_ops)
        lh0 = L.rdk_compute_root_loglikelihood(g.p, root_clv, root_scaler, zeros, None)
        if chunk_off is None:
            rc = L.rdk_sweep_root_placements_ex(g.p, n_pl, zeros, zeros, p_pmo, p_mi, p_bl, p_opo, sw_arr, root_clv,
                                                root_scaler, sweep_flags, p_out)
        else:
            rc = L.rdk_sweep_root_placements_chunks(g.p, n_pl, zeros, zeros, p_pmo, p_mi, p_bl, p_opo, sw_arr, root_clv,
                                                    root_scaler, sweep_flags, n_co, p_co, p_out)
        if rc != capi.RDK_SUCCESS:
            raise RuntimeError("sweep failed: rdk_errno %d" % L.rdk_errno_location()[0])
        out = np.empty(len(pos))
        out[pos] = sw_out
        return lh0, gather_placements(out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the clock sampler runs from before the warm-up to the end of the measurements (it covers every timed
    # region); it is started, and past its start-up, before anything is timed
    sampler = ClockSampler(list(range(n_gpus))) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_first()
    for _ in range(max(3, args.warmup)):
        lh0, sweep_lh = step()
    g.set_timing(True)
    g.reset_stats()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        lh0, sweep_lh = step()
    ev1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, logl_root0=np.array([lh0]), placement_logl=sweep_lh)
    ms = ev0.elapsed_time(ev1)
    st = g.stats()
    g.set_timing(False)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    agg = torch.tensor([float(st["algorithmic_bytes"]), float(st["kernel_launches"])], dtype=torch.float64,
                       device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = placements * args.steps / (ms * 1e-3)
    total_alg_bytes = float(agg[0].item())
    clv_gbs = total_alg_bytes / (ms * 1e-3) / 1e9

    # roofline of the dominant kernel on this rank (rank 0 reports)
    peak, peak_src = peaks()
    prog_s = st["program_time_ns"] * 1e-9
    achieved = st["algorithmic_bytes"] / prog_s / 1e9 if prog_s > 0 else 0.0
    per_launch = st["algorithmic_bytes"] / max(1, st["program_timed"])
    prof = dram_traffic_from_profiles(n, cnt, K)
    launches_per_step = max(1, st["program_timed"]) / args.steps
    traffic = prof["dram_bytes_per_step"] / launches_per_step if prof else None
    roofline = {"bound": "hbm", "kernel": "clv_program_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                # measured DRAM bytes / kernel time / peak: how busy HBM really is (the contract `frac` counts
                # the algorithmic bytes, most of which the kernel forwards in registers or finds in L2)
                "dram_frac": (traffic / (prog_s / max(1, st["program_timed"])) / 1e9 / peak) if traffic and prog_s > 0 else None,
                "traffic_source": prof["source"] if prof else "this per-GPU configuration (%dx%dx%d) has no committed ncu "
                                                              "capture: null, not a number from another shape" % (n, cnt, K),
                "min_traffic": min_step_traffic(n, cnt, K) / launches_per_step,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": per_launch,
                "avg_launch_ms": prog_s * 1e3 / max(1, st["program_timed"]),
                "launches_timed": st["program_timed"],
                "kernel_share_of_step": prog_s * 1e3 / ms if ms > 0 else None,
                # where the rest of a step goes on the host (engine counters, ms per step, this rank)
                "host_ms_per_step": {"recording": st["host_record_ns"] * 1e-6 / args.steps,
                                     "lowering_and_enqueue": st["host_lower_ns"] * 1e-6 / args.steps,
                                     "waiting_for_device": st["host_wait_ns"] * 1e-6 / args.steps}}

    # ---- the unit of exhaustive mode / BFGS: one full evaluation (compute_lh), timed alone
    g.set_timing(True)
    g.reset_stats()
    barrier()
    fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fe0.record()
    for _ in range(args.steps):
        g.update_prob_matrices(full_pm, full_br)
        g.L.rdk_update_clvs(g.p, full_arr, len(full_ops))
        lh_full = g.root_loglikelihood(case.root_clv, case.root_scaler)
    fe1.record()
    barrier()
    fst = g.stats()
    g.set_timing(False)
    fe_ms = torch.tensor([fe0.elapsed_time(fe1) / args.steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(fe_ms, op=dist.ReduceOp.MAX)
    fe_ms = float(fe_ms.item())
    fe_kernel_s = fst["program_time_ns"] * 1e-9 / max(1, fst["program_timed"])
    fe_bytes = fst["algorithmic_bytes"] / args.steps
    full_eval = {"evaluations_per_sec": 1e3 / fe_ms, "ms": fe_ms, "kernel_ms": fe_kernel_s * 1e3,
                 "algorithmic_bytes_per_gpu": fe_bytes,
                 "kernel_gbs_per_gpu": fe_bytes / fe_kernel_s / 1e9 if fe_kernel_s > 0 else None,
                 "frac_of_hbm_peak": fe_bytes / fe_kernel_s / 1e9 / peak if fe_kernel_s > 0 else None,
                 "logl_matches_step": bool(lh_full == lh0)}

    # ---- e2e: the same step through the host model_t mirror (public API, host buffers)
    e2e = None
    if not args.no_e2e:
        tree = RootedTree(case.newick)
        aln = {l: s[sl] for l, s in case.aln.items()}
        m = Model(tree, aln, K, site_offset=off if G_s > 1 else 0, global_sites=S if G_s > 1 else 0,
                  nranks=G_s, rank=site_rank, comm_id=fresh_comm_id())
        m.initialize_partitions()
        m.set_params(rates=case.rates, freqs=case.freqs)
        m.set_sweep_mode(m.SWEEP_DIRECTED if args.sweep == "directed" else m.SWEEP_PATH)
        part = C.cast(m.L.rdh_model_partition(m.h, 0), C.POINTER(capi.PartitionStruct))
        L = capi.load_engine()

        def mstats():
            s = capi.Stats()
            L.rdk_partition_stats(part, C.byref(s))
            return s.asdict()

        def mstep():
            a = m.compute_lh(0, 0.5)
            b = m.sweep_root_lh(roots[0], roots[-1] + 1) if G_r > 1 else m.sweep_root_lh()
            return a, gather_placements(b)

        for _ in range(max(3, args.warmup)):
            a, b = mstep()
        L.rdk_partition_reset_stats(part)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            a, b = mstep()
        barrier()
        dt = time.perf_counter() - t0
        ms2 = torch.tensor([dt * 1e3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        s2 = mstats()
        e2e = {"value": placements * args.steps / (float(ms2.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": s2["h2d_bytes"] / args.steps, "d2h_bytes_per_step": s2["d2h_bytes"] / args.steps,
               "ms_per_step": float(ms2.item()) / args.steps,
               "api": "librd_host.so model_t::compute_lh + model_t::suggest_roots_lh sweep (host scheduler, "
                      "programs H2D, log-likelihoods D2H; alignment resident as in the reference partition"
                      + ("; + all-gather of the placement log-likelihoods)" if G_r > 1 else ")"),
               "logl_root0": a, "matches_device_arm": bool(a == lh0 and np.array_equal(b, sweep_lh)),
               "placements_sha256": placements_digest(b)}
        if args.exhaustive_branches > 0:
            e2e["exhaustive"] = exhaustive_sample(m, args.exhaustive_branches, stats=mstats, taxa=n, barrier=barrier)
        m.close()
    clocks = sampler.stop() if sampler else None

    cpu = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        _, cpu, _ = cpu_reference_run(args, case, steps=3, warmup=1, threads=threads, target_step_s=3.0)
        cpu["single_thread"] = cpu_single_thread(args, case)

    g.close()
    north_star = None
    ns = args.north_star
    if ns == "auto":
        ns = "all" if world == 8 else "off"
    if ns != "off":
        import bench_northstar as bn
        names = list(bn.CONFIGS) if ns == "all" else [x for x in ns.split(",") if x]
        north_star = {}
        for name in names:
            cfg = bn.scaled(bn.CONFIGS[name], args.ns_scale)
            try:
                res = bn.run_config(name, cfg, torch=torch, dist=dist, rank=rank, world=world, local=local,
                                    peak_gbs=peak, exhaustive_branches=args.ns_exhaustive_branches if name == "cfg3" else 0,
                                    exhaustive_iterations=args.ns_exhaustive_iterations,
                                    log=(lambda *a: print("[north_star]", *a, file=sys.stderr, flush=True)) if rank == 0
                                    else (lambda *a: None))
            except Exception as exc:  # a failed extra must not take the headline line with it
                res = {"error": "%s: %s" % (type(exc).__name__, exc)}
            if world > 1:
                # every rank learns whether ANY rank failed this extra (an error raised on all ranks alike --
                # the usual kind -- leaves the job in step, and the next extra and the headline line go on)
                failed = isinstance(res, dict) and "error" in res
                flag = torch.tensor([1.0 if failed else 0.0], device="cuda")
                dist.all_reduce(flag, op=dist.ReduceOp.MAX)
                if flag.item() > 0 and not failed:
                    res = {"error": "failed on another rank"}
            torch.cuda.empty_cache()
            if rank == 0:
                north_star[name] = res

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(workload_config(args, placements, (G_s, G_r)), sweep=(
                "directed-CLV pre-order pass (1 CLV op + 1 root evaluation per placement; same bits as the "
                "reference's loop)" if args.sweep == "directed" else
                "reference-shaped: move_root path ops + root op per placement, one engine call"),
                sweep_chunks=n_chunks,
                clv_ops_per_step=st["clv_ops"] / args.steps, root_evals_per_step=st["root_evals"] / args.steps),
            "clv_update_gbs": clv_gbs, "clv_update_gbs_per_gpu": clv_gbs / n_gpus,
            "algorithmic_bytes_per_step": total_alg_bytes / args.steps,
            "roofline": roofline, "full_evaluation": full_eval, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": int(agg[1].item()), "clocks": clocks,
            "logl_root0": lh0, "best_placement": int(np.argmax(sweep_lh)),
            # SHA-256 of the bit patterns of all 2n-3 placement log-likelihoods: must be the same string in the
            # N = 1, 2, 4, 8 lines (site shards add exact zeros: DESIGN section 3) and in the e2e arm
            "placements_sha256": placements_digest(sweep_lh),
            # the sweep scores root 0 at ratio 0.5 too: same bits as the full evaluation (the reference's
            # compute_lh == compute_lh_root invariant) -- also a cross-rank check that every shard walked
            # the placements in the same order
            "sweep_root0_equals_full_evaluation": bool(sweep_lh[0] == lh0),
        }
        if north_star is not None:
            line["north_star"] = north_star
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def exhaustive_sample(m, branches: int, tol=(1e-7, 1e-7, 1e-12, 1e4), stats=None, taxa=0, barrier=lambda: None):
    """exhaustive mode (reference src/model.cpp:1140-1235) on a bounded sample: the first `branches`
    root ids, each optimised to convergence (BFGS over rates / frequencies / Gamma shape + Brent on the
    root position), timed by wall clock.  stats: optional callable returning the engine's counters.
    Returns branches/s, full evaluations/s (the unit BFGS is made of: 13 per step on the 12 rates,
    src/model.cpp:1488-1502) and the latency of compute_dlh (2 root-only evaluations, :481-519: the unit
    of the alpha loop).  Site-sharded runs call this on every rank (each evaluation all-reduces)."""
    branches = max(1, min(int(branches), m.root_count))
    num_tasks = max(1, -(-m.root_count // branches))  # rank 0 of that many tasks gets <= `branches` ids
    s0 = stats() if stats else None
    barrier()
    t0 = time.perf_counter()
    ids, llh, alpha = m.exhaustive_search(*tol, rank=0, num_tasks=num_tasks)
    barrier()
    dt = time.perf_counter() - t0
    out = {"branches": int(len(ids)), "seconds": dt, "branches_per_sec": len(ids) / dt if dt > 0 else None,
           "best_branch": int(ids[int(np.argmax(llh))]), "best_llh": float(np.max(llh)),
           "tolerances": "atol 1e-7, pgtol 1e-7, brtol 1e-12, factor 1e4"}
    if s0 is not None:
        s1 = stats()
        ev = s1["root_evals"] - s0["root_evals"]
        full = (s1["clv_ops"] - s0["clv_ops"]) // max(1, taxa - 1) if taxa else None
        out.update(root_evaluations=int(ev), evaluations_per_sec=ev / dt if dt > 0 else None,
                   full_traversals=full, full_evaluations_per_sec=(full / dt if full and dt > 0 else None))
    # the alpha loop (H3): latency of one slope (compute_dlh = 2 root-only evaluations) and of one
    # optimize_alpha, with the evaluations handed to the engine as fused batches (the default,
    # DESIGN 5.5) and one by one as the reference issues them; same values either way
    reps = 50
    was = m.batched_probes
    for batched, key in ((True, "us_per_compute_dlh"), (False, "us_per_compute_dlh_unbatched")):
        m.set_batched_probes(batched)
        barrier()
        t1 = time.perf_counter()
        for i in range(reps):
            m.compute_dlh(int(ids[0]), 0.25 + 0.01 * i)
        barrier()
        out[key] = (time.perf_counter() - t1) / reps * 1e6
    alphas = {}
    try:  # (every rank sees the same values, so a failure here is a failure on all ranks at the same call)
        for batched, key in ((True, "us_per_optimize_alpha"), (False, "us_per_optimize_alpha_unbatched")):
            m.set_batched_probes(batched)
            alphas[key], spent = [], 0.0
            for r in ids[:4]:
                m.compute_lh(int(r), 0.5)  # CLVs oriented towards this branch (not timed)
                barrier()
                t1 = time.perf_counter()
                alphas[key].append(m.optimize_alpha(int(r), 0.5, 1e-12))
                barrier()
                spent += time.perf_counter() - t1
            out[key] = spent / max(1, len(alphas[key])) * 1e6
        out["optimize_alpha_same_bits"] = bool(
            np.array_equal(np.array(alphas["us_per_optimize_alpha"]).view(np.uint64),
                           np.array(alphas["us_per_optimize_alpha_unbatched"]).view(np.uint64)))
    except RuntimeError as exc:  # a measurement extra must not take the line with it
        out["optimize_alpha_error"] = str(exc)
    m.set_batched_probes(was)
    out["root_only_evaluations"] = m.probe_counters()  # fused batches / evaluations in them / issued singly
    return out


def dram_traffic_from_profiles(taxa, sites_per_gpu, cats):
    """measured DRAM bytes of the program-kernel launches of one step for THIS per-GPU configuration, from
    the committed ncu --set full summaries (profiles/clv_program_traffic.json); None when that
    configuration was never profiled -- a number measured on another shape is not reported"""
    p = ROOT / "profiles" / "clv_program_traffic.json"
    try:
        return json.loads(p.read_text())["entries"].get("%dx%dx%d" % (taxa, sites_per_gpu, cats))
    except Exception:
        return None


def placements_digest(values) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(values, dtype="<f8").tobytes()).hexdigest()


def min_step_traffic(n, sites, K):
    """bytes one step cannot avoid moving through HBM (SURVEY 8d sizes): the full evaluation writes every
    inner CLV once and reads the tips; the directed sweep reads every inner CLV once (as the sibling of
    the placement next to it -- the directed CLVs it derives can live in L2 / registers) and the tips"""
    clv = 32 * K * sites
    return (n - 1) * clv + n * sites + (n - 2) * clv + n * sites


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
