"""One rank of the 2-GPU run of tests/test_gpu_zz_branch_support_shards.py: branch support on a site
shard per GPU (model_t with a communicator attached), for the shard layouts in LAYOUTS.  Every rank
saves its results and its rows; the test compares them with one GPU holding every site."""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import gpu_multi_worker as base  # noqa: E402  (the 60-taxon x 5000-site case of the NCCL parity run)

REPLICATES, SEED = 300, 0x5EED
# (offset, count) per rank: the planned layout and an unequal one (offsets are multiples of 256)
LAYOUTS = {"planned": None, "unequal": [(0, 1024), (1024, base.SITES - 1024)]}


KEYS = ("root_id", "alpha", "llh", "bp_count", "kh_count", "sh_count", "lnl_fixed", "scale_counts", "elw_fixed")


def result_arrays(res, tag):
    out = {tag + "_" + k: np.asarray(res[k]) for k in KEYS}
    out[tag + "_O"] = np.array([str(v) for v in res["O"]])
    out[tag + "_scalars"] = np.array([res["exponent"], res["best"]])
    return out


def main(ckp_prefix, out_path):
    import torch
    import torch.distributed as dist
    from root_digger_b200 import capi, sharding
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def comm_id():
        ids = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            ids = torch.tensor(list(capi.comm_unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(ids, 0)
        return bytes(ids.cpu().tolist())

    case = base.build_case()
    res = {}
    for tag, layout in LAYOUTS.items():
        off, cnt = (layout or sharding.plan_site_shards(base.SITES, world))[rank]
        aln = {l: s[off:off + cnt] for l, s in case.aln.items()}
        m = capi.Model(capi.RootedTree(case.newick), aln, base.K, site_offset=off, global_sites=base.SITES,
                       nranks=world, rank=rank, comm_id=comm_id())
        m.initialize_partitions()
        got = m.branch_support(ckp_prefix, replicates=REPLICATES, seed=SEED, keep_rows=True, au_scales=capi.AU_SCALES)
        res.update(result_arrays(got, tag))
        res[tag + "_rows"] = m.site_lnl_rows(0)[0]
        res[tag + "_offset"] = np.array([off, cnt])
        m.close()
    np.savez(out_path + ".rank%d.npz" % rank, **res)
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
