"""Branch support on site shards over NCCL (DESIGN.md section 10, items 9-10): two GPUs, each holding a
shard of the sites -- the planned layout and an unequal one -- must return on every rank the rows (bits),
the positions, log-likelihoods, e, O, every count and lnl_fixed of ONE GPU holding every site.  Skipped
below two devices."""
import os
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu


def test_branch_support_on_site_shards_returns_the_bits_of_one_gpu(tmp_path):
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    sys.path.insert(0, str(ROOT / "tests"))
    import gpu_branch_support_shard_worker as w
    from root_digger_b200 import capi
    from test_branch_support_cpu import search_log

    case = w.base.build_case()
    m = capi.Model(capi.RootedTree(case.newick), case.aln, w.base.K)
    m.initialize_partitions()
    prefix = str(tmp_path / "records")
    search_log(capi.load_tree_lib(), prefix, m, seed=8)
    want = w.result_arrays(m.branch_support(prefix, replicates=w.REPLICATES, seed=w.SEED, keep_rows=True,
                                            au_scales=capi.AU_SCALES), "one")
    rows = m.site_lnl_rows(0)[0]
    m.close()

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "shards")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(ROOT / "tests" / "gpu_branch_support_shard_worker.py"), prefix,
           out]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for rank in (0, 1):
        got = dict(np.load(out + ".rank%d.npz" % rank))
        for tag in w.LAYOUTS:
            off, cnt = got[tag + "_offset"]
            assert got[tag + "_rows"].tobytes() == np.ascontiguousarray(rows[:, off:off + cnt]).tobytes(), (rank, tag)
            for k in w.KEYS + ("O", "scalars"):
                a, b = got[tag + "_" + k], want["one_" + k]
                assert a.shape == b.shape and a.tobytes() == b.tobytes(), (rank, tag, k)
