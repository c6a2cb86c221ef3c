"""Row-partitioned mode (K10): slices of W^T on several GPUs with a per-iteration NCCL allGather, against the oracle.
Needs >= 2 GPUs (skipped on a single-GPU box; `gpurun --gpus 2 -- python -m pytest tests -m gpu -k partitioned`)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

import recommendersystems_b200 as rs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_single_rank_communicator_degenerates_to_the_whole_graph():
    """n_ranks == 1: NCCL is bound and initialised, the slice is the whole graph, results equal the plain path."""
    import numpy as np
    # torch first, as in every process that creates a Comm: the library dlopens "libnccl.so.2" with RTLD_GLOBAL, and an older
    # system NCCL loaded first would be bound by torch's libtorch_cuda.so too when a later test of this process imports torch
    import torch  # noqa: F401
    from recommendersystems_b200.rwr import run_fixed
    comm = rs.Comm(0, 1, rs.Comm.unique_id(), device=0)
    spec = dict(seed=3, n_users=500, n_items=4000, n_third=50, authorship_per_mille=800, n_like=15000, n_friend=3000,
                n_follow=100, n_mention=0, undefined_per_mille=10, scramble=1, p1_byte=61)
    gp = rs.Graph.synthetic(spec, comm=comm)
    gp.buildGraph()
    g = rs.Graph.synthetic(spec)
    g.buildGraph()
    i = gp.info()
    assert (i.row_begin, i.row_end, i.n_ranks) == (0, i.n_nodes, 1)
    seed = int(np.flatnonzero(g.degrees(raw=True) > 2)[0])
    a = run_fixed(gp, [seed], rs.widen_float(0.15), 8)
    b = run_fixed(g, [seed], rs.widen_float(0.15), 8)
    assert np.array_equal(a.scores(0), b.scores(0))
    a.close(); b.close(); gp.close(); g.close(); comm.close()


MODES = {
    "overlapped": {"RWR_DIST_OVERLAP": "1"},           # copy-engine pushes overlapped with the next SpMV (default from 3 ranks on)
    "overlapped_slow": {"RWR_DIST_OVERLAP": "1", "RWR_DIST_PUSH_DELAY": "2000"},   # the slices arrive 2 ms late: every gather must wait
    "peer_stores": {},                                  # two ranks: the epilogue kernel stores the slice into the peer's vector
    "replicated_build": {"RWR_PART_REPLICATED": "1"},  # every rank builds the whole graph and keeps its slice (round 1)
    "nccl": {"RWR_DIST_NO_P2P": "1"},                  # grouped ncclBroadcast of the slices
    "peer_stores_blocked": {"RWR_DIST_LEGACY": "1", "RWR_X_BLOCKS": "3"},   # padded column blocks on a slice
}


@pytest.mark.parametrize("mode", list(MODES))
def test_two_ranks_match_the_oracle(mode):
    """Two ranks, every exchange path, against the CPU oracle (FP64 1e-12, FP32, threshold iteration counts, top-10)."""
    if rs._native.lib().rwr_device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(29611 + list(MODES).index(mode)), os.path.join(ROOT, "tests", "partitioned_worker.py"), mode]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=dict(os.environ, **MODES[mode]))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("PARTITIONED OK") == 2
