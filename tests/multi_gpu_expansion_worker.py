"""Worker of tests/test_multigpu_expansion_gpu.py (one process per GPU, NCCL): GreConD+'s expansion and _expansion on
generate.DeviceBits inputs whose rows are sharded over the ranks must give, on EVERY rank, what one process computes on
the same matrices as host csr.  One case has m <= 256, so that at world 2 rank 1 holds no rows.
Usage: torchrun --nproc-per-node N tests/multi_gpu_expansion_worker.py"""
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)
import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

from expansion_reference import planted_case, random_case
from pybmf_b200 import device, expansion, generate, models
from pybmf_b200.engine import ShardPlan

rank, world, local = (int(os.environ[v]) for v in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
models.SILENT = True


def shard(A):
    r0, r1 = ShardPlan(A.shape[0], world).rows(rank)
    bits = torch.from_numpy(device.dense_to_words(A[r0:r1] if r1 > r0 else np.zeros((1, A.shape[1]), np.uint8))).cuda()
    return generate.DeviceBits(bits, A.shape[0], A.shape[1], r0, r1)


# every case adds rows and columns; the rows of the 1000-row cases fall on both ranks
for make, m, n, w, seed in ((random_case, 1000, 701, (0.2, 0.8), 2), (random_case, 1000, 701, (0.3, 0.6), 2),
                            (planted_case, 700, 4100, (0.3, 0.6), 3), (random_case, 200, 333, (0.2, 0.8), 5),
                            (random_case, 200, 333, (0.3, 0.6), 5)):
    assert m > 256 or ShardPlan(m, world).rows(world - 1)[0] == m or world == 1
    X, O, u, v, w_fp, w_fn = make(m, n, *w, seed=seed)
    Xh, Oh = sp.csr_matrix(X), sp.csr_matrix(O)
    Xd, Od = shard(X.astype(np.uint8)), shard(O.astype(np.uint8))
    want = expansion.expansion_log(Xh, Oh, u, v, w_fp, w_fn)               # host inputs: this process alone
    got = expansion.expansion_log(Xd, Od, u, v, w_fp, w_fn)
    assert np.array_equal(got, want), (m, rank, got[:4], want[:4])
    ue, ve = expansion.expansion(Xd, Od, u, v, w_fp, w_fn)
    uh, vh = expansion.expansion(Xh, Oh, u, v, w_fp, w_fn)
    assert (ue != uh).nnz == 0 and (ve != vh).nnz == 0, (m, rank)
    assert (want[:, 0] == 0).any() and (want[:, 0] == 1).any(), m
    for axis in (0, 1):
        a = expansion._expansion(Xd, Od, u, v, w_fp, w_fn, axis)
        b = expansion._expansion(Xh, Oh, u, v, w_fp, w_fn, axis)
        assert a[0].tobytes() == b[0].tobytes() and a[1] == b[1], (m, rank, axis, a, b)
    # the same answer on every rank
    mine = got.tobytes()
    every = [None] * world
    dist.all_gather_object(every, mine)
    assert all(e == mine for e in every), (m, rank)

dist.barrier()
dist.destroy_process_group()
print("rank %d of %d ok" % (rank, world))
