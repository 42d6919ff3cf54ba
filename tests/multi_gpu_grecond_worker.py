"""Worker of tests/test_multigpu_grecond_gpu.py (one process per GPU, NCCL): GreConD fitted on row-sharded inputs (a host
matrix whose rows each rank packs, a generate.DeviceBits, and the genuine reference run of tests/golden/grecond.npz)
gives every rank the factors and train metrics of the numpy restatement, i.e. of world 1.  Cases with m <= 256 leave
rank 1 without rows at world 2.
Usage: torchrun --nproc-per-node N tests/multi_gpu_grecond_worker.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

from grecond_reference import grecond, metrics, planted
from pybmf_b200 import generate, models
from pybmf_b200.engine import ShardPlan

rank, world, local = (int(os.environ[v]) for v in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
models.SILENT = True
KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)


def dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


g = np.load(os.path.join(ROOT, "tests", "golden", "grecond.npz"))
cases = [(g["X"], 6), (planted(1000, 300, 4, 0.2, 0.03, 1), 8), (planted(200, 130, 3, 0.3, 0.02, 2), None),
         (planted(3000, 700, 5, 0.1, 0.01, 3), 10)]
for X, k in cases:
    m = X.shape[0]
    if world == 2 and m <= 256:
        assert ShardPlan(m, world).rows(1)[0] == m                      # rank 1 holds no rows
    U, V, covers = grecond(X, k)
    for src in (sp.csr_matrix(X), generate.bits_from_host(X)):
        mdl = models.GreConD(k=k)
        mdl.fit(src, **KW)
        assert np.array_equal(dense(mdl.U), U) and np.array_equal(dense(mdl.V), V), (m, rank)
        want = metrics(X, covers)
        for i, c in enumerate(("Recall", "Precision", "Accuracy", "F1")):
            got = np.array([float(v) for v in mdl.logs["updates"][("train", 0, c)]])
            assert np.array_equal(got, want[:, i]), (m, c, rank)

dist.barrier()
dist.destroy_process_group()
print("rank %d of %d ok" % (rank, world))
