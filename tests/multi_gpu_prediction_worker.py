"""Worker of tests/test_multigpu_prediction_gpu.py (one process per GPU, NCCL): with row-sharded inputs, every rank's
rows of generate.ratio_split equal those of the world-1 split, a fit with DeviceEntries splits gives the world-1 logs on
every rank, and a DeviceBits X_train under task='prediction' fits like a host csr of its ones.  One case has m <= 256,
so that at world 2 rank 1 holds no rows.
Usage: torchrun --nproc-per-node N tests/multi_gpu_prediction_worker.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import pandas as pd
import scipy.sparse as sp
import torch
import torch.distributed as dist

from pybmf_b200 import generate, models, utils
from pybmf_b200.engine import ShardPlan
from split_reference import ratio_split_rows, stored_csr

rank, world, local = (int(os.environ[v]) for v in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
models.SILENT = True
KW = dict(task="prediction", save_model=False, show_logs=False, show_result=False)
NAMES = ["TP", "FP", "TN", "FN", "PPV", "ACC", "ERR", "F1"]


def dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def log(df):
    return df.loc[:, [c for c in df.columns if "time" not in c]]


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.tobytes() == b.tobytes()


def fit(X, w):
    mdl = models.Asso(tau=0.4, k=4, w_fp=w)
    mdl.fit(X[0], X[1], X[2], **KW)
    U0, V0 = dense(mdl.U), dense(mdl.V)
    it = models.AssoIter(model=mdl, w_fp=w)
    it.fit(X[0], X[1], X[2], **KW)
    return U0, V0, mdl.logs["updates"], dense(it.U), it.logs.get("refinements")


for m, n, w in ((1000, 701, 0.5), (1000, 701, 0.2), (200, 333, 0.5)):
    assert m > 256 or ShardPlan(m, world).rows(world - 1)[0] == m or world == 1
    Xs = generate.planted_bits(m, n, 5, 0.2, 0.15, 0.2, 0.03, seed=3)                      # this rank's rows
    X1 = generate.planted_bits(m, n, 5, 0.2, 0.15, 0.2, 0.03, seed=3, rank=0, world=1)     # all rows, one process
    d = generate.ratio_split(Xs, 0.1, 0.15, neg_ratio=1.0, seed=7)
    r0, r1 = ShardPlan(m, world).rows(rank)
    x = dense(X1.to_csr())
    th = generate.split_thresholds(int(x.sum()), m, n, 0.1, 0.15, 1.0)
    want = ratio_split_rows(x[r0:r1], r0, n, 7, th)
    got = [d[0], d[1].ones, d[1].zeros, d[2].ones, d[2].zeros]
    for g, wnt in zip(got, want):
        assert (g.r0, g.r1) == (r0, r1)
        if r1 > r0:
            assert np.array_equal(dense(g.to_csr()).astype(bool), wnt), (m, rank)
    # the world-1 split as host csr (stored zeros explicit) is the reference of the sharded fit
    full = [None] * world
    dist.all_gather_object(full, list(want))
    cat = [np.concatenate([f[i] for f in full], axis=0) for i in range(5)]
    h = [sp.csr_matrix(cat[0].astype(np.int64)), stored_csr(cat[1], cat[2]), stored_csr(cat[3], cat[4])]
    a, b = fit(d, w), fit(h, w)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[3], b[3]), (m, rank)
    pd.testing.assert_frame_equal(log(a[2]), log(b[2]))
    assert (a[4] is None) == (b[4] is None)
    if a[4] is not None:
        pd.testing.assert_frame_equal(log(a[4]), log(b[4]))
    U, V = sp.lil_matrix(b[0].astype(float)), sp.lil_matrix(b[1].astype(float))
    for task in ("prediction", "reconstruction"):
        g_ = utils.eval(NAMES, task, X_gt=d[1], U=U, V=V)
        w_ = utils.eval(NAMES, task, X_gt=h[1], U=U, V=V)
        assert all(same(p, q) for p, q in zip(g_, w_)), (task, m, rank)

dist.barrier()
dist.destroy_process_group()
print("rank %d of %d ok" % (rank, world))
