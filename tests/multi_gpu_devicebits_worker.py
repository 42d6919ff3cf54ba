"""Worker of tests/test_multigpu_devicebits_gpu.py (one process per GPU, NCCL): with the rows of generate.DeviceBits
inputs sharded over the ranks, the fits with DeviceBits validation / test splits, the utils counts, generate.transpose and
TransposedModel must give, on EVERY rank, what one process computes on the same matrices as host csr.  One case has
m <= 256, so that at world 2 rank 1 holds no rows.
Usage: torchrun --nproc-per-node N tests/multi_gpu_devicebits_worker.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import pandas as pd
import scipy.sparse as sp
import torch
import torch.distributed as dist

from pybmf_b200 import generate, models, utils
from pybmf_b200.engine import ShardPlan

rank, world, local = (int(os.environ[v]) for v in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
models.SILENT = True
KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)
NAMES = ["TP", "FP", "TN", "FN", "TPR", "FPR", "PPV", "ACC", "ERR", "F1"]


def dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def log(df):
    return df.loc[:, [c for c in df.columns if "time" not in c]]


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.tobytes() == b.tobytes()


def mats(m, n, seeds, sharded):
    kw = {} if sharded else dict(rank=0, world=1)
    out = [generate.planted_bits(m, n, 5, 0.2, 0.15, 0.2, 0.03, seed=s, **kw) for s in seeds]
    return out if sharded else [X.to_csr() for X in out]


def gather_rows(T):
    """All ranks' rows of a DeviceBits as one dense host array (row order), on every rank."""
    parts = [None] * world
    dist.all_gather_object(parts, dense(T.to_csr()) if T.r1 > T.r0 else np.zeros((0, T.n), np.uint8))
    return np.concatenate(parts, axis=0)


for m, n, w in ((1000, 701, 0.5), (1000, 701, 0.2), (200, 333, 0.5)):
    assert m > 256 or ShardPlan(m, world).rows(world - 1)[0] == m or world == 1
    d = mats(m, n, (3, 4, 5, 6), True)
    h = mats(m, n, (3, 4, 5, 6), False)
    k = 4
    # Asso + AssoIter with DeviceBits val / test splits
    fits = []
    for X in (d, h):
        mdl = models.Asso(tau=0.4, k=k, w_fp=w)
        mdl.fit(X[0], X[1], X[2], **KW)
        U0, V0 = dense(mdl.U), dense(mdl.V)
        it = models.AssoIter(model=mdl, w_fp=w)
        it.fit(X[0], X[1], X[2], **KW)
        fits.append((U0, V0, mdl.logs["updates"], dense(it.U), it.logs.get("refinements")))
    assert np.array_equal(fits[0][0], fits[1][0]) and np.array_equal(fits[0][1], fits[1][1]), (m, rank)
    pd.testing.assert_frame_equal(log(fits[0][2]), log(fits[1][2]))
    assert np.array_equal(fits[0][3], fits[1][3]), (m, rank)
    assert (fits[0][4] is None) == (fits[1][4] is None)
    if fits[0][4] is not None:
        pd.testing.assert_frame_equal(log(fits[0][4]), log(fits[1][4]))
    # utils on the sharded matrices (collectives) against the full host matrices
    U, V = sp.lil_matrix(fits[1][0].astype(float)), sp.lil_matrix(fits[1][1].astype(float))
    got = utils.eval(NAMES, "reconstruction", X_gt=d[1], U=U, V=V)
    want = utils.eval(NAMES, "reconstruction", X_gt=h[1], U=U, V=V)
    assert all(same(a, b) for a, b in zip(got, want)), (m, rank)
    assert utils.confusion_counts(d[0], d[3]) == utils.confusion_counts(h[0], h[3]), (m, rank)
    for f in (utils.TP, utils.FN, utils.TN, utils.F1, utils.coverage_score, utils.weighted_error):
        assert same(f(d[0], d[3]), f(h[0], h[3])), (f.__name__, m, rank)
    assert all(same(a, b) for a, b in zip(utils.get_metrics(d[0], d[3], NAMES), utils.get_metrics(h[0], h[3], NAMES)))
    assert same(utils.description_length(d[0], U, V), utils.description_length(h[0], U, V))
    # transpose: rows ShardPlan(n, world) of X^T on every rank, the same bits as one process
    T = generate.transpose(d[0])
    assert (T.m, T.n, (T.r0, T.r1)) == (n, m, ShardPlan(n, world).rows(rank))
    assert np.array_equal(gather_rows(T), dense(h[0]).T), (m, rank)
    assert not T.bits[:, (m + 63) // 64:].any() and (m % 64 == 0 or not (T.bits[:, m // 64] >> (m % 64)).any())
    # TransposedModel on the sharded matrix and a DeviceBits split against the host fit
    got = []
    for X in (d, h):
        tm = models.TransposedModel(models.Asso(tau=0.4, k=3, w_fp=w))
        tm.fit(X[0], X[1], **KW)
        got.append((dense(tm.U), dense(tm.V), tm.model.logs["updates"]))
    assert np.array_equal(got[0][0], got[1][0]) and np.array_equal(got[0][1], got[1][1]), (m, rank)
    pd.testing.assert_frame_equal(log(got[0][2]), log(got[1][2]))

dist.barrier()
dist.destroy_process_group()
print("rank %d of %d ok" % (rank, world))
