"""Worker of tests/test_multigpu_residual_gpu.py (one process per GPU, NCCL): with row-sharded inputs, every rank's rows of
generate.prediction and of utils.get_residual on a generate.DeviceBits equal the matching rows of the world-1 result, and
the metrics of a genuine GreConD run (tests/golden/grecond.npz) replayed on the device hold on every rank.  One case has
m <= 256, so that at world 2 rank 1 holds no rows.
Usage: torchrun --nproc-per-node N tests/multi_gpu_residual_worker.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

from pybmf_b200 import generate, utils
from pybmf_b200.engine import ShardPlan

rank, world, local = (int(os.environ[v]) for v in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))


def dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


for m, n, k in ((1000, 701, 5), (3000, 130, 70), (200, 333, 4)):
    assert m > 256 or ShardPlan(m, world).rows(world - 1)[0] == m or world == 1
    rng = np.random.default_rng(m + n + k)
    X = (rng.random((m, n)) < 0.3).astype(np.int64)
    U = sp.lil_matrix((rng.random((m, k)) < 2.0 / k).astype(float))
    V = sp.lil_matrix((rng.random((n, k)) < 0.1).astype(float))
    r0, r1 = ShardPlan(m, world).rows(rank)
    P = generate.prediction(U, V)
    R = utils.get_residual(generate.bits_from_host(X), U, V)
    want_p = dense(utils.get_prediction(U, V))
    want_r = dense(utils.get_residual(X, U, V))
    for S, want in ((P, want_p), (R, want_r)):
        assert (S.m, S.n, S.r0, S.r1) == (m, n, r0, r1), (m, rank)
        if r1 > r0:
            assert np.array_equal(dense(S.to_csr()), want[r0:r1]), (m, rank)

g = np.load(os.path.join(ROOT, "tests", "golden", "grecond.npz"))
X = generate.bits_from_host(g["X"])
U, V = sp.lil_matrix(g["U"].astype(float)), sp.lil_matrix(g["V"].astype(float))
for t in range(g["U"].shape[1]):
    Ut, Vt = sp.lil_matrix(U[:, : t + 1]), sp.lil_matrix(V[:, : t + 1])
    X_pd = generate.prediction(Ut, Vt)
    X_rs = utils.get_residual(X, Ut, Vt)
    assert float(utils.ERR(gt=X, pd=X_pd)) == g["step_ERR"][t]
    assert float(utils.weighted_error(gt=X, pd=X_pd, w_fp=0.3, w_fn=0.7)) == g["step_weighted_error"][t]
    assert float(utils.description_length(gt=X, U=Ut, V=Vt, w_model=1.0, w_fp=1.0, w_fn=1.0)) == g["step_desc_len"][t]
    assert float(utils.coverage_score(gt=X, pd=X_pd, w_fp=0.5)) == g["step_coverage"][t]
    assert utils.confusion_counts(X_rs, X_rs)[0] == int(g["step_rs_sum"][t])
    assert utils.confusion_counts(X_pd, X_pd)[0] == int(g["step_pd_sum"][t])
    got = utils.get_metrics(gt=X, pd=X_pd, metrics=["Recall", "Precision", "Accuracy", "F1"])
    assert [float(v) for v in got] == [float(g["log_" + c][t]) for c in ("Recall", "Precision", "Accuracy", "F1")]

dist.barrier()
dist.destroy_process_group()
print("rank %d of %d ok" % (rank, world))
