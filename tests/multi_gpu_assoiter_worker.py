"""Worker of tests/test_multigpu_assoiter_gpu.py (one process per GPU, NCCL): AssoIter.fit() and AssoOpt.optimal_rows()
with the rows of X sharded over the ranks must give, on EVERY rank, the results of one process: golden vectors of the
genuine reference, the c3 and iter_scale fixtures of the C restatement, device-generated input against the full csr,
val / test counts against the numpy restatement, and the IndexError after a D1 truncation without a hang.
Usage: torchrun --nproc-per-node N tests/multi_gpu_assoiter_worker.py"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

from conftest import GOLDEN, load_golden
from oracle import asso_oracle as O
from pybmf_b200 import generate, models, synth
from pybmf_b200.engine import ShardPlan

rank, world, local = (int(os.environ[v]) for v in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
models.SILENT = True
KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)


def dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def u_hash(U):
    h = hashlib.sha256()
    for c in range(U.shape[1]):
        h.update(np.packbits(U[:, c], bitorder="little").tobytes())
    return h.hexdigest()


def refinements(it):
    if "refinements" not in it.logs:
        return []
    df = it.logs["refinements"]
    return [(int(a), float(b), float(c)) for a, b, c in zip(df.iloc[:, 1], df[("train", 0, "score")], df[("train", 0, "error")])]


# golden vectors of the genuine reference; planted_w02 / planted_w025 have 240 rows, so at world 2 rank 1 owns none
for name in ("ex01_6", "c1_noisy", "planted_w02", "planted_w025"):
    c = load_golden(name)
    g = c["g"]
    mdl = models.Asso(tau=c["tau"], k=c["k"], w_fp=c["w_fp"], w_fn=c["w_fn"])
    mdl.fit(sp.csr_matrix(c["X"]), **KW)
    it = models.AssoIter(model=mdl, w_fp=c["w_fp"], w_fn=c["w_fn"])
    it.fit(sp.csr_matrix(c["X"]), **KW)
    assert it.U is mdl.U and np.array_equal(dense(it.U), g["iter_U"]), (name, rank)
    assert [r[0] for r in refinements(it)] == [int(r) for r, a in g["iter_trace"] if a == 1], (name, rank)
    assert [r[2] for r in refinements(it)] == [float(v) for v in g["iter_error"]][: len(refinements(it))], (name, rank)
assert ShardPlan(240, world).rows(world - 1)[0] == 240 or world == 1

# the D1 truncation leaves k > U.shape[1]: every rank raises IndexError before any collective
c = load_golden("c1_clean")
mdl = models.Asso(tau=c["tau"], k=c["k"], w_fp=c["w_fp"], w_fn=c["w_fn"])
mdl.fit(sp.csr_matrix(c["X"]), **KW)
try:
    models.AssoIter(model=mdl, w_fp=0.5).fit(sp.csr_matrix(c["X"]), **KW)
    raise SystemExit("AssoIter should have raised IndexError")
except IndexError:
    pass
dist.barrier()

# BASELINE configs[2] (c3) and the iter_scale fixture (accepts a column, stops mid-sweep) of the C restatement
for fixture, make in (("c3", lambda d: (synth.config_c2(), 0.5, 20, 0.5)),
                      ("iter_scale", lambda d: (synth.planted(*d["planted"]), d["tau"], d["k"], d["w_fp"]))):
    with open(os.path.join(GOLDEN, fixture + "_digest.json")) as fh:
        want = json.load(fh)
    X, tau, k, w_fp = make(want)
    mdl = models.Asso(tau=tau, k=k, w_fp=w_fp)
    mdl.fit(X, **KW)
    it = models.AssoIter(model=mdl, w_fp=w_fp)
    it.fit(X, **KW)
    U = dense(it.U)
    assert u_hash(U) == want["u_sha256"] and int(U.sum()) == want["u_ones"], (fixture, rank)
    rows = refinements(it)
    assert [r[0] for r in rows] == [c_ for c_, a in want["trace"] if a], (fixture, rank)
    assert [np.float64(r[1]).tobytes().hex() for r in rows] == want["score_bits"], (fixture, rank)
    assert [np.float64(r[2]).tobytes().hex() for r in rows] == want["error_bits"], (fixture, rank)

# an input generated ON the devices (every rank only its own rows) against the same matrix as a host csr
Xd = generate.planted_bits(3000, 900, 6, 0.2, 0.2, 0.3, 0.05, seed=5)
Xfull = generate.planted_bits(3000, 900, 6, 0.2, 0.2, 0.3, 0.05, seed=5, rank=0, world=1).to_csr()
got = []
for X in (Xd, Xfull):
    mdl = models.Asso(tau=0.35, k=6, w_fp=0.5)
    mdl.fit(X, **KW)
    U0, V0 = dense(mdl.U), dense(mdl.V)
    it = models.AssoIter(model=mdl, w_fp=0.5)
    it.fit(X, **KW)
    opt = models.AssoOpt(model=mdl, w_fp=0.5, w_fn=0.5)
    opt.load_dataset(X_train=X)
    best, score = opt.optimal_rows()
    got.append((dense(it.U), refinements(it), best, score))
ref = O.asso_iter_fit(Xfull, U0, V0, 6, 0.5)
for a, b in zip(*got):
    assert np.array_equal(np.asarray(a), np.asarray(b)), rank
assert np.array_equal(got[0][0], ref["U"]), rank
assert got[0][1] == [(r["k"], r["score"], r["error"]) for r in ref["refinements"]], rank

# AssoOpt: the sharded row search and the U built from it against the reference's golden vectors
g = np.load(os.path.join(GOLDEN, "assoopt.npz"))
for ci in g["cases"]:
    p = "c%d_" % ci
    X = sp.csr_matrix(g[p + "X"])
    k, tau = int(g[p + "k"]), float(g[p + "tau"])
    base = models.Asso(tau=tau, k=k, w_fp=0.5)
    base.fit(X, **KW)
    opt = models.AssoOpt(model=base, w_fp=float(g[p + "w"][0]), w_fn=float(g[p + "w"][1]))
    try:
        opt.fit(X, **KW)
        raise SystemExit("AssoOpt.fit should have raised AttributeError (D4)")
    except AttributeError:
        pass
    bits = ((g[p + "best"][:, None] >> (k - 1 - np.arange(k))[None, :]) & 1).astype(np.uint8)
    assert np.array_equal(dense(opt.U), bits), (ci, rank)

# val / test splits: the logged counts after every accepted column against the numpy restatement of the same run
X = synth.planted(900, 700, 8, 0.15, 0.15, 0.25, 0.03, seed=11)
Xd_ = O.as_dense01(X)
rng = np.random.RandomState(0)
val = sp.csr_matrix(Xd_ * (rng.rand(*Xd_.shape) < 0.2))
mdl = models.Asso(tau=0.35, k=8, w_fp=0.5)
mdl.fit(X, **KW)
U, V = dense(mdl.U), dense(mdl.V)
it = models.AssoIter(model=mdl, w_fp=0.5)
it.fit(X, X_val=val, X_test=val, **KW)
ref = O.asso_iter_fit(X, U, V, 8, 0.5)
assert np.array_equal(dense(it.U), ref["U"]), rank
# replay the oracle's sweeps to get U after each accepted column
Ur, size, want_rows = U.copy(), Xd_.size, []
tr = list(ref["trace"])
while tr:
    for col in range(8):
        if not tr:
            break
        c_, acc = tr.pop(0)
        assert c_ == col
        idx = [i for i in range(8) if i != col]
        _s, u = O.get_vector(Xd_, O.bool_product(Ur[:, idx], V[:, idx]), V[:, col], 0.5, 0.5)
        Ur[:, col] = u
        if acc:
            tp, fp, fn = O.confusion(O.as_dense01(val), O.bool_product(Ur, V))
            want_rows.append(O.rates_from_counts(tp, fp, fn, size))
df = it.logs["refinements"] if want_rows else None
for j, want in enumerate(want_rows):
    for split in ("val", "test"):
        for col in ("Recall", "Precision", "Accuracy", "F1"):
            assert float(df[(split, 0, col)].iloc[j]) == float(want[col]), (split, col, j, rank)
assert len(want_rows) > 0

dist.barrier()
dist.destroy_process_group()
print("rank %d of %d ok" % (rank, world))
