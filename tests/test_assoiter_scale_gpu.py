"""GPU: the one-pass AssoIter sweep (bmf_refine_sweep) against successive bmf_refine_column launches and the numpy
restatement, AssoIter / AssoOpt on device-generated inputs, and AssoIter at a scale above c3 where it accepts a column
and stops in the middle of a sweep (fixture: oracle/make_iter_digest.py)."""
import hashlib
import io
import json
import os
from contextlib import redirect_stdout

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from conftest import GOLDEN  # noqa: E402
from oracle import asso_oracle as O  # noqa: E402

FIT_KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)


@pytest.fixture(scope="module")
def M():
    from pybmf_b200 import _native, models
    _native.require_gpu()
    models.SILENT = True
    return models


def _dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def _sweep_inputs(seed, m, n, k):
    rng = np.random.RandomState(seed)
    X = (rng.rand(m, n) < 0.3).astype(np.uint8)
    U = (rng.rand(m, k) < 0.3).astype(np.uint8)
    V = (rng.rand(n, k) < 0.2).astype(np.uint8)
    U[0::7] = 0                                                    # rows using no factor
    U[3::11] = 1                                                   # rows using all of them
    return X, U, V


@pytest.mark.parametrize("m,n,k", [(1, 1, 1), (37, 63, 5), (300, 64, 5), (513, 65, 64), (2000, 190, 70), (700, 4100, 5),
                                   (3000, 190, 64), (64, 4100, 70)])
@pytest.mark.parametrize("w", [(0.5, 0.5), (0.2, 0.8), (0.25, 0.75)])
def test_refine_sweep_equals_successive_columns_and_numpy(M, m, n, k, w):
    from pybmf_b200 import _native, device
    w_fp, w_fn = w
    iw = O.integer_weights(w_fp, w_fn)
    wa, wb = (iw[0], iw[1]) if iw else (0, 0)
    X, U, V = _sweep_inputs(m * 7 + n + k, m, n, k)
    words = device.words_for(n)
    kw = (k + 63) // 64
    xb = torch.from_numpy(device.dense_to_words(X, words)).cuda()
    vt = torch.from_numpy(device.dense_to_words(V.T, words)).cuda()
    u0 = torch.from_numpy(device.dense_to_words(U, kw)).cuda()
    for col0, ncols in ((0, k), (k // 3, max(1, k // 2)), (k - 1, 1)):
        uw_s, uw_c = u0.clone(), u0.clone()
        out = device.zeros((ncols, 5), torch.int64)
        _native.call("bmf_refine_sweep", xb, m, n, words, uw_s, kw, vt, k, col0, ncols, wa, wb, w_fp, w_fn, out)
        per_col = device.zeros((ncols, 5), torch.int64)
        for j in range(ncols):
            _native.call("bmf_refine_column", xb, m, n, words, uw_c, kw, vt, k, col0 + j, wa, wb, w_fp, w_fn, per_col[j])
        assert torch.equal(uw_s, uw_c), (col0, ncols)
        assert torch.equal(out, per_col), (col0, ncols)
        # the independent reference: AssoIter.get_refined_column column by column in numpy
        Ur = U.copy()
        want = np.zeros((ncols, 5), np.int64)
        for j in range(ncols):
            c = col0 + j
            idx = [i for i in range(k) if i != c]
            C_old = O.bool_product(Ur[:, idx], V[:, idx])
            _s, use, P, N, _t, _f = O.score_candidates(X, C_old, V[:, c].reshape(1, -1), w_fp, w_fn)
            u = use[:, 0]
            Ur[:, c] = u
            tp, fp, _ = O.confusion(X, O.bool_product(Ur, V))
            want[j] = [tp, fp, u.sum(), P[u, 0].sum(), N[u, 0].sum()]
        assert np.array_equal(out.cpu().numpy(), want), (col0, ncols)
        assert np.array_equal(device.words_to_dense(uw_s.cpu().numpy(), k), Ur), (col0, ncols)


def test_refine_sweep_rejects_bad_columns(M):
    from pybmf_b200 import _native, device
    xb = device.zeros((4, 2), torch.int64)
    uw = device.zeros((4, 1), torch.int64)
    vt = device.zeros((5, 2), torch.int64)
    out = device.zeros((5, 5), torch.int64)
    for col0, ncols in ((-1, 2), (0, 0), (3, 3)):
        with pytest.raises(ValueError):
            _native.call("bmf_refine_sweep", xb, 4, 100, 2, uw, 1, vt, 5, col0, ncols, 1, 1, 0.5, 0.5, out)


def _iter_fit_with_trace(M, it, X):
    M.SILENT = False
    buf = io.StringIO()
    try:
        with redirect_stdout(buf):
            it.fit(X, **FIT_KW)
    finally:
        M.SILENT = True
    trace = []
    for line in buf.getvalue().splitlines():
        if "Refined column" in line:
            trace.append((int(line.split("column i:")[1].split(",")[0]), True))
        elif "Skipped column" in line:
            trace.append((int(line.split("column i:")[1].strip(" .")), False))
    return trace


def _refinement_rows(it):
    if "refinements" not in it.logs:
        return []
    df = it.logs["refinements"]
    return [(int(a), float(b), float(c)) for a, b, c in zip(df.iloc[:, 1], df[("train", 0, "score")], df[("train", 0, "error")])]


def test_assoiter_and_assoopt_on_device_bits(M):
    """AssoIter.fit / AssoOpt.optimal_rows on a matrix generated on the device equal the same calls on the matrix
    downloaded to a host csr, and the numpy restatement on that csr."""
    from pybmf_b200 import generate
    Xd = generate.planted_bits(3000, 900, 6, 0.2, 0.2, 0.3, 0.05, seed=5)
    Xh = Xd.to_csr()
    fits = []
    for X in (Xd, Xh):
        mdl = M.Asso(tau=0.35, k=6, w_fp=0.5)
        mdl.fit(X, **FIT_KW)
        U0, V0 = _dense(mdl.U), _dense(mdl.V)
        it = M.AssoIter(model=mdl, w_fp=0.5)
        trace = _iter_fit_with_trace(M, it, X)
        assert it.U is mdl.U
        opt = M.AssoOpt(model=mdl, w_fp=0.5, w_fn=0.5)
        opt.load_dataset(X_train=X)
        best, score = opt.optimal_rows()
        fits.append((U0, V0, _dense(it.U), trace, _refinement_rows(it), best, score, opt.set_optimal_row(2999)))
    a, b = fits
    for x, y in zip(a, b):
        assert np.array_equal(np.asarray(x), np.asarray(y))
    U0, V0, U, trace, rows = a[:5]
    ref = O.asso_iter_fit(Xh, U0, V0, 6, 0.5)
    assert np.array_equal(U, ref["U"])
    assert trace == [(c, bool(t)) for c, t in ref["trace"]]
    assert rows == [(r["k"], r["score"], r["error"]) for r in ref["refinements"]]


def test_assoiter_scale_fixture(M):
    """AssoIter above the c3 scale, where it accepts a column and stops in the middle of the next sweep, against the C
    restatement's fixture: the Asso factors it starts from, the accept / skip trace, score / error bits and U."""
    from pybmf_b200 import synth
    from pybmf_b200.digest import result_digest
    with open(os.path.join(GOLDEN, "iter_scale_digest.json")) as fh:
        want = json.load(fh)
    X = synth.planted(*want["planted"])
    mdl = M.Asso(tau=want["tau"], k=want["k"], w_fp=want["w_fp"])
    mdl.fit(X, **FIT_KW)
    d = result_digest(mdl)
    assert (d["u_sha256"], d["v_sha256"]) == (want["asso_u_sha256"], want["asso_v_sha256"])
    it = M.AssoIter(model=mdl, w_fp=want["w_fp"])
    trace = _iter_fit_with_trace(M, it, X)
    assert [[c, int(a)] for c, a in trace] == want["trace"]
    assert any(a for _c, a in trace) and trace[-1][0] < want["k"] - 1        # accepts, then stops mid-sweep
    U = _dense(it.U)
    h = hashlib.sha256()
    for c in range(U.shape[1]):
        h.update(np.packbits(U[:, c], bitorder="little").tobytes())
    assert h.hexdigest() == want["u_sha256"] and int(U.sum()) == want["u_ones"]
    df = it.logs["refinements"]
    assert [np.float64(v).tobytes().hex() for v in df[("train", 0, "score")]] == want["score_bits"]
    assert [np.float64(v).tobytes().hex() for v in df[("train", 0, "error")]] == want["error_bits"]
