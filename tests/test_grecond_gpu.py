"""GPU: pybmf_b200.models.GreConD against the genuine reference run (tests/golden/grecond.npz) from host and device inputs,
the concept kernels (bmf_concept_*) against numpy for every candidate, whole fits against the numpy restatement
(tests/grecond_reference.py) on ragged shapes and at 20000 x 3000, validation / test splits under both tasks, and every
error case."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import GOLDEN
from grecond_reference import grecond, grecond_packed, planted, ragged_cases

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)
METRICS = ("Recall", "Precision", "Accuracy", "F1")


@pytest.fixture(scope="module")
def L():
    from pybmf_b200 import _native, device, generate, models, utils
    _native.require_gpu()
    models.SILENT = True
    return _native, device, generate, models, utils


def _dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def _log(mdl, split, name):
    return np.array([float(v) for v in mdl.logs["updates"][(split, 0, name)]])


@pytest.mark.parametrize("form", ["csr", "ndarray", "device_bits", "device_entries"])
def test_golden_run(L, form):
    _native, device, generate, models, utils = L
    g = np.load(os.path.join(GOLDEN, "grecond.npz"))
    X = {"csr": lambda: sp.csr_matrix(g["X"]), "ndarray": lambda: g["X"],
         "device_bits": lambda: generate.bits_from_host(g["X"]),
         "device_entries": lambda: generate.entries_from_host(sp.csr_matrix(g["X"]))}[form]()
    mdl = models.GreConD(k=6, tol=0)
    mdl.fit(X, **KW)
    assert sp.isspmatrix_lil(mdl.U) and mdl.U.dtype == np.float64 and sp.isspmatrix_lil(mdl.V)
    assert np.array_equal(_dense(mdl.U), g["U"]) and np.array_equal(_dense(mdl.V), g["V"])
    for c in METRICS:
        assert np.array_equal(_log(mdl, "train", c), g["log_" + c]), c
    assert len(mdl.logs["updates"]) == 6
    assert np.array_equal(_dense(mdl.X_pd), g["X_pd"])


def test_available_as_pybmf(L):
    import pybmf_b200
    pybmf_b200.install_as_pybmf(force=True)
    from PyBMF.models import GreConD
    assert GreConD is L[3].GreConD


def _scores(Xc, Rc, C, D, pos):
    """Intent and cover of every candidate j > pos, j not in D, over the rows in C."""
    n = Xc.shape[1]
    out = {}
    for j in range(pos + 1, n):
        if D[j]:
            continue
        Cj = C & Xc[:, j]
        I = Xc[Cj].all(axis=0) if Cj.any() else np.ones(n, bool)
        out[j] = (I, int(Rc[np.ix_(Cj, I)].sum()), int(Cj.sum()))
    return out


@pytest.mark.parametrize("rows,n,pos", [(1, 1, -1), (70, 130, 5), (300, 64, -1), (1000, 700, 200), (4100, 3000, 64),
                                        (257, 2100, 2050)])
def test_round_kernels_score_every_candidate(L, rows, n, pos):
    _native, device, *_ = L
    rng = np.random.default_rng(rows + n)
    X = rng.random((rows, n)) < 0.4
    R = X & (rng.random((rows, n)) < 0.7)
    C = rng.random(rows) < 0.6
    D = np.zeros(n, bool)
    D[rng.choice(n, size=n // 5, replace=False)] = True
    W = device.words_for(n)
    d = device.dev()
    xc, rc = (torch.from_numpy(device.dense_to_words(A, W)).to(d) for A in (X, R))
    c_bits = torch.from_numpy(device.dense_to_words(C[None])[0]).to(d)
    d_bits = torch.from_numpy(device.dense_to_words(D[None], W)[0]).to(d)
    ncw = (n + 63) // 64
    intents = device.zeros((ncw * 64, W), torch.int64)
    covers = device.zeros((ncw * 64,), torch.int64)
    state = torch.tensor([pos, 0, 0, 0], dtype=torch.int64, device=d)
    _native.call("bmf_concept_intents", xc, rows, W, n, c_bits, 0, ncw, 0, state, d_bits, intents, None)
    _native.call("bmf_concept_covers", xc, rc, rows, W, n, c_bits, 0, ncw, 0, state, d_bits, intents, 1, 0, covers)
    want = _scores(X, R, C, D, pos)
    got_i = device.words_to_dense(intents.cpu().numpy(), n)
    got_c = covers.cpu().numpy()
    for j, (I, s, _cnt) in want.items():
        assert got_c[j] == s, j
        assert np.array_equal(got_i[j] != 0, I), j
    assert not got_c[[j for j in range(ncw * 64) if j not in want]].any()
    # the decision: the first candidate whose cover exceeds `best`
    best = int(np.median([s for _i, s, _c in want.values()])) if want else 0
    state = torch.tensor([pos, best, 0, 0], dtype=torch.int64, device=d)
    _native.call("bmf_concept_decide", xc, rows, W, n, covers, intents, state, c_bits, d_bits)
    st = state.cpu().numpy()
    first = [j for j in sorted(want) if want[j][1] > best]
    if first:
        j = first[0]
        assert list(st) == [j, want[j][1], 0, 1]
        assert np.array_equal(device.words_to_dense(d_bits.cpu().numpy()[None], n)[0] != 0, want[j][0])
        assert np.array_equal(device.words_to_dense(c_bits.cpu().numpy()[None], rows)[0] != 0, C & X[:, j])
    else:
        assert st[2] == 1


@pytest.mark.parametrize("m,n,p", [(1, 1, 0), (700, 130, 0), (70000, 300, 70), (5000, 200, 130)])
def test_seed_window_kernels(L, m, n, p):
    """Seed mode: all rows, one column word from col_lo = p, partial intents ANDed over two parts, row counts."""
    _native, device, *_ = L
    rng = np.random.default_rng(m + n)
    X = rng.random((m, n)) < 0.3
    R = X & (rng.random((m, n)) < 0.5)
    W = device.words_for(n)
    d = device.dev()
    cw = p // 64
    h = m // 2
    parts = device.zeros((2, 64 * W + 64), torch.int64)
    halves = [(0, h), (h, m)]
    for q, (a, b) in enumerate(halves):
        xq = torch.from_numpy(device.dense_to_words(X[a:b], W)).to(d) if b > a else device.zeros((1, W), torch.int64)
        _native.call("bmf_concept_intents", xq, b - a, W, n, None, cw, 1, p, None, None, parts[q, :64 * W],
                     parts[q, 64 * W:])
    x, r = (torch.from_numpy(device.dense_to_words(A, W)).to(d) for A in (X, R))
    covers = device.zeros((64,), torch.int64)
    _native.call("bmf_concept_covers", x, r, m, W, n, None, cw, 1, p, None, None, parts, 2, 64 * W + 64, covers)
    got_c, P = covers.cpu().numpy(), parts.cpu().numpy()
    for j in range(64 * cw, min(n, 64 * cw + 64)):
        b = j - 64 * cw
        if j < p:
            assert got_c[b] == 0
            continue
        Cj = X[:, j]
        I = X[Cj].all(axis=0) if Cj.any() else np.ones(n, bool)
        assert got_c[b] == int(R[np.ix_(Cj, I)].sum()), j
        for q, (a, e) in enumerate(halves):
            assert P[q, 64 * W + b] == int(X[a:e, j].sum())


@pytest.mark.parametrize("case", range(9))
def test_fit_against_restatement(L, case):
    _native, device, generate, models, utils = L
    name, X, k = ragged_cases()[case]
    U, V, covers = grecond(X, k)
    for src in (sp.csr_matrix(X), generate.bits_from_host(X)):
        mdl = models.GreConD(k=k)
        mdl.fit(src, **KW)
        assert mdl.U.shape == U.shape and mdl.V.shape == V.shape, name
        assert np.array_equal(_dense(mdl.U), U) and np.array_equal(_dense(mdl.V), V), name
        if covers:
            assert [int(c) for c in mdl.logs["updates"][("train", 0, "cover")]] == covers
        else:
            assert "updates" not in mdl.logs


def test_property_20000_by_3000(L):
    _native, device, generate, models, utils = L
    X = planted(20000, 3000, 8, 0.08, 0.004, 99)
    U, V, covers = grecond_packed(X, 12)
    mdl = models.GreConD(k=12)
    mdl.fit(generate.bits_from_host(X), **KW)
    assert np.array_equal(_dense(mdl.U), U) and np.array_equal(_dense(mdl.V), V)
    assert [int(c) for c in mdl.logs["updates"][("train", 0, "cover")]] == covers


def _counts(G, Z, P):
    """(TP, FP, FN) of the prediction P over stored ones G and stored zeros Z (Z None: reconstruction over all cells)."""
    tp = int((G & P).sum())
    fp = int(((~G) & P).sum()) if Z is None else int((Z & P).sum())
    return tp, fp, int(G.sum()) - tp


def test_splits_reconstruction(L):
    _native, device, generate, models, utils = L
    X = planted(400, 300, 4, 0.2, 0.03, 21)
    rng = np.random.default_rng(3)
    Xv, Xt = (X & (rng.random(X.shape) < 0.5)).astype(np.uint8), (X | (rng.random(X.shape) < 0.01)).astype(np.uint8)
    U, V, _c = grecond(X, 5)
    for a, b, c in ((X, Xv, Xt), tuple(generate.bits_from_host(M) for M in (X, Xv, Xt))):
        mdl = models.GreConD(k=5)
        mdl.fit(a, b, c, **KW)
        assert np.array_equal(_dense(mdl.U), U) and np.array_equal(_dense(mdl.V), V)
        for split, G in (("val", Xv), ("test", Xt)):
            for t in range(5):
                P = (U[:, : t + 1].astype(np.int64) @ V[:, : t + 1].T.astype(np.int64)) > 0
                tp, fp, fn = _counts(G != 0, None, P)
                assert _log(mdl, split, "Precision")[t] == np.float64(tp) / np.float64(tp + fp)
                assert _log(mdl, split, "Recall")[t] == np.float64(tp) / np.float64(tp + fn)


def test_prediction_task_with_device_entries(L):
    _native, device, generate, models, utils = L
    X = planted(500, 260, 4, 0.2, 0.03, 31)
    tr, va, te = generate.ratio_split(generate.bits_from_host(X), 0.2, 0.1, seed=5)
    ones = _dense(tr.to_csr())
    U, V, _c = grecond(ones, 4)
    # trained on a DeviceEntries: its ones
    train = generate.DeviceEntries(tr, generate.DeviceBits(torch.zeros_like(tr.bits), tr.m, tr.n, tr.r0, tr.r1))
    mdl = models.GreConD(k=4)
    mdl.fit(train, va, te, **dict(KW, task="prediction"))
    assert np.array_equal(_dense(mdl.U), U) and np.array_equal(_dense(mdl.V), V)
    for split, E in (("val", va), ("test", te)):
        G, Z = _dense(E.ones.to_csr()) != 0, _dense(E.zeros.to_csr()) != 0
        for t in range(U.shape[1]):
            P = (U[:, : t + 1].astype(np.int64) @ V[:, : t + 1].T.astype(np.int64)) > 0
            tp, fp, fn = _counts(G, Z, P)
            assert _log(mdl, split, "Recall")[t] == np.float64(tp) / np.float64(tp + fn)
            if tp + fp:
                assert _log(mdl, split, "Precision")[t] == np.float64(tp) / np.float64(tp + fp)


def test_errors(L):
    _native, device, generate, models, utils = L
    X = planted(100, 80, 3, 0.3, 0.02, 1)
    with pytest.raises(NotImplementedError):
        models.GreConD(k=2, tol=0.5)
    with pytest.raises(NotImplementedError):
        models.GreConD(k=2).fit(X, tol=0.5, **KW)
    for k in (0, -2, 2.5):
        with pytest.raises(ValueError):
            models.GreConD(k=k)
    B = generate.bits_from_host(X)
    wrong = generate.DeviceBits(B.bits, B.m, B.n, 0, 64)
    with pytest.raises(ValueError):
        models.GreConD(k=2).fit(wrong, **KW)
    with pytest.raises(ValueError):
        models.GreConD(k=2).fit(B, generate.bits_from_host(X[:50]), **KW)
    with pytest.raises(ValueError):                                    # a DeviceBits split under 'prediction'
        models.GreConD(k=2).fit(B, B, **dict(KW, task="prediction"))
    with pytest.raises(TypeError):
        models.GreConD(k=2).fit(None, **KW)
    W = device.words_for(80)
    buf = device.zeros((64, W), torch.int64)
    with pytest.raises(ValueError):                                    # column words past the row
        _native.call("bmf_concept_intents", B.bits, 100, W, 80, None, W, 1, 0, None, None, buf, None)
    with pytest.raises(ValueError):
        _native.call("bmf_concept_covers", B.bits, B.bits, 100, W, 80, None, 0, 1, 0, None, None, buf, 0, 0, buf)
    with pytest.raises(ValueError):
        _native.call("bmf_concept_decide", None, 1, W, 80, buf, buf, buf, buf, buf)
    with pytest.raises(ValueError):
        _native.call("bmf_concept_extent", B.bits, B.bits, 100, W, 0, 64 * W, 1, buf, buf, buf, buf)
    with pytest.raises(ValueError):
        _native.call("bmf_concept_residual", B.bits, 5, 4, W, buf, 1, buf, buf)
