"""GPU: the incremental, device-resident GreConD+ expansion (pybmf_b200.expansion.expansion on bmf_expand_init /
bmf_expand_step_rows / bmf_expand_step_decide) and _expansion on generate.DeviceBits inputs, against the genuine
reference's golden vectors and against the numpy restatement of the loop (tests/expansion_reference.py), iteration by
iteration; the init pass's counts against numpy; and every input error."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from conftest import GOLDEN  # noqa: E402
from expansion_reference import (SHAPES, STOP, WEIGHTS, block_case, planted_case, random_case,  # noqa: E402
                                 reference_loop, tie_case)


@pytest.fixture(scope="module")
def E():
    from pybmf_b200 import _native, expansion, models
    _native.require_gpu()
    models.SILENT = True
    return expansion


def _bits(A):
    from pybmf_b200 import device, generate
    A = (np.asarray(A) != 0).astype(np.uint8)
    m, n = A.shape
    return generate.DeviceBits(torch.from_numpy(device.dense_to_words(A)).cuda(), m, n, 0, m)


def _w(arr):
    return float(arr[0]), (None if arr[1] != arr[1] else float(arr[1]))


def _flags(vec):
    return (np.asarray(vec.toarray()).ravel() != 0).astype(np.uint8)


def test_golden_cases_on_device_bits(E):
    g = np.load(os.path.join(GOLDEN, "expansion.npz"))
    for ci in g["cases"]:
        p = "c%d_" % ci
        X, O = _bits(g[p + "X"]), _bits(g[p + "X_old"])
        u, v = sp.lil_matrix(g[p + "u"].reshape(-1, 1)), sp.lil_matrix(g[p + "v"].reshape(-1, 1))
        w_fp, w_fn = _w(g[p + "w"])
        for axis, key in ((1, "row"), (0, "col")):
            score, index = E._expansion(X, O, u, v, w_fp, w_fn, axis=axis)
            assert type(score) is np.float64 and type(index) is int
            want = g[p + key]
            assert np.float64(score).tobytes() == np.float64(want[0]).tobytes() and index == int(want[1]), (ci, axis)
        u_exp, v_exp = E.expansion(X_gt=X, X_old=O, u=u, v=v, w_fp=w_fp, w_fn=w_fn)
        assert sp.isspmatrix_lil(u_exp) and u_exp.shape == (X.m, 1) and v_exp.shape == (X.n, 1)
        assert np.array_equal(_flags(u_exp), g[p + "u_exp"]) and np.array_equal(_flags(v_exp), g[p + "v_exp"]), ci


def _cases():
    out = []
    for (m, n) in SHAPES:
        for (w_fp, w_fn) in WEIGHTS:
            out.append(("planted", m, n, planted_case(m, n, w_fp, w_fn, seed=m + n)))
            out.append(("random", m, n, random_case(m, n, w_fp, w_fn, seed=m * n)))
    for mode in (("empty", "random"), ("all", "random"), ("random", "all")):
        for (m, n) in SHAPES[1:]:
            out.append(("u_%s_v_%s" % mode, m, n, random_case(m, n, 0.3, 0.6, seed=7, u_mode=mode[0], v_mode=mode[1])))
    for rows in (64, 65):                                                      # exactly one stretch, and one more
        out.append(("block%d" % rows, 600, 4100, block_case(600, 4100, rows, 0.5, 0.5, seed=3)))
    return out


CASES = _cases()


@pytest.mark.parametrize("case", CASES, ids=["%s_%dx%d_%d" % (c[0], c[1], c[2], i) for i, c in enumerate(CASES)])
def test_loop_against_numpy_reference_iteration_by_iteration(E, case):
    _name, m, n, (X, O, u, v, w_fp, w_fn) = case
    want = np.array(reference_loop(X, O, u, v, w_fp, w_fn), dtype=np.int64).reshape(-1, 2)
    for inputs in ((sp.csr_matrix(X), sp.csr_matrix(O)), (_bits(X), _bits(O))):
        got = E.expansion_log(*inputs, u.reshape(-1, 1), v.reshape(-1, 1), w_fp, w_fn)
        assert np.array_equal(got, want), (m, n, w_fp, got[:5], want[:5])
        u_exp, v_exp = E.expansion(*inputs, sp.lil_matrix(u.reshape(-1, 1)), sp.lil_matrix(v.reshape(-1, 1)), w_fp, w_fn)
        assert np.array_equal(np.flatnonzero(_flags(u_exp)), np.sort(want[want[:, 0] == 0, 1]))
        assert np.array_equal(np.flatnonzero(_flags(v_exp)), np.sort(want[want[:, 0] == 1, 1]))


def test_run_lengths(E):
    """>= 200 iterations, 64 (one stretch) and 65, and a stop on r_score == c_score > 0."""
    X, O, u, v, w_fp, w_fn = planted_case(33, 1000, 0.2, 0.8, seed=1033)
    assert len(E.expansion_log(_bits(X), _bits(O), u, v, w_fp, w_fn)) >= 200
    for rows in (64, 65):
        X, O, u, v, w_fp, w_fn = block_case(600, 4100, rows, 0.5, 0.5, seed=3)
        got = E.expansion_log(_bits(X), _bits(O), u, v, w_fp, w_fn)
        assert len(got) == rows and got[-1].tolist() == [STOP, -1] and (got[:-1, 0] == 0).all()
    X, O, u, v = tie_case(70, 130)
    r_score, _ = E._expansion(_bits(X), _bits(O), u, v, 0.3, 0.6, axis=1)
    c_score, _ = E._expansion(_bits(X), _bits(O), u, v, 0.3, 0.6, axis=0)
    assert r_score == c_score > 0
    assert E.expansion_log(_bits(X), _bits(O), u, v, 0.3, 0.6).tolist() == [[STOP, -1]]


@pytest.mark.parametrize("m,n,row0", [(1, 1, 0), (70, 130, 0), (257, 65, 256), (33, 1000, 512), (600, 4100, 0),
                                      (5000, 2100, 0), (3000, 4097, 256)])
def test_init_counts_against_numpy(E, m, n, row0):
    """Per-row (TP_old, FP_old, P, N) against v and per-column counts over the rows in u, with pad bits (n % 64 != 0, a
    whole pad word when words * 64 - n >= 64) that ~x & ~old would set; row0 > 0 is a rank's slice of a taller u."""
    from pybmf_b200 import _native, device
    rng = np.random.RandomState(m + n)
    X = (rng.rand(m, n) < 0.3).astype(np.int64)
    O = (rng.rand(m, n) < 0.2).astype(np.int64)
    u_all = (rng.rand(row0 + m + 3) < 0.4).astype(np.int64)
    v = (rng.rand(n) < 0.3).astype(np.int64)
    u = u_all[row0:row0 + m]
    words = device.words_for(n)
    row_cnt = torch.full((m, 4), -7, dtype=torch.int32, device="cuda")
    col_cnt = torch.full((4, n), -7, dtype=torch.int64, device="cuda")
    _native.call("bmf_expand_init", _bits(X).bits, _bits(O).bits, m, n, words, row0,
                 torch.from_numpy(device.dense_to_words(u_all.reshape(1, -1))).cuda(),
                 torch.from_numpy(device.dense_to_words(v.reshape(1, -1))).cuda(), row_cnt, col_cnt)
    pos, neg = X * (1 - O), (1 - X) * (1 - O)
    want_rows = np.stack([(X * O).sum(1), ((1 - X) * O).sum(1), pos @ v, neg @ v], axis=1)
    want_cols = np.stack([(X * O).sum(0), ((1 - X) * O).sum(0), pos.T @ u, neg.T @ u])
    assert np.array_equal(row_cnt.cpu().numpy(), want_rows)
    assert np.array_equal(col_cnt.cpu().numpy(), want_cols)


def test_init_counts_many_rows_per_warp(E):
    """Five million rows: every warp counts the most rows its bit-sliced counters hold between two flushes, with an
    all-ones column reaching the largest count."""
    from pybmf_b200 import _native, device
    m, n = 5_000_000, 3
    rng = np.random.RandomState(0)
    X = (rng.rand(m, n) < 0.5).astype(np.uint8)
    O = (rng.rand(m, n) < 0.3).astype(np.uint8)
    X[:, 0], O[:, 0] = 1, 1
    u = (rng.rand(m) < 0.7).astype(np.uint8)
    def words(A):                                        # three columns: bits 0..2 of the first of two words per row
        w = np.zeros((m, 2), np.int64)
        w[:, 0] = A[:, 0].astype(np.int64) | (A[:, 1].astype(np.int64) << 1) | (A[:, 2].astype(np.int64) << 2)
        return torch.from_numpy(w).cuda()
    xb, ob = words(X), words(O)
    row_cnt = device.zeros((m, 4), torch.int32)
    col_cnt = device.zeros((4, n), torch.int64)
    vb = torch.from_numpy(device.dense_to_words(np.array([[1, 0, 1]]))).cuda()
    _native.call("bmf_expand_init", xb, ob, m, n, device.words_for(n), 0,
                 torch.from_numpy(device.dense_to_words(u.reshape(1, -1))).cuda(), vb, row_cnt, col_cnt)
    X, O, u = X.astype(np.int64), O.astype(np.int64), u.astype(np.int64)
    want = np.stack([(X * O).sum(0), ((1 - X) * O).sum(0), (X * (1 - O) * u[:, None]).sum(0),
                     ((1 - X) * (1 - O) * u[:, None]).sum(0)])
    assert np.array_equal(col_cnt.cpu().numpy(), want)
    rc = row_cnt.cpu().numpy()
    assert np.array_equal(rc[:, 0], (X * O).sum(1)) and np.array_equal(rc[:, 3], ((1 - X) * (1 - O))[:, 2])


def test_input_errors(E):
    from pybmf_b200 import generate
    rng = np.random.RandomState(1)
    X = (rng.rand(300, 70) < 0.3).astype(np.int64)
    u, v = np.zeros(300, np.int64), np.zeros(70, np.int64)
    u[0] = v[0] = 1
    Xd = _bits(X)
    for fn in (lambda *a: E.expansion(*a, 0.5, 0.5), lambda *a: E._expansion(*a, 0.5, 0.5, 1),
               lambda *a: E._expansion(*a, 0.5, 0.5, 0)):
        with pytest.raises(TypeError):
            fn(Xd, sp.csr_matrix(X), u, v)
        with pytest.raises(TypeError):
            fn(sp.csr_matrix(X), Xd, u, v)
        half = generate.DeviceBits(Xd.bits, 300, 70, 0, 256)                 # not the ShardPlan rows of one rank
        with pytest.raises(ValueError):
            fn(half, half, u, v)
        with pytest.raises(ValueError):
            fn(Xd, _bits(np.zeros((300, 71), np.int64)), u, v)
        with pytest.raises(AssertionError):
            fn(Xd, Xd, u[:-1], v)
        with pytest.raises(AssertionError):
            fn(Xd, Xd, u, np.zeros(71))
