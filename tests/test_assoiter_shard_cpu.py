"""CPU: the algebra behind the row-sharded AssoIter.  A sweep's per-column table (TP, FP, #used, sum P, sum N after each
column) is a sum over rows, and each row's refinement depends on that row alone, so tables computed on disjoint row
blocks and summed, then replayed by models.replay_sweep, must reproduce AssoIter on the whole matrix: trace, logged
scores / errors and U."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import asso_oracle as O


def _sweep_table(X, U, V, upto, w_fp, w_fn):
    """Columns 0 .. upto-1 of AssoIter.get_refined_column on the rows of X (U refined in place), as the per-column table
    of bmf_refine_sweep."""
    k = V.shape[1]
    table = np.zeros((max(upto, 1), 5), np.int64)
    for c in range(upto):
        idx = [i for i in range(k) if i != c]
        C_old = O.bool_product(U[:, idx], V[:, idx])
        _s, use, P, N, _t, _f = O.score_candidates(X, C_old, V[:, c].reshape(1, -1), w_fp, w_fn)
        u = use[:, 0]
        U[:, c] = u
        tp, fp, _ = O.confusion(X, O.bool_product(U, V))
        table[c] = [tp, fp, u.sum(), P[u, 0].sum(), N[u, 0].sum()]
    return table


def _sharded_iter(X, U, V, k, w_fp, w_fn, cuts):
    from pybmf_b200.models import replay_sweep
    from pybmf_b200 import utils as U_
    U = U.copy()
    m, n = X.shape
    size = m * n
    parts = list(zip(cuts[:-1], cuts[1:]))
    tot = sum(np.array(O.confusion(X[a:b], O.bool_product(U[a:b], V)), np.int64) for a, b in parts)
    tp, fp, fn = (int(v) for v in tot)
    sum_x = tp + fn
    best_score = -w_fp * np.array(fp, dtype=np.int64) + w_fn * np.array(tp, dtype=np.int64)
    best_error = U_.rates(tp, fp, fn, size)["ERR"]
    n_stop = 0
    trace, scores, errors = [], [], []
    while True:
        snapshot = U.copy()
        table = sum(_sweep_table(X[a:b], U[a:b], V, k, w_fp, w_fn) for a, b in parts)     # U[a:b] is a view: refined in place
        steps, stop, best_error, best_score, n_stop = replay_sweep(table, k, sum_x, size, w_fp, w_fn, best_error,
                                                                   best_score, n_stop)
        for s in steps:
            trace.append((s["k"], s["accepted"]))
            if s["accepted"]:
                scores.append(float(s["score"]))
                errors.append(float(s["error"]))
        if stop is not None:
            U = snapshot
            for a, b in parts:
                _sweep_table(X[a:b], U[a:b], V, stop + 1, w_fp, w_fn)
            return U, trace, scores, errors


@pytest.mark.parametrize("name", ["ex01_6", "c1_noisy", "planted_w02", "planted_w025"])
def test_summed_row_block_tables_replay_to_the_whole_matrix_fit(name):
    c = load_golden(name)
    g = c["g"]
    X = c["X"].astype(np.uint8)
    U0, V0 = (np.asarray(g["U"]) != 0).astype(np.uint8), (np.asarray(g["V"]) != 0).astype(np.uint8)
    k = U0.shape[1]
    w_fp, w_fn = O.resolve_weights(c["w_fp"], c["w_fn"])
    ref = O.asso_iter_fit(X, U0, V0, k, w_fp, w_fn)
    m = X.shape[0]
    for cuts in ([0, m // 2, m], [0, m // 3, m // 3, m], [0, 1, (2 * m) // 3, m]):        # incl. an empty block
        U, trace, scores, errors = _sharded_iter(X, U0, V0, k, w_fp, w_fn, cuts)
        assert trace == [(c_, bool(a)) for c_, a in ref["trace"]], cuts
        assert np.array_equal(U, ref["U"]), cuts
        assert scores == [r["score"] for r in ref["refinements"]]
        assert errors == [r["error"] for r in ref["refinements"]]


def test_replay_stops_mid_sweep_and_carries_state():
    from pybmf_b200.models import replay_sweep
    size, sum_x = 1000, 100
    # column 0 improves the error, columns 1 and 2 do not: with k = 3 and n_stop = 1 on entry the stop comes at column 2
    table = np.array([[90, 5, 0, 0, 0], [80, 5, 0, 0, 0], [85, 9, 0, 0, 0]], np.int64)
    steps, stop, err, score, n_stop = replay_sweep(table, 3, sum_x, size, 0.5, 0.5, 0.02, 40.0, 1)
    assert [(s["k"], s["accepted"]) for s in steps] == [(0, True), (1, False), (2, False)]
    assert stop is None and n_stop == 2 and err == pytest.approx(0.015) and float(score) == 42.5
    steps, stop, err2, _s, n_stop = replay_sweep(table, 3, sum_x, size, 0.5, 0.5, err, score, n_stop)
    assert [(s["k"], s["accepted"]) for s in steps] == [(0, False)] and stop == 0 and n_stop == 3 and err2 == err
