"""numpy statements of GreConD as the reference runs it (recovered from tests/golden/grecond.npz, the genuine run of
oracle/make_golden_ext.py:grecond_case), shared by the GreConD tests: the plain one-pass first-improvement loop, a
simulation of the protocol of pybmf_b200.concept over R ranks, and the seeded cases both are run on.

The rule, per factor: C = all rows, D = {}, best = 0; ONE pass over the columns j in order, skipping j in D:
C_j = C & X[:, j], D_j = AND of the rows of C_j (all columns when C_j is empty), s = |R & (C_j x D_j)|, and
`if s > best` (strict) the pair replaces (C, D).  best == 0 after the pass ends the fit.  Then R &= ~(C x D).  The
textbook GreConD (best of all j per step) and a non-strict `>=` both disagree with the golden; whether the reference
repeats the pass until nothing changes is not pinned by it (the one pass is what is built)."""
import numpy as np

from pybmf_b200.concept import extent_layout, first_cover
from pybmf_b200.engine import ShardPlan


def _intent(X, C):
    return X[C].all(axis=0) if C.any() else np.ones(X.shape[1], bool)


def grecond(X, k=None):
    """(U [m, t] uint8, V [n, t] uint8, covers [t]) of the reference loop, t <= k factors (k=None: until no cover)."""
    X = np.asarray(X) != 0
    m, n = X.shape
    R = X.copy()
    Us, Vs, covers = [], [], []
    while k is None or len(Us) < k:
        C, D, best = np.ones(m, bool), np.zeros(n, bool), 0
        for j in range(n):
            if D[j]:
                continue
            Cj = C & X[:, j]
            Dj = _intent(X, Cj)
            s = int(R[np.ix_(Cj, Dj)].sum())
            if s > best:
                best, C, D = s, Cj, Dj
        if best == 0:
            break
        Us.append(C)
        Vs.append(D)
        covers.append(best)
        R &= ~(C[:, None] & D[None, :])
    return _stack(Us, m), _stack(Vs, n), covers


def grecond_packed(X, k=None):
    """grecond() on bit-packed rows (np.bitwise_count), for the larger property cases; same results."""
    Xb = np.asarray(X) != 0
    m, n = Xb.shape
    Xp = np.packbits(Xb, axis=1, bitorder="little")
    Rp = Xp.copy()
    full = np.packbits(np.ones(n, bool), bitorder="little")
    Us, Vs, covers = [], [], []
    while k is None or len(Us) < k:
        C, D, Dp, best = np.ones(m, bool), np.zeros(n, bool), None, 0
        for j in range(n):
            if D[j]:
                continue
            rows = np.flatnonzero(C & Xb[:, j])
            if not len(rows):
                continue                                                # empty extent: cover 0
            Dj = np.bitwise_and.reduce(Xp[rows], axis=0)
            s = int(np.bitwise_count(Rp[rows] & Dj).sum())
            if s > best:
                best, Dp = s, Dj
                C = np.zeros(m, bool)
                C[rows] = True
                D = np.unpackbits(Dj, bitorder="little")[:n] != 0
        if best == 0:
            break
        Us.append(C)
        Vs.append(D)
        covers.append(best)
        Rp[C] &= ~Dp & full
    return _stack(Us, m), _stack(Vs, n), covers


def _stack(cols, rows):
    return np.stack(cols, 1).astype(np.uint8) if cols else np.zeros((rows, 0), np.uint8)


def metrics(X, covers):
    """The train log columns of the reference (Recall, Precision, Accuracy, F1) after each factor: TP is the running sum
    of the covers and FP = 0, because every factor is a formal concept of X."""
    X = np.asarray(X) != 0
    size, ones = X.size, int(X.sum())
    out = []
    for tp in np.cumsum(covers):
        tp, fp, fn = np.float64(tp), np.float64(0), np.float64(ones - tp)
        rec, prec = tp / (tp + fn), tp / (tp + fp)
        out.append((rec, prec, (size - fp - fn) / size, 2 * prec * rec / (prec + rec)))
    return np.array(out).reshape(-1, 4)


def seed_scan(R, X, j):
    """cover1_j = |R & (X[:, j] x closure{j})|: the cover of column j against all rows."""
    Cj = X[:, j]
    return int(R[np.ix_(Cj, _intent(X, Cj))].sum())


def sharded_grecond(X, k=None, world=1, window=64):
    """The protocol of pybmf_b200.concept over `world` ranks holding ShardPlan rows: the seed pointer that only moves
    forward, seed windows scored from per-rank partial intents (ANDed) and summed covers, the extent rows gathered in
    extent_layout, first-exceeding rounds on them, and each rank's own rows of the residual updated.  Returns what
    grecond() returns plus the seed columns."""
    X = np.asarray(X) != 0
    m, n = X.shape
    bounds = ShardPlan(m, world).bounds
    R = X.copy()
    p, Us, Vs, covers, seeds = 0, [], [], [], []
    while k is None or len(Us) < k:
        j0 = -1
        while p < n:
            cw = p // window
            cols = [j for j in range(cw * window, min(n, (cw + 1) * window))]
            parts = []                                                  # per rank: (intents, counts) of the window
            for a, b in bounds:
                Xs = X[a:b]
                parts.append(([np.logical_and.reduce(Xs[Xs[:, j]], axis=0) if Xs[:, j].any() else np.ones(n, bool)
                               for j in cols], [int(Xs[:, j].sum()) for j in cols]))
            covers64 = np.zeros(64, np.int64)
            for i, j in enumerate(cols):
                if j < p:
                    continue
                I = np.logical_and.reduce([pt[0][i] for pt in parts])
                covers64[i] = sum(int(R[a:b][np.ix_(X[a:b, j], I)].sum()) for a, b in bounds)
            j0 = first_cover(covers64, cw, n)
            if j0 >= 0:
                p = j0
                counts = [pt[1][j0 - cw * window] for pt in parts]
                break
            p = window * (cw + 1)
        if j0 < 0:
            break
        L = extent_layout(counts)
        rows_of = np.full(L["rows"], -1)
        for q, (a, b) in enumerate(bounds):
            got = a + np.flatnonzero(X[a:b, j0])
            rows_of[q * L["cap"]: q * L["cap"] + len(got)] = got
        valid = np.unpackbits(L["valid"].view(np.uint8), bitorder="little")[: L["rows"]] != 0
        assert np.array_equal(valid, rows_of >= 0)
        Xc, Rc = X[np.maximum(rows_of, 0)], R[np.maximum(rows_of, 0)]
        C, D, pos, best = valid, np.zeros(n, bool), j0 - 1, 0
        while True:                                                     # rounds: first j > pos with s_j > best
            s = np.zeros(n, np.int64)
            for j in range(pos + 1, n):
                if not D[j]:
                    Cj = C & Xc[:, j]
                    s[j] = int(Rc[np.ix_(Cj, _intent(Xc, Cj))].sum())
            live = np.flatnonzero((s > best) & (np.arange(n) > pos) & ~D)
            if not len(live):
                break
            pos = int(live[0])
            C = C & Xc[:, pos]
            D, best = _intent(Xc, C), int(s[pos])
        U = np.zeros(m, bool)
        U[rows_of[C]] = True
        for a, b in bounds:
            R[a:b] &= ~(U[a:b, None] & D[None, :])
        Us.append(U)
        Vs.append(D)
        covers.append(best)
        seeds.append(j0)
    return _stack(Us, m), _stack(Vs, n), covers, seeds


def planted(m, n, k, density, noise, seed):
    """A planted Boolean matrix with noise (uint8)."""
    rng = np.random.RandomState(seed)
    U = rng.rand(m, k) < density
    V = rng.rand(n, k) < density
    X = (U.astype(np.int64) @ V.T.astype(np.int64)) > 0
    X ^= rng.rand(m, n) < noise
    return X.astype(np.uint8)


def ragged_cases():
    """(name, X, k) of the shapes the device fit is checked on against grecond()."""
    rng = np.random.RandomState(11)
    cases = [("m<64", planted(40, 90, 3, 0.3, 0.05, 1), 5),
             ("n%64", planted(300, 130, 4, 0.2, 0.03, 2), 8),
             ("n=1", (rng.rand(77, 1) < 0.5).astype(np.uint8), 3),
             ("zeros", np.zeros((50, 70), np.uint8), 4),
             ("ones", np.ones((65, 129), np.uint8), 3),
             ("k_none", planted(120, 70, 3, 0.25, 0.02, 3), None),
             ("truncated", planted(30, 20, 2, 0.3, 0.0, 4), 50)]
    X = planted(200, 150, 4, 0.2, 0.05, 5)
    X[:, [0, 17, 64, 149]] = 0                                          # empty columns, at the start of a word too
    cases.append(("empty_cols", X, 10))
    X = planted(260, 200, 4, 0.2, 0.05, 6)
    X[:, 70] = 1                                                        # a column with a one in every row
    cases.append(("full_col", X, 6))
    return cases
