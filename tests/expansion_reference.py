"""numpy statements of GreConD+'s expansion loop (PyBMF/models/GreConDPlus.py:207-308) shared by the expansion tests:
the reference loop that recomputes every row and column delta in each iteration, a simulation of the sharded protocol of
pybmf_b200.expansion over R ranks, and the seeded cases both are run on."""
import numpy as np

from pybmf_b200 import device
from pybmf_b200.engine import ShardPlan
from pybmf_b200.expansion import exchange_layout, merge_slots, pack_slot

STOP = 2


def deltas(X, O, u, v, w_fp, w_fn):
    """Per-row deltas of adding v to every row outside u (GreConDPlus.py:275-308); rows in u get +0.0."""
    X, O = X.astype(np.int64), O.astype(np.int64)
    tp, fp = (X * O).sum(1), ((1 - X) * O).sum(1)
    P, N = (X * (1 - O)) @ v.astype(np.int64), ((1 - X) * (1 - O)) @ v.astype(np.int64)
    d = (-w_fp * (fp + N) + w_fn * (tp + P)) - (-w_fp * fp + w_fn * tp)
    d[u != 0] = 0.0
    return d


def rule(r_score, r_index, c_score, c_index):
    """GreConDPlus.py:221-236: (0, row) | (1, column) | (STOP, -1)."""
    if r_score > c_score and r_score > 0:
        return 0, int(r_index)
    if c_score > r_score and c_score > 0:
        return 1, int(c_index)
    return STOP, -1


def reference_loop(X, O, u, v, w_fp, w_fn):
    """[(kind, index)] of every iteration, the last one (STOP, -1).  Every row and column delta is recomputed in each
    iteration (the fixed matrices are formed once, the products with u and v are exact in fp64)."""
    u, v = (np.asarray(u) != 0).astype(np.int64), (np.asarray(v) != 0).astype(np.int64)
    X, O = (X != 0).astype(np.int64), (O != 0).astype(np.int64)
    pos, neg = (X * (1 - O)).astype(np.float64), ((1 - X) * (1 - O)).astype(np.float64)
    tp_r, fp_r, tp_c, fp_c = (X * O).sum(1), ((1 - X) * O).sum(1), (X * O).sum(0), ((1 - X) * O).sum(0)

    def d(tp, fp, A, pat, exc):
        P, N = (A[0] @ pat).astype(np.int64), (A[1] @ pat).astype(np.int64)
        out = (-w_fp * (fp + N) + w_fn * (tp + P)) - (-w_fp * fp + w_fn * tp)
        out[exc != 0] = 0.0
        return out

    steps = []
    while True:
        r, c = d(tp_r, fp_r, (pos, neg), v, u), d(tp_c, fp_c, (pos.T, neg.T), u, v)
        kind, at = rule(r.max(), r.argmax(), c.max(), c.argmax())
        steps.append((kind, at))
        if kind == STOP:
            return steps
        (u if kind == 0 else v)[at] = 1


def sharded_loop(X, O, u, v, w_fp, w_fn, world):
    """The protocol of expansion() over `world` ranks holding ShardPlan rows: integer counts kept incrementally, each rank
    fills only its slot and, when it owns the row chosen last, that row's words; the buffers are summed and every rank
    merges the slots and decides.  Returns the steps (as reference_loop) and the summed buffers of every iteration."""
    m, n = X.shape
    X, O = (X != 0).astype(np.int64), (O != 0).astype(np.int64)
    u, v = (np.asarray(u) != 0).astype(np.int64), (np.asarray(v) != 0).astype(np.int64)
    words = device.words_for(n)
    L = exchange_layout(world, words)
    pos, neg = X * (1 - O), (1 - X) * (1 - O)
    bounds = ShardPlan(m, world).bounds
    # per-rank row counts and the column counts summed over the ranks (bmf_expand_init + one all-reduce)
    rows = [dict(tp=(X[a:b] * O[a:b]).sum(1), fp=((1 - X[a:b]) * O[a:b]).sum(1), P=pos[a:b] @ v, N=neg[a:b] @ v)
            for a, b in bounds]
    tpc, fpc = (X * O).sum(0), ((1 - X) * O).sum(0)
    Pc, Nc = sum(pos[a:b].T @ u[a:b] for a, b in bounds), sum(neg[a:b].T @ u[a:b] for a, b in bounds)
    last_row, last_col, steps = -1, -1, []
    while True:
        bufs = []
        for rank, (a, b) in enumerate(bounds):
            R = rows[rank]
            if last_col >= 0:
                R["P"] += pos[a:b, last_col]
                R["N"] += neg[a:b, last_col]
            buf = np.zeros(L["size"], np.int64)
            if b > a:
                d = (-w_fp * (R["fp"] + R["N"]) + w_fn * (R["tp"] + R["P"])) - (-w_fp * R["fp"] + w_fn * R["tp"])
                d[u[a:b] != 0] = 0.0
                pack_slot(buf, rank, d.max(), a + int(d.argmax()))
            else:
                pack_slot(buf, rank, 0.0, -1)
            if a <= last_row < b:
                buf[slice(*L["row_pos"])] = device.dense_to_words(pos[last_row:last_row + 1], words)[0]
                buf[slice(*L["row_neg"])] = device.dense_to_words(neg[last_row:last_row + 1], words)[0]
            bufs.append(buf)
        total = np.sum(bufs, axis=0)
        if last_row >= 0:
            Pc = Pc + device.words_to_dense(total[None, slice(*L["row_pos"])], n)[0]
            Nc = Nc + device.words_to_dense(total[None, slice(*L["row_neg"])], n)[0]
        c = (-w_fp * (fpc + Nc) + w_fn * (tpc + Pc)) - (-w_fp * fpc + w_fn * tpc)
        c[v != 0] = 0.0
        r_score, r_index = merge_slots(total, world)
        kind, at = rule(r_score, r_index, c.max(), c.argmax())
        steps.append((kind, at))
        if kind == STOP:
            return steps
        last_row, last_col = (at, -1) if kind == 0 else (-1, at)
        (u if kind == 0 else v)[at] = 1


def block_case(m, n, rows, w_fp, w_fn, seed):
    """A block of `rows` rows x n // 3 columns, v = the block's columns, u = its first row: exactly `rows` iterations
    (rows - 1 rows join, then every delta is <= 0)."""
    rng = np.random.RandomState(seed)
    X = (rng.rand(m, n) < 0.02).astype(np.int64)
    X[: rows] = 0
    cols = n // 3
    X[:rows, :cols] = 1
    X[rows:, :cols] = 0
    perm_r, perm_c = rng.permutation(m), rng.permutation(n)
    u = np.zeros(m, np.int64)
    u[0] = 1
    v = np.zeros(n, np.int64)
    v[:cols] = 1
    O = np.zeros((m, n), np.int64)
    return X[perm_r][:, perm_c], O, u[perm_r], v[perm_c], w_fp, w_fn


def planted_case(m, n, w_fp, w_fn, seed, density=0.08, old=0.1):
    """A planted block (about half the rows and a third of the columns) with noise, X_old a noisy part of it, and a seed
    pattern inside the block: long runs that mix rows and columns."""
    rng = np.random.RandomState(seed)
    br, bc = max(1, m // 2), max(1, n // 3)
    X = (rng.rand(m, n) < density).astype(np.int64)
    X[:br, :bc] |= (rng.rand(br, bc) < 0.9).astype(np.int64)
    O = (X * (rng.rand(m, n) < old)).astype(np.int64)
    O |= (rng.rand(m, n) < 0.01).astype(np.int64)
    u, v = np.zeros(m, np.int64), np.zeros(n, np.int64)
    u[: max(1, br // 8)] = 1
    v[: max(1, bc // 8)] = 1
    pr, pc = rng.permutation(m), rng.permutation(n)
    return X[pr][:, pc], O[pr][:, pc], u[pr], v[pc], w_fp, w_fn


def tie_case(m, n):
    """A k x k block of ones, u = its first row, v = its first column, X_old empty: the first row and the first column
    both gain w_fn, so the loop stops on r_score == c_score > 0 in its first iteration."""
    k = min(m, n, 5)
    X = np.zeros((m, n), np.int64)
    X[:k, :k] = 1
    u, v = np.zeros(m, np.int64), np.zeros(n, np.int64)
    u[0], v[0] = 1, 1
    return X, np.zeros((m, n), np.int64), u, v


def random_case(m, n, w_fp, w_fn, seed, u_mode="random", v_mode="random"):
    rng = np.random.RandomState(seed)
    X = (rng.rand(m, n) < 0.3).astype(np.int64)
    O = (rng.rand(m, n) < 0.2).astype(np.int64)
    pick = {"random": lambda k: (rng.rand(k) < 0.3).astype(np.int64), "empty": lambda k: np.zeros(k, np.int64),
            "all": lambda k: np.ones(k, np.int64)}
    return X, O, pick[u_mode](m), pick[v_mode](n), w_fp, w_fn


SHAPES = [(1, 1), (70, 130), (257, 65), (33, 1000), (600, 4100)]
WEIGHTS = [(0.5, 0.5), (0.2, 0.8), (0.3, 0.6)]
