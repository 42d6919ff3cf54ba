"""GreConD+'s pattern expansion on the GPU -- `expansion` / `_expansion` of PyBMF/models/GreConDPlus.py:207-308
(SURVEY.md section 8f, rank 1), same names, arguments and return values.

`_expansion(X_gt, X_old, u, v, w_fp, w_fn, axis)` is get_vector's shape seen from the other side: instead of asking
which rows should use a given pattern, it asks which ONE row (axis = 1) or column (axis = 0) gains most from joining
the pattern u x v.  Per row i outside u:  delta_i = coverage_score(x_i, old_i | v) - coverage_score(x_i, old_i), evaluated
with the reference's fp64 expression (PyBMF/utils/metrics.py:201) on integer TP / FP counts; rows already in u get
exactly 0.  For host matrices the counts come from one streaming pass over the bit rows (bmf_expand_scores); column-wise
expansion runs the same kernel on the transposed bit matrices.

`expansion()` grows the pattern incrementally on the row layout.  X_old is fixed for the whole loop, so one pass
(bmf_expand_init) gives every row's and every column's TP_old / FP_old and the increments P / N against (u, v); an
iteration then changes P / N by one bit per row (a column joined v) or by one row's bits per column (a row joined u), and
costs O(m + n) instead of two passes over all four bit matrices.  Iterations are enqueued in stretches and decided on the
device; the iteration log is read once per stretch.

Both functions accept generate.DeviceBits inputs (this rank's ShardPlan rows); under an initialised process group they are
then collectives.  `expansion()` does ONE all-reduce per iteration (exchange_layout / merge_slots).
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
import torch

from . import _native, device
from . import utils as U_

FIRST_STRETCH = 64                                           # iterations enqueued before the log is first read


def _vec_bits(vec, length):
    """0/1 vector (any container, (len, 1) / (1, len) / flat) -> device bit row [1, words_for(length)]."""
    v = vec.toarray() if sp.issparse(vec) else np.asarray(vec)
    v = (np.asarray(v).reshape(-1) != 0).astype(np.uint8)
    assert v.size == length, "u and v should match the shape of X"
    return torch.from_numpy(device.dense_to_words(v.reshape(1, -1))).to(device.dev())


# ---- the per-iteration exchange (pure host logic, CPU-testable) -------------------------------------------------------
def exchange_layout(world, words):
    """Layout of the int64 buffer that expansion() sums over the ranks once per iteration.

    [0, 2 world): one slot per rank, (bits of the rank's max row delta as int64, the logical row of that max or -1 when the
    rank has no rows); each rank writes only its own slot and zeros elsewhere.  Then `words` words of x & ~old and `words`
    words of ~x & ~old (masked to n) of the row chosen by the previous decision: its owner writes them, the other ranks
    zeros.  Summing with zeros is exact, so the SUM is a gather."""
    return {"slots": (0, 2 * world), "row_pos": (2 * world, 2 * world + words),
            "row_neg": (2 * world + words, 2 * world + 2 * words), "size": 2 * world + 2 * words}


def merge_slots(slots, world):
    """(score, logical row) of the summed slots: the maximum, and among equal maxima the lowest row; ranks whose index is
    -1 hold no rows.  This is the first argmax over the concatenated rows, because every rank's slot holds its own first
    argmax (bmf_expand_step_decide applies the same rule on the device)."""
    s = np.asarray(slots, dtype=np.int64)[: 2 * world]
    best, idx = np.float64(0.0), -1
    for q in range(world):
        val, i = s[2 * q: 2 * q + 1].view(np.float64)[0], int(s[2 * q + 1])
        if i >= 0 and (idx < 0 or val > best or (val == best and i < idx)):
            best, idx = val, i
    return best, idx


def pack_slot(buf, rank, score, index):
    """Write (score, index) into rank's slot of an int64 exchange buffer (index -1: the rank has no rows)."""
    buf[2 * rank] = np.array([score], dtype=np.float64).view(np.int64)[0] if index >= 0 else 0
    buf[2 * rank + 1] = index


# ---- inputs ---------------------------------------------------------------------------------------------------------
class _Rows:
    """X_gt / X_old as bit rows on the device: all rows of host matrices (world 1, no collective), or this rank's
    ShardPlan rows of generate.DeviceBits (every check raises on every rank, before any collective)."""

    def __init__(self, X_gt, X_old):
        _native.require_gpu()
        from .engine import dist_ctx
        if U_.on_device(X_gt, X_old):
            if X_gt.shape != X_old.shape or X_gt.bits.shape[1] != X_old.bits.shape[1]:
                raise ValueError("X_gt %s and X_old %s should have the same shape" % (X_gt.shape, X_old.shape))
            self.rank, self.world = dist_ctx()
            (self.m, self.n), self.r0, self.r1 = X_gt.shape, X_gt.r0, X_gt.r1
            self.x, self.o = X_gt.bits, X_old.bits
        else:
            G, O = U_._pattern(X_gt), U_._pattern(X_old)
            assert G.shape == O.shape, "X_gt and X_old should have the same shape"
            self.rank, self.world = 0, 1
            (self.m, self.n), self.r0, self.r1 = G.shape, 0, G.shape[0]
            self.x, self.o = U_._bits_on_device(G), U_._bits_on_device(O)
        self.m_loc = self.r1 - self.r0
        self.words = self.x.shape[1]

    def all_reduce(self, t):
        """SUM over the ranks when the inputs are sharded (host inputs stay local)."""
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t

    def counts(self, u_bits, v_bits):
        """bmf_expand_init: per-row (TP_old, FP_old, P, N) [m_loc, 4] int32 and the per-column counts [4, n] int64 summed
        over the ranks."""
        row_cnt = device.zeros((max(self.m_loc, 1), 4), torch.int32)
        col_cnt = device.zeros((4, self.n), torch.int64)
        _native.call("bmf_expand_init", self.x, self.o, self.m_loc, self.n, self.words, self.r0, u_bits, v_bits, row_cnt,
                     col_cnt)
        return row_cnt, self.all_reduce(col_cnt)


class _ExpansionState:
    """X_gt and X_old as host-packed bit rows in both orientations, resident on the device (the host `_expansion` path)."""

    def __init__(self, X_gt, X_old):
        _native.require_gpu()
        G, O = U_._pattern(X_gt), U_._pattern(X_old)
        assert G.shape == O.shape, "X_gt and X_old should have the same shape"
        self.m, self.n = G.shape
        self.x = U_._bits_on_device(G)
        self.o = U_._bits_on_device(O)
        self.xt = U_._bits_on_device(G, transposed=True)
        self.ot = U_._bits_on_device(O, transposed=True)
        self.delta = device.zeros((max(self.m, self.n),), torch.float64)
        self.best = device.zeros((2,), torch.int64)

    def score(self, u_bits, v_bits, w_fp, w_fn, axis):
        """(max delta, first argmax) over rows (axis = 1) or columns (axis = 0) -- GreConDPlus.py:275-308."""
        w_fn = 1 - w_fp if w_fn is None else w_fn
        if axis == 1:
            x, o, rows, pat, exc = self.x, self.o, self.m, v_bits, u_bits
        elif axis == 0:
            x, o, rows, pat, exc = self.xt, self.ot, self.n, u_bits, v_bits
        else:
            raise UnboundLocalError("cannot access local variable '_u' where it is not associated with a value")
        _native.call("bmf_expand_scores", x, o, rows, x.shape[1], pat, exc, float(w_fp), float(w_fn), self.delta, self.best)
        b = self.best.cpu().numpy()
        return np.float64(b[0:1].view(np.float64)[0]), int(b[1])


def _expansion(X_gt, X_old, u, v, w_fp, w_fn, axis):
    """Row-wise (axis = 1) or column-wise (axis = 0) expansion score of the pattern u x v -- GreConDPlus.py:267-308.
    Returns (score, index) = (d_scores.max(), d_scores.argmax()).

    With generate.DeviceBits inputs, axis = 1 scores this rank's rows (bmf_expand_scores) and merges the ranks' (max,
    argmax) slots; axis = 0 sums the column counts of bmf_expand_init over the ranks and scores the columns.  Either way
    one all-reduce: a collective under an initialised process group."""
    if not U_.on_device(X_gt, X_old):
        st = _ExpansionState(X_gt, X_old)
        return st.score(_vec_bits(u, st.m), _vec_bits(v, st.n), w_fp, w_fn, axis)
    if axis not in (0, 1):
        raise UnboundLocalError("cannot access local variable '_u' where it is not associated with a value")
    R = _Rows(X_gt, X_old)
    u_bits, v_bits = _vec_bits(u, R.m), _vec_bits(v, R.n)
    w_fn = 1 - w_fp if w_fn is None else w_fn
    best = device.zeros((2,), torch.int64)
    if axis == 0:
        _row_cnt, col_cnt = R.counts(u_bits, v_bits)
        delta = device.zeros((R.n,), torch.float64)
        _native.call("bmf_expand_col_scores", col_cnt, R.n, v_bits, float(w_fp), float(w_fn), delta, best)
        b = best.cpu().numpy()
        return np.float64(b[0:1].view(np.float64)[0]), int(b[1])
    slots = device.zeros((2 * R.world,), torch.int64)
    slots[2 * R.rank + 1] = -1
    if R.m_loc > 0:
        delta = device.zeros((R.m_loc,), torch.float64)
        _native.call("bmf_expand_scores", R.x, R.o, R.m_loc, R.words, v_bits, u_bits[:, R.r0 // 64:], float(w_fp),
                     float(w_fn), delta, best)
        slots[2 * R.rank] = best[0]
        slots[2 * R.rank + 1] = best[1] + R.r0
    score, index = merge_slots(R.all_reduce(slots).cpu().numpy(), R.world)
    return np.float64(score), int(index)


def expansion(X_gt, X_old, u, v, w_fp, w_fn):
    """Grow the pattern (u, v) one row or column at a time while that raises the coverage score --
    GreConDPlus.py:207-264.  Returns the expansion parts (u_exp, v_exp) as (m, 1) / (n, 1) lil matrices.

    Host matrices are packed once in the row layout and expanded on this process alone.  generate.DeviceBits inputs are
    expanded on this rank's rows, with ONE all-reduce per iteration: a collective under an initialised process group,
    whose result is the same on every rank."""
    R = _Rows(X_gt, X_old)
    m, n = R.m, R.n
    steps = _loop(R, u, v, w_fp, w_fn)
    rows, cols = steps[steps[:, 0] == 0, 1], steps[steps[:, 0] == 1, 1]
    u_exp = sp.csr_matrix((np.ones(len(rows)), (rows, np.zeros(len(rows), np.int64))), shape=(m, 1)).tolil()
    v_exp = sp.csr_matrix((np.ones(len(cols)), (cols, np.zeros(len(cols), np.int64))), shape=(n, 1)).tolil()
    from .models import _say
    _say(f"[I]     expansion() finished after {len(steps)} iterations.")
    return u_exp, v_exp


def expansion_log(X_gt, X_old, u, v, w_fp, w_fn):
    """The iterations of expansion() as an int64 array [n_iter, 2] of (0, row) | (1, column) | (2, -1) for the final
    stop, in order."""
    return _loop(_Rows(X_gt, X_old), u, v, w_fp, w_fn)


def _loop(R, u, v, w_fp, w_fn):
    """The incremental loop on the rows R (see the module docstring); returns expansion_log's array."""
    m, n, words = R.m, R.n, R.words
    u_bits, v_bits = _vec_bits(u, m), _vec_bits(v, n)
    w_fn = 1 - w_fp if w_fn is None else w_fn
    row_cnt, col_cnt = R.counts(u_bits, v_bits)
    cap = m + n + 1                                          # every iteration but the last adds a new row or column
    log = torch.full((cap, 2), -1, dtype=torch.int64, device=device.dev())
    state = torch.tensor([0, -1, -1, 0, 0, 0, 0, 0], dtype=torch.int64, device=device.dev())
    partials = device.zeros((4 * 1024,), torch.int64)
    xbuf = device.zeros((exchange_layout(R.world, words)["size"],), torch.int64)
    done, stretch, entries = 0, FIRST_STRETCH, []
    while True:
        k = min(stretch, cap - done)
        for _ in range(k):
            _native.call("bmf_expand_step_rows", R.x, R.o, R.m_loc, n, words, R.r0, u_bits, row_cnt, float(w_fp),
                         float(w_fn), state, partials, xbuf, R.world, R.rank)
            R.all_reduce(xbuf)
            _native.call("bmf_expand_step_decide", col_cnt, n, words, u_bits, v_bits, float(w_fp), float(w_fn), state,
                         partials, xbuf, R.world, log, cap)
        got = log[done:done + k].cpu().numpy()
        done += k
        entries.append(got)
        if (got[:, 0] == 2).any() or done >= cap:
            break
        stretch *= 2
    steps = np.concatenate(entries)
    return steps[steps[:, 0] >= 0]
