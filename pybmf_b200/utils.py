"""Host-side mirror of the `PyBMF.utils` helpers that sit on the Asso hot path.

Same names, argument meaning, return containers and error behaviour as the reference
(file:line cited per function, relative to /root/reference), but every Boolean product and
every TP/FP/FN count is computed by the bit-packed kernels of libbmf_b200.so.  There is
no CPU fallback: without a B200 these functions raise `_native.NativeError`.

Only BINARY matrices are supported (non-zero = 1), which is what the reference's Boolean
helpers assume; real-valued `matmul(boolean=False)` and friends are out of scope.
"""
from __future__ import annotations

import numpy as np
import pandas as pd_
import scipy.sparse as sp
import torch
from scipy.sparse import coo_matrix, csc_matrix, csr_matrix, issparse, lil_matrix, spmatrix

from . import _native, device

# --------------------------------------------------------------------------------------------
# container helpers (PyBMF/utils/sparse_utils.py:5-55) -- pure format conversion, no arithmetic
# --------------------------------------------------------------------------------------------


def to_sparse(X, type="csr"):
    """PyBMF/utils/sparse_utils.py:5-20."""
    assert type in ["coo", "csr", "csc", "lil"], "Matrix type not available"
    return {"coo": coo_matrix, "csr": csr_matrix, "csc": csc_matrix, "lil": lil_matrix}[type](X)


def to_dense(X, squeeze=False, keep_nan=False):
    """PyBMF/utils/sparse_utils.py:23-36."""
    if keep_nan and issparse(X):
        coo = coo_matrix(X)
        out = np.full(X.shape, np.nan)
        out[coo.row, coo.col] = coo.data
        X = out
    if issparse(X):
        X = X.toarray()
    elif isinstance(X, np.matrix):
        X = np.asarray(X)
    return X.squeeze() if squeeze else X


def to_triplet(X):
    """PyBMF/utils/sparse_utils.py:39-46."""
    coo = coo_matrix(X)
    return (np.asarray(coo.row, dtype="int"), np.asarray(coo.col, dtype="int"), np.asarray(coo.data, dtype="float"))


def check_sparse(X, sparse=None):
    """PyBMF/utils/sparse_utils.py:49-55."""
    if sparse is True and not issparse(X):
        return to_sparse(X)
    if sparse is False and issparse(X):
        return to_dense(X)
    return X


def isnum(X):
    return isinstance(X, (int, float))


def ismat(X):
    return isinstance(X, (np.ndarray, spmatrix))


def binarize(X, threshold=0.5):
    """`(X > threshold).astype(int)`, strict -- PyBMF/utils/common.py:64-79."""
    Y = (X > threshold).astype(int)
    if isinstance(X, spmatrix):
        Y = to_sparse(Y, type=X.format)
    return Y


# --------------------------------------------------------------------------------------------
# device round trips
# --------------------------------------------------------------------------------------------
def _pattern(X) -> csr_matrix:
    if not ismat(X):
        raise TypeError("expected an ndarray or a scipy sparse matrix")
    if isinstance(X, np.ndarray) and X.ndim == 1:
        X = X.reshape(1, -1)
    return device.to_csr_pattern(X)


def _bits_on_device(X: csr_matrix, transposed=False):
    ip, ix = device.upload_csr(X)
    return device.pack_csr(ip, ix, X.shape[0], X.shape[1], transposed=transposed)


def _bits_to_csr(bits, m, n, dtype=np.int64, chunk_rows=8192) -> csr_matrix:
    """Bit matrix on device -> csr on host, unpacked in row chunks to bound host memory."""
    parts = []
    for r0 in range(0, m, chunk_rows):
        r1 = min(m, r0 + chunk_rows)
        dense = device.words_to_dense(bits[r0:r1].cpu().numpy(), n)
        parts.append(csr_matrix(dense, dtype=dtype))
    if not parts:
        return csr_matrix((m, n), dtype=dtype)
    return sp.vstack(parts, format="csr", dtype=dtype) if len(parts) > 1 else parts[0]


def _factor_words(U: csr_matrix):
    """Usage matrix (rows x k) -> k-bit words per row [rows, kw] on device."""
    k = U.shape[1]
    kw = max((k + 63) // 64, 1)
    ip, ix = device.upload_csr(U)
    words = kw + (kw & 1)                                    # pack_csr wants an even word count
    bits = device.zeros((max(U.shape[0], 1), words), torch.int64)
    if U.nnz:
        _native.call("bmf_pack_csr", ip, ix, U.shape[0], k, 0, bits, words)
    return bits[:, :kw].contiguous(), kw


def on_device(*mats, entries=False):
    """True when the given matrices (None skipped) are generate.DeviceBits (or DeviceEntries), False when they are host
    matrices.  A mix is a TypeError; a DeviceEntries is a TypeError unless `entries` is set (only eval takes one); a
    device matrix must hold this rank's ShardPlan rows (ValueError), so that a sum over the ranks counts every row once."""
    given = [X for X in mats if X is not None]
    kinds = {(hasattr(X, "bits") or hasattr(X, "zeros")) and hasattr(X, "r0") for X in given}
    if len(kinds) > 1:
        raise TypeError("cannot mix a generate.DeviceBits / DeviceEntries with a host matrix")
    if kinds != {True}:
        return False
    if not entries and any(hasattr(X, "zeros") for X in given):
        raise TypeError("a generate.DeviceEntries is taken by eval(X_gt=, U=, V=) only")
    from .engine import local_plan
    for X in mats:
        if X is not None:
            local_plan(X)
    return True


def _bits_confusion(G, P):
    """(TP, FP, FN) of two generate.DeviceBits with the same shape and rows, summed over the ranks (one all-reduce: a
    collective under an initialised process group)."""
    from .engine import all_reduce_sum
    if G.shape != P.shape:
        raise ValueError("shapes differ: %s and %s" % (G.shape, P.shape))
    counts = device.zeros((3,), torch.int64)
    if G.r1 > G.r0:
        _native.call("bmf_confusion_bits", G.bits, P.bits, G.r1 - G.r0, G.bits.shape[1], -1, counts, None, None)
    tp, fp, fn = (int(v) for v in all_reduce_sum(counts).cpu().numpy())
    return tp, fp, fn


def factor_counts(X, U, V):
    """(TP, FP, FN, size) of X against the Boolean product U o V^T, by bmf_confusion_factors (the product is never formed).

    X is a host matrix, or a generate.DeviceBits: then only this rank's rows of U are packed and the counts are summed
    over the ranks (one all-reduce: a collective under an initialised process group)."""
    Up, Vp = _pattern(U), _pattern(V)
    vt = _bits_on_device(Vp.T.tocsr())
    counts = device.zeros((3,), torch.int64)
    if not on_device(X):
        G = _pattern(X)
        uw, kw = _factor_words(Up)
        _native.call("bmf_confusion_factors", _bits_on_device(G), G.shape[0], device.words_for(G.shape[1]), uw, kw, vt,
                     Up.shape[1], int(G.nnz), counts, None, None)
        tp, fp, fn = (int(v) for v in counts.cpu().numpy())
        return tp, fp, fn, G.shape[0] * G.shape[1]
    from .engine import all_reduce_sum
    if Up.shape[0] != X.m or Vp.shape[0] != X.n or Up.shape[1] != Vp.shape[1]:
        raise ValueError("factors U %s and V %s do not fit X %s" % (Up.shape, Vp.shape, X.shape))
    if X.r1 > X.r0:
        uw, kw = _factor_words(Up[X.r0:X.r1])
        _native.call("bmf_confusion_factors", X.bits, X.r1 - X.r0, X.bits.shape[1], uw, kw, vt, Up.shape[1], -1, counts,
                     None, None)
    tp, fp, fn = (int(v) for v in all_reduce_sum(counts).cpu().numpy())
    return tp, fp, fn, X.m * X.n


def entry_counts(X, U, V):
    """(TP, FP, FN, size) over the STORED entries (evaluate_utils.py:32-44) of a generate.DeviceEntries -- or of a
    DeviceBits, whose stored entries are its ones -- against U o V^T, in one bmf_confusion_entries_factors pass over this
    rank's rows, summed over the ranks (one all-reduce: a collective under an initialised process group)."""
    from .engine import all_reduce_sum
    Up, Vp = _pattern(U), _pattern(V)
    if Up.shape[0] != X.m or Vp.shape[0] != X.n or Up.shape[1] != Vp.shape[1]:
        raise ValueError("factors U %s and V %s do not fit X %s" % (Up.shape, Vp.shape, X.shape))
    ones, zeros = (X.ones.bits, X.zeros.bits) if hasattr(X, "zeros") else (X.bits, None)
    counts = device.zeros((4,), torch.int64)
    if X.r1 > X.r0:
        uw, kw = _factor_words(Up[X.r0:X.r1])
        _native.call("bmf_confusion_entries_factors", ones, zeros, X.r1 - X.r0, ones.shape[1], uw, kw,
                     _bits_on_device(Vp.T.tocsr()), Up.shape[1], counts)
    tp, fp, n1, n0 = (int(v) for v in all_reduce_sum(counts).cpu().numpy())
    return tp, fp, n1 - tp, n1 + n0


def _product_bits(U: csr_matrix, Vt: csr_matrix):
    """bits of (U o Vt) for U (m x k) and Vt (k x n) given as patterns."""
    m, k = U.shape
    n = Vt.shape[1]
    uw, kw = _factor_words(U)
    vt = _bits_on_device(Vt)
    words = device.words_for(n)
    out = device.zeros((max(m, 1), words), torch.int64)
    if m > 0:
        _native.call("bmf_bool_product", uw, m, kw, vt, k, words, out)
    return out


# --------------------------------------------------------------------------------------------
# Boolean algebra (PyBMF/utils/boolean_utils.py)
# --------------------------------------------------------------------------------------------
def matmul(U, V, sparse=None, boolean=False):
    """`boolean_utils.matmul` (PyBMF/utils/boolean_utils.py:61-84), Boolean case on the GPU.

    OR-AND product: csr int64 when either input is sparse or `sparse=True`, else ndarray int64.
    """
    if not boolean:
        raise NotImplementedError("pybmf_b200.utils.matmul accelerates boolean=True only "
                                  "(the Asso hot path); real-valued products are out of scope")
    _native.require_gpu()
    want_sparse = bool(sparse or (issparse(U) or issparse(V)))
    Up, Vp = _pattern(U), _pattern(V)
    assert Up.shape[1] == Vp.shape[0], "U and V should be multiplicable"
    bits = _product_bits(Up, Vp)
    m, n = Up.shape[0], Vp.shape[1]
    if want_sparse:
        X = _bits_to_csr(bits, m, n, dtype=np.int64)
    else:
        X = device.bits_to_host(bits, n)[:m].astype(np.int64)
    return check_sparse(X, sparse=want_sparse)


def get_prediction(U, V, boolean=True, sparse=True):
    """`matmul(U, V.T, boolean, sparse)` -- PyBMF/utils/common.py:98-107."""
    return matmul(U, V.T, boolean=boolean, sparse=sparse)


def _elementwise(X, Y, op):
    """Bit-packed OR / AND on the device (bmf_bits_combine); returns (bits, m, n)."""
    _native.require_gpu()
    Xp, Yp = _pattern(X), _pattern(Y)
    assert Xp.shape == Yp.shape, "U and V should have the same shape"
    m, n = Xp.shape
    out = device.zeros((max(m, 1), device.words_for(n)), torch.int64)
    if m > 0:
        _native.call("bmf_bits_combine", _bits_on_device(Xp), _bits_on_device(Yp), m, out.shape[1],
                     {"or": 0, "and": 1}[op], out)
    return out, m, n


def add(X, Y, sparse=None, boolean=False):
    """`boolean_utils.add` (PyBMF/utils/boolean_utils.py:87-107): Boolean OR, returned as float64
    (the reference casts `.astype(bool).astype(float)`)."""
    if not boolean:
        raise NotImplementedError("only boolean=True is supported")
    bits, m, n = _elementwise(X, Y, "or")
    if sparse or issparse(X) or issparse(Y):
        return _bits_to_csr(bits, m, n, dtype=np.float64)
    return device.bits_to_host(bits, n)[:m].astype(np.float64)


def multiply(U, V, sparse=None, boolean=False):
    """`boolean_utils.multiply` (PyBMF/utils/boolean_utils.py:6-33), Boolean AND."""
    if not boolean:
        raise NotImplementedError("only boolean=True is supported")
    assert U.shape == V.shape, "U and V should have the same shape"
    bits, m, n = _elementwise(U, V, "and")
    if issparse(U) or issparse(V) or sparse:
        return check_sparse(_bits_to_csr(bits, m, n, dtype=np.int64), sparse=sparse)
    return check_sparse(device.bits_to_host(bits, n)[:m].astype(int), sparse=sparse)


def _residual_bits(x_bits, rows, U: csr_matrix, vt):
    """bits of (x AND NOT (U o V^T)) for `rows` bit rows x_bits and the rows of U, by one bmf_residual_factors launch
    (the product is never formed)."""
    out = device.zeros((max(rows, 1), x_bits.shape[1]), torch.int64)
    if rows > 0:
        uw, kw = _factor_words(U)
        _native.call("bmf_residual_factors", x_bits, rows, x_bits.shape[1], uw, kw, vt, U.shape[1], out)
    return out


def get_residual(X, U, V):
    """`X AND NOT (U o V^T)` -- PyBMF/utils/common.py:154-160 (returns lil like the reference).

    A generate.DeviceBits X gives a DeviceBits with the same shape and rows: this rank's rows of the residual, from this
    rank's rows of U (no collective)."""
    _native.require_gpu()
    Up, Vp = _pattern(U), _pattern(V)
    if on_device(X):
        if Up.shape[0] != X.m or Vp.shape[0] != X.n or Up.shape[1] != Vp.shape[1]:
            raise ValueError("factors U %s and V %s do not fit X %s" % (Up.shape, Vp.shape, X.shape))
        from .generate import DeviceBits
        bits = _residual_bits(X.bits, X.r1 - X.r0, Up[X.r0:X.r1], _bits_on_device(Vp.T.tocsr()))
        return DeviceBits(bits, X.m, X.n, X.r0, X.r1)
    assert Up.shape[1] == Vp.shape[1], "U and V should be multiplicable"
    Xp = _pattern(X)
    assert Xp.shape == (Up.shape[0], Vp.shape[0]), "U and V should have the same shape"
    m, n = Xp.shape
    bits = _residual_bits(_bits_on_device(Xp), m, Up, _bits_on_device(Vp.T.tocsr()))
    return lil_matrix(_bits_to_csr(bits, m, n, dtype=sp.csr_matrix(X).dtype))


# --------------------------------------------------------------------------------------------
# confusion counts and metrics (PyBMF/utils/metrics.py)
# --------------------------------------------------------------------------------------------
def confusion_counts(gt, pd, axis=None):
    """(TP, FP, FN) of PyBMF/utils/metrics.py:56-76 via bmf_confusion_bits.

    axis=None -> three Python ints; axis=1 -> per-row int64 arrays; axis=0 -> per-column.  Two generate.DeviceBits are
    counted on this rank's rows and summed over the ranks (axis=None only)."""
    _native.require_gpu()
    if on_device(gt, pd):
        if axis is not None:
            raise NotImplementedError("per-row / per-column counts of a generate.DeviceBits are not supported")
        return _bits_confusion(gt, pd)
    G, P = _pattern(gt), _pattern(pd)
    assert G.shape == P.shape, "U and V should have the same shape"
    if axis == 0:
        G, P = G.T.tocsr(), P.T.tocsr()
    m, n = G.shape
    words = device.words_for(n)
    counts = device.zeros((3,), torch.int64)
    row_tp = device.zeros((max(m, 1),), torch.int32)
    row_fp = device.zeros((max(m, 1),), torch.int32)
    if m > 0:
        gb, pb = _bits_on_device(G), _bits_on_device(P)
        _native.call("bmf_confusion_bits", gb, pb, m, words, int(G.nnz), counts, row_tp, row_fp)
    if axis is None:
        tp, fp, fn = (int(v) for v in counts.cpu().numpy())
        return tp, fp, fn
    tp = row_tp.cpu().numpy()[:m].astype(np.int64)
    fp = row_fp.cpu().numpy()[:m].astype(np.int64)
    fn = np.asarray(G.sum(axis=1)).ravel().astype(np.int64) - tp
    return tp, fp, fn


def _as_count(v):
    return np.array(v, dtype=np.int64) if np.ndim(v) == 0 else v


def TP(gt, pd, axis=None):
    """PyBMF/utils/metrics.py:56-58."""
    return _as_count(confusion_counts(gt, pd, axis)[0])


def FP(gt, pd, axis=None):
    """PyBMF/utils/metrics.py:61-68."""
    return _as_count(confusion_counts(gt, pd, axis)[1])


def FN(gt, pd, axis=None):
    """PyBMF/utils/metrics.py:75-76."""
    return _as_count(confusion_counts(gt, pd, axis)[2])


def _size(X, axis):
    if len(X.shape) == 2:
        return X.shape[0] * X.shape[1] if axis is None else X.shape[1 - axis]
    return len(X)


def TN(gt, pd, axis=None):
    """PyBMF/utils/metrics.py:71-72 -- `TP(invert(gt), invert(pd))`, computed from the identity
    TN = size - TP - FP - FN instead of two dense m x n inversions."""
    tp, fp, fn = confusion_counts(gt, pd, axis)
    return _as_count(_size(gt, axis) - tp - fp - fn)


def invert(X):
    """PyBMF/utils/metrics.py:163-170 (kept for API parity; dense, avoid on large inputs)."""
    if issparse(X):
        return csr_matrix(np.ones(X.shape)) - X
    if isinstance(X, np.ndarray):
        return 1 - X
    raise TypeError


def rates(tp, fp, fn, size, sum_pd=None):
    """Scalar metrics of PyBMF/utils/metrics.py:79-139 from integer counts, with the reference's
    literal float formulas (FPR = 1 - TNR, ERR = 1 - ACC, 0 when a denominator is 0)."""
    tp, fp, fn, size = int(tp), int(fp), int(fn), int(size)
    tn = size - tp - fp - fn
    sum_gt = tp + fn
    sum_pd = tp + fp if sum_pd is None else int(sum_pd)
    inv_gt = size - sum_gt
    f = np.float64
    tpr = f(tp) / f(sum_gt) if sum_gt > 0 else 0
    tnr = f(tn) / f(inv_gt) if inv_gt > 0 else 0
    ppv = f(tp) / f(sum_pd) if sum_pd > 0 else 0
    acc = f(tp + tn) / size
    denom = ppv + tpr
    out = {"TP": np.array(tp, dtype=np.int64), "FP": np.array(fp, dtype=np.int64),
           "TN": np.array(tn, dtype=np.int64), "FN": np.array(fn, dtype=np.int64),
           "TPR": tpr, "TNR": tnr, "FPR": 1 - tnr, "FNR": 1 - tpr, "PPV": ppv, "ACC": acc, "ERR": 1 - acc,
           "F1": 2 * ppv * tpr / denom if denom > 0 else 0}
    out.update({"Recall": out["TPR"], "Precision": out["PPV"], "Accuracy": out["ACC"], "Error": out["ERR"]})
    return out


def _rate(name):
    def fn(gt, pd, axis=None):
        if axis is not None:
            raise NotImplementedError("%s: only axis=None is supported (as used by evaluate())" % name)
        tp, fp, fn_ = confusion_counts(gt, pd, None)
        return rates(tp, fp, fn_, _size(gt, None))[name]
    fn.__name__ = name
    fn.__doc__ = "PyBMF/utils/metrics.py `%s` from the GPU confusion counts." % name
    return fn


TPR, TNR, FPR, FNR, PPV, ACC, ERR, F1 = (_rate(n) for n in ("TPR", "TNR", "FPR", "FNR", "PPV", "ACC", "ERR", "F1"))


def coverage_score(gt, pd, w_fp=0.5, w_fn=None, axis=None):
    """`- w_fp * FP + w_fn * TP` -- PyBMF/utils/metrics.py:189-201 (literal fp64 expression)."""
    w_fn = 1 - w_fp if w_fn is None else w_fn
    tp, fp, _ = confusion_counts(gt, pd, axis)
    return -w_fp * _as_count(fp) + w_fn * _as_count(tp)


def weighted_error(gt, pd, w_fp=0.5, w_fn=None, axis=None):
    """PyBMF/utils/metrics.py:182-186."""
    w_fn = 1 - w_fp if w_fn is None else w_fn
    _, fp, fn = confusion_counts(gt, pd, axis)
    return w_fp * _as_count(fp) + w_fn * _as_count(fn)


def description_length(gt, U, V, pd=None, w_model=1.0, w_fp=1.0, w_fn=1.0):
    """PyBMF/utils/metrics.py:173-179.  A generate.DeviceBits `gt` without `pd` is counted against the factors."""
    if pd is None and on_device(gt):
        _, fp, fn, _ = factor_counts(gt, U, V)
    else:
        pd = matmul(U, V.T, sparse=True, boolean=True) if pd is None else pd
        _, fp, fn = confusion_counts(gt, pd, None)
    return w_model * (U.sum() + V.sum()) + w_fp * _as_count(fp) + w_fn * _as_count(fn)


METRIC_NAMES = ("TP", "FP", "TN", "FN", "TPR", "FPR", "TNR", "FNR", "PPV", "ACC", "ERR", "F1",
                "Recall", "Precision", "Accuracy", "Error")


def metrics_from_counts(metrics, tp, fp, fn, size, sum_pd=None):
    """The dispatch of get_metrics (PyBMF/utils/metrics.py:31-52) once the counts are known;
    unknown names give None exactly as the reference does."""
    r = rates(tp, fp, fn, size, sum_pd)
    return [r[m] if m in r else None for m in metrics]


def get_metrics(gt, pd, metrics, axis=None):
    """PyBMF/utils/metrics.py:8-53."""
    if axis is not None:
        raise NotImplementedError("get_metrics: only axis=None is supported")
    host_pd = not on_device(pd)                             # bit rows hold no NaN
    if host_pd and (np.isnan(to_dense(pd, squeeze=True)).any() if not issparse(pd) else np.isnan(pd.data).any()):
        raise TypeError("NaN is found in prediction.")
    if isinstance(gt, np.ndarray) and gt.ndim == 1:        # triplet form of task='prediction'
        g = np.asarray(gt) != 0
        p = np.asarray(pd) != 0
        tp, fp, fn = int((g & p).sum()), int((~g & p).sum()), int((g & ~p).sum())
        return metrics_from_counts(metrics, tp, fp, fn, len(g))
    tp, fp, fn = confusion_counts(gt, pd, None)
    return metrics_from_counts(metrics, tp, fp, fn, _size(gt, None))


def eval(metrics, task, X_gt, X_pd=None, U=None, V=None):
    """PyBMF/utils/evaluate_utils.py:12-54 -- counts on the GPU; for task='prediction' the
    per-triplet Python loop (:41-44) becomes bmf_confusion_triplets.

    A generate.DeviceBits `X_gt` is compared with factors `U`, `V` under task='reconstruction' only, a
    generate.DeviceEntries under both tasks ('reconstruction' counts its ones, as of a host csr with stored zeros): this
    rank's rows against this rank's rows of U, summed over the ranks (a collective under an initialised process group)."""
    using_matrix = X_pd is not None
    using_factors = U is not None and V is not None
    assert using_matrix or using_factors, "[E] User should provide either `U`, `V` or `X_pd`."
    assert task in ["prediction", "reconstruction"], "[E] Task should be either 'prediction' or 'reconstruction'."
    _native.require_gpu()
    if on_device(X_gt, X_pd, entries=True):
        if using_matrix:
            raise TypeError("eval: a generate.DeviceBits / DeviceEntries X_gt is compared with factors U, V, not with X_pd")
        if hasattr(X_gt, "zeros"):
            if task == "reconstruction":
                return metrics_from_counts(metrics, *factor_counts(X_gt.ones, U, V))
            return metrics_from_counts(metrics, *entry_counts(X_gt, U, V))
        if task != "reconstruction":
            raise ValueError("eval: task='prediction' counts stored entries, which a generate.DeviceBits cannot hold")
    if not using_factors:
        if task == "reconstruction":
            return get_metrics(gt=to_sparse(X_gt, "csr"), pd=to_sparse(X_pd, "csr"), metrics=metrics)
        r, c, g = to_triplet(X_gt)
        P = csr_matrix(X_pd)
        pd_data = np.asarray(P[r, c]).ravel() if len(r) else np.zeros(0)
        return get_metrics(gt=g, pd=pd_data, metrics=metrics)
    if task == "reconstruction":
        return metrics_from_counts(metrics, *factor_counts(X_gt, U, V))
    Up, Vp = _pattern(U), _pattern(V)
    uw, kw = _factor_words(Up)
    r, c, g = to_triplet(X_gt)
    vw, _ = _factor_words(Vp)
    counts = device.zeros((4,), torch.int64)
    d = device.dev()
    _native.call("bmf_confusion_triplets", torch.from_numpy(r.astype(np.int32)).to(d),
                 torch.from_numpy(c.astype(np.int32)).to(d), torch.from_numpy((g != 0).astype(np.uint8)).to(d),
                 len(g), uw, kw, vw, counts)
    tp, fp, fn, _tn = (int(v) for v in counts.cpu().numpy())
    return metrics_from_counts(metrics, tp, fp, fn, len(g))


# --------------------------------------------------------------------------------------------
# log bookkeeping (PyBMF/utils/evaluate_utils.py:57-98) -- pandas only
# --------------------------------------------------------------------------------------------
def header(names, levels, depth=None):
    """PyBMF/utils/evaluate_utils.py:85-98."""
    depth = levels if depth is None else depth
    out = []
    for name in names:
        cells = [""] * levels
        cells[depth - 1] = name
        out.append(tuple(cells))
    return out


def record(df_dict, df_name, columns, records, verbose=False):
    """PyBMF/utils/evaluate_utils.py:57-82: append a timestamped row to logs[df_name]."""
    if df_name not in df_dict:
        if isinstance(columns[0], tuple):
            columns = pd_.MultiIndex.from_tuples(header(["time"], levels=len(columns[0])) + columns)
        else:
            columns = ["time"] + columns
        df_dict[df_name] = pd_.DataFrame(columns=columns)
    ts = [pd_.Timestamp.now().strftime("%d/%m/%y %I:%M:%S")]
    df = df_dict[df_name]
    df.loc[len(df.index)] = ts + records
    if verbose:
        print(df.tail())


def record_many(df_dict, df_name, columns, rows):
    """`record` for several rows at once (each row already starts with its timestamp): same table layout -- a `time`
    column first, MultiIndex columns when the names are tuples, object dtype like the reference's row-wise `.loc`."""
    if isinstance(columns[0], tuple):
        cols = pd_.MultiIndex.from_tuples(header(["time"], levels=len(columns[0])) + columns)
    else:
        cols = ["time"] + columns
    new = pd_.DataFrame([list(r) for r in rows], columns=cols, dtype=object)
    if df_name in df_dict and len(df_dict[df_name].index):
        old = df_dict[df_name]
        new.index = range(len(old.index), len(old.index) + len(new.index))
        df_dict[df_name] = pd_.concat([old, new])
    else:
        df_dict[df_name] = new
