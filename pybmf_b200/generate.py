"""Synthetic Boolean matrices generated ON the device (SURVEY.md section 8f, rank 3).

The reference builds its inputs on the host: `matmul(U, V.T, boolean=True)` of two random factors
(PyBMF/generators/BaseGenerator.py:202-221) followed by `add_noise` (PyBMF/utils/generator_utils.py:30-49).  At the
Netflix-shaped config that is a 1e8-nnz scipy matrix per rank (~10 s and 3 GB of host memory each).  Here the same recipe
runs on bit rows in HBM with a counter-based generator, so a rank generates only ITS rows of the one logical matrix and the
result does not depend on how many ranks there are.  It is not bit-identical to numpy's Mersenne-twister draws; tests pin
the densities, the shard independence and a whole fit against the CPU restatement run on the downloaded bits.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
import torch

from . import _native, device
from .engine import ShardPlan, dist_ctx, local_plan


class DeviceBits:
    """Rows [r0, r1) of a logical m x n Boolean matrix as bit rows on the current device."""

    def __init__(self, bits, m, n, r0, r1):
        self.bits, self.m, self.n, self.r0, self.r1 = bits, int(m), int(n), int(r0), int(r1)
        self.shape = (self.m, self.n)

    def to_csr(self) -> sp.csr_matrix:
        """This rank's rows as a host csr int64 (for cross-checks; moves m_loc * n / 8 bytes)."""
        from .utils import _bits_to_csr
        return _bits_to_csr(self.bits, self.r1 - self.r0, self.n)


class DeviceEntries:
    """The device form of a split with stored entries (task='prediction', evaluate_utils.py:32-44): `ones` holds the
    stored non-zeros and `zeros` the explicitly stored zeros of rows [r0, r1) of a logical m x n matrix, both
    DeviceBits over the same shape and the same ShardPlan rows.  The two must be disjoint (not checked: the producers
    here, entries_from_host and ratio_split, guarantee it)."""

    def __init__(self, ones: DeviceBits, zeros: DeviceBits):
        if ones.shape != zeros.shape or (ones.r0, ones.r1) != (zeros.r0, zeros.r1):
            raise ValueError("DeviceEntries: ones %s rows [%d, %d) and zeros %s rows [%d, %d) differ"
                             % (ones.shape, ones.r0, ones.r1, zeros.shape, zeros.r0, zeros.r1))
        local_plan(ones)
        self.ones, self.zeros = ones, zeros
        self.shape, self.m, self.n, self.r0, self.r1 = ones.shape, ones.m, ones.n, ones.r0, ones.r1

    def to_csr(self) -> sp.csr_matrix:
        """This rank's rows as a host csr int64 with the zeros stored explicitly (for cross-checks)."""
        ones = self.ones.to_csr().tocoo()
        zeros = self.zeros.to_csr().tocoo()
        rows = np.concatenate([ones.row, zeros.row])
        cols = np.concatenate([ones.col, zeros.col])
        data = np.concatenate([np.ones(ones.nnz, np.int64), np.zeros(zeros.nnz, np.int64)])
        order = np.lexsort((cols, rows))
        indptr = np.searchsorted(rows[order], np.arange(self.r1 - self.r0 + 1))
        return sp.csr_matrix((data[order], cols[order], indptr), shape=(self.r1 - self.r0, self.n))


def bits_from_host(X) -> DeviceBits:
    """This rank's ShardPlan rows of a host csr / ndarray as a DeviceBits; stored zeros are dropped."""
    from .utils import _bits_on_device, to_sparse
    X = X if sp.isspmatrix_csr(X) else to_sparse(X, "csr")
    _plan, r0, r1 = local_plan(X)
    Xl = device.csr_rows_view(X, r0, r1)
    if device.has_stored_zeros(Xl):                             # the packer takes every STORED entry as a one
        Xl = device.drop_stored_zeros(Xl)
    return DeviceBits(_bits_on_device(Xl), X.shape[0], X.shape[1], r0, r1)


def entries_from_host(X) -> DeviceEntries:
    """This rank's ShardPlan rows of a host matrix as a DeviceEntries: stored non-zeros into `ones`, explicitly stored
    zeros into `zeros` (an ndarray, converted to csr like everywhere else, stores none)."""
    from .utils import _bits_on_device, to_sparse
    X = X if sp.isspmatrix_csr(X) else to_sparse(X, "csr")
    _plan, r0, r1 = local_plan(X)
    Xl = device.csr_rows_view(X, r0, r1)
    zeros = Xl.copy()
    zeros.data = (zeros.data == 0).astype(np.int8)
    zeros.eliminate_zeros()
    m, n = X.shape
    return DeviceEntries(bits_from_host(X), DeviceBits(_bits_on_device(zeros), m, n, r0, r1))


def _rows_of(m, rank=None, world=None):
    if rank is None or world is None:
        rank, world = dist_ctx()
    return ShardPlan(m, world).rows(rank)


def random_bits(m, n, p, seed, stream_id=0, rank=None, world=None) -> DeviceBits:
    """Bernoulli(p) m x n matrix (this rank's rows)."""
    _native.require_gpu()
    r0, r1 = _rows_of(m, rank, world)
    words = device.words_for(n)
    bits = device.zeros((max(r1 - r0, 1), words), torch.int64)
    if r1 > r0:
        _native.call("bmf_random_bits", bits, r1 - r0, n, words, r0, int(seed), int(stream_id), float(p))
    return DeviceBits(bits, m, n, r0, r1)


def add_noise_bits(X: DeviceBits, noise=(0.0, 0.0), seed=0) -> DeviceBits:
    """`add_noise` (PyBMF/utils/generator_utils.py:30-49) in place: ones dropped with probability noise[0], then entries set
    with probability noise[1]."""
    if X.r1 > X.r0:
        _native.call("bmf_noise_bits", X.bits, X.r1 - X.r0, X.n, X.bits.shape[1], X.r0, int(seed), float(noise[0]),
                     float(noise[1]))
    return X


def planted_bits(m, n, k_true, d_u, d_v, p_fn, p_fp, seed, rank=None, world=None) -> DeviceBits:
    """The planted recipe of pybmf_b200.synth.planted on the device: U* ~ Bern(d_u)^{m x k}, V* ~ Bern(d_v)^{n x k},
    X = (U* o V*^T) with ones dropped with probability p_fn and entries set with probability p_fp."""
    _native.require_gpu()
    assert 1 <= k_true <= 64, "k_true <= 64 (one usage word per row)"
    r0, r1 = _rows_of(m, rank, world)
    rows = r1 - r0
    words = device.words_for(n)
    uw = device.zeros((max(rows, 1), 2), torch.int64)           # usage words (k bits; an even word count for alignment)
    vt = device.zeros((k_true, words), torch.int64)             # rows of V*^T, identical on every rank
    _native.call("bmf_random_bits", vt, k_true, n, words, 0, int(seed), 2, float(d_v))
    bits = device.zeros((max(rows, 1), words), torch.int64)
    if rows > 0:
        _native.call("bmf_random_bits", uw, rows, k_true, 2, r0, int(seed), 1, float(d_u))
        _native.call("bmf_bool_product", uw[:, :1].contiguous(), rows, 1, vt, k_true, words, bits)
        _native.call("bmf_noise_bits", bits, rows, n, words, r0, int(seed), float(p_fn), float(p_fp))
    return DeviceBits(bits, m, n, r0, r1)


def prediction(U, V, rank=None, world=None) -> DeviceBits:
    """The device form of utils.get_prediction: this rank's ShardPlan rows of the Boolean product U o V^T (m = U.shape[0],
    n = V.shape[0]) as a DeviceBits, from host factors (lil, csr or ndarray).  One bmf_bool_product launch on this rank's
    rows of U, no collective; the result does not depend on the number of ranks.  A factor column mismatch raises
    ValueError."""
    from .utils import _bits_on_device, _factor_words, _pattern
    _native.require_gpu()
    Up, Vp = _pattern(U), _pattern(V)
    if Up.shape[1] != Vp.shape[1]:
        raise ValueError("factors U %s and V %s should have the same number of columns" % (Up.shape, Vp.shape))
    (m, k), n = Up.shape, Vp.shape[0]
    r0, r1 = _rows_of(m, rank, world)
    words = device.words_for(n)
    bits = device.zeros((max(r1 - r0, 1), words), torch.int64)
    if r1 > r0:
        uw, kw = _factor_words(Up[r0:r1])
        _native.call("bmf_bool_product", uw, r1 - r0, kw, _bits_on_device(Vp.T.tocsr()), k, words, bits)
    return DeviceBits(bits, m, n, r0, r1)


_TRANSPOSE_STEP = 64 * 65535                                    # rows per bmf_transpose_bits launch (grid.y limit)


def _transpose_into(bits, rows, ncols, out, words_t):
    """Transpose the bit rows [rows][ncols bits] (row stride bits.stride(0)) into the first words of the rows of `out`
    (row stride words_t), in row chunks of _TRANSPOSE_STEP (a multiple of 64, so every chunk starts at a whole word)."""
    for a in range(0, rows, _TRANSPOSE_STEP):
        b = min(rows, a + _TRANSPOSE_STEP)
        _native.call("bmf_transpose_bits", bits[a:b], b - a, ncols, bits.stride(0), out[:, a // 64:], words_t)


def transpose_bits(bits, rows, ncols):
    """Bit matrix [rows][words(ncols)] -> its transpose [ncols][words(rows)] on the device."""
    words_t = device.words_for(rows)
    out = device.zeros((max(ncols, 1), words_t), torch.int64)
    _transpose_into(bits, rows, ncols, out, words_t)
    return out


def transpose_slots(m, n, world):
    """Layout of the one all-to-all exchange of `transpose` for an m x n matrix over `world` ranks (pure host logic).

    Rank r holds rows rows[r] of X and receives rows cols[r] of X^T (both ShardPlan).  Every rank sends every rank s one
    slot of slot_rows x slot_words int64 words: the transpose of its rows restricted to columns cols[s], which start at
    word src_word[s] of its bit rows.  The slot rank s receives from rank r fills used_words[r] words of each of its X^T
    rows (words_t words), starting at word dst_word[r].  Slots of a rank without rows or columns are sent all the same,
    as zeros."""
    rows, cols = ShardPlan(m, world).bounds, ShardPlan(n, world).bounds
    for lo, hi in rows + cols:
        assert lo % 64 == 0 or lo == hi, "the ranges of ranks that hold rows start at whole words"
    used = [(r1 - r0 + 63) // 64 for r0, r1 in rows]
    return {"rows": rows, "cols": cols, "slot_rows": max(c1 - c0 for c0, c1 in cols), "slot_words": max(used),
            "src_word": [c0 // 64 for c0, _c1 in cols], "dst_word": [r0 // 64 for r0, _r1 in rows], "used_words": used,
            "words_t": device.words_for(m)}


def transpose(X: DeviceBits) -> DeviceBits:
    """X^T of a row-sharded bit matrix, sharded the same way: this rank gets rows ShardPlan(n, world).rows(rank) of X^T,
    whatever the number of ranks.  With several ranks this is a collective (ONE all_to_all_single of transpose_slots);
    the send and the receive buffer take about m_loc * n / 8 bytes each."""
    local_plan(X)
    rank, world = dist_ctx()
    if world == 1:
        return DeviceBits(transpose_bits(X.bits, X.m, X.n), X.n, X.m, 0, X.n)
    import torch.distributed as dist
    L = transpose_slots(X.m, X.n, world)
    sr, sw, wt = L["slot_rows"], L["slot_words"], L["words_t"]
    send = device.zeros((world, sr, sw), torch.int64)
    m_loc = X.r1 - X.r0
    for s, (c0, c1) in enumerate(L["cols"]):
        if m_loc > 0 and c1 > c0:
            _transpose_into(X.bits[:, L["src_word"][s]:], m_loc, c1 - c0, send[s], sw)
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv, send)
    c0, c1 = L["cols"][rank]
    out = device.zeros((max(c1 - c0, 1), wt), torch.int64)
    for r in range(world):
        w0, nw = L["dst_word"][r], L["used_words"][r]
        if nw > 0 and c1 > c0:
            out[: c1 - c0, w0:w0 + nw] = recv[r, : c1 - c0, :nw]
    return DeviceBits(out, X.n, X.m, c0, c1)


SPLIT_STREAMS = (5, 6)                                          # counter streams of ratio_split: ones, zeros


def _threshold(p):
    """bmf_random_bits' probability -> 32-bit threshold (bernoulli_threshold in bmf_bits.cu)."""
    if not p > 0.0:
        return 0
    if p >= 1.0:
        return 0xFFFFFFFF
    return int(p * 4294967296.0)


def split_thresholds(ones, m, n, val_size, test_size, neg_ratio=1.0):
    """The thresholds of ratio_split (pure host logic): (t_v, t_t, q_v, q_t).  A one draws u and goes to val below t_v,
    to test below t_v + t_t; a zero becomes a stored zero of val below q_v, of test below q_v + q_t, where
    q_s = thr(neg_ratio * s_size * ones / (m * n - ones)).  Bad sizes, or too few zeros, raise ValueError."""
    for name, v in (("val_size", val_size), ("test_size", test_size)):
        if not 0.0 <= v <= 1.0:
            raise ValueError("%s must be in [0, 1], got %r" % (name, v))
    if val_size + test_size > 1.0:
        raise ValueError("val_size + test_size must not exceed 1, got %r" % (val_size + test_size))
    if not neg_ratio >= 0.0:
        raise ValueError("neg_ratio must be >= 0, got %r" % (neg_ratio,))
    zeros = m * n - ones
    need = neg_ratio * (val_size + test_size) * ones
    if need > 0 and (zeros == 0 or need / zeros > 1.0):
        raise ValueError("neg_ratio %r asks for %.0f negatives, the matrix has %d zeros" % (neg_ratio, need, zeros))
    q_v = neg_ratio * val_size * ones / zeros if zeros else 0.0
    q_t = neg_ratio * test_size * ones / zeros if zeros else 0.0
    return _threshold(val_size), _threshold(test_size), _threshold(q_v), _threshold(q_t)


def ratio_split(X: DeviceBits, val_size, test_size, neg_ratio=1.0, seed=0):
    """Split the ones of a row-sharded bit matrix into train / val / test and sample stored zeros (negatives) for val and
    test: returns (X_train: DeviceBits, X_val: DeviceEntries, X_test: DeviceEntries) on this rank's rows.

    Every one at (i, j) draws a 32-bit uniform number from the counter scheme of random_bits (stream SPLIT_STREAMS[0],
    global bit index as random_bits) and goes to val with probability val_size, to test with probability test_size,
    else to train.  Every zero draws from stream SPLIT_STREAMS[1] and becomes a stored zero of val (test) with probability
    neg_ratio * val_size (test_size) * |X| / (m n - |X|): about neg_ratio negatives per positive in each split.  The result
    depends on (seed, i, j) only, not on the number of ranks.  This is this project's own recipe: it does not reproduce
    the random draws of the reference's RatioSplit.

    A collective under an initialised process group (ONE all-reduce of |X|); bad sizes raise ValueError on every rank."""
    from .engine import all_reduce_sum
    local_plan(X)
    _native.require_gpu()
    rows, words = X.r1 - X.r0, X.bits.shape[1]
    ones = device.zeros((3,), torch.int64)
    if rows > 0:
        _native.call("bmf_confusion_bits", X.bits, X.bits, rows, words, -1, ones, None, None)
    total = int(all_reduce_sum(ones)[0])
    t_v, t_t, q_v, q_t = split_thresholds(total, X.m, X.n, val_size, test_size, neg_ratio)
    out = device.zeros((5, max(rows, 1), words), torch.int64)
    if rows > 0:
        _native.call("bmf_split_bits", X.bits, rows, X.n, words, X.r0, int(seed), SPLIT_STREAMS[0], SPLIT_STREAMS[1],
                     t_v, t_t, q_v, q_t, out)
    part = [DeviceBits(out[i], X.m, X.n, X.r0, X.r1) for i in range(5)]
    return part[0], DeviceEntries(part[1], part[2]), DeviceEntries(part[3], part[4])
