"""GreConD's concept search on the GPU (`pybmf_b200.models.GreConD`; DESIGN.md section 1 row f5).

The reference's rule, recovered from its golden run (tests/grecond_reference.py states it in numpy): a factor starts from
C = all rows, D = {}, best = 0 and makes ONE pass over the columns in order; column j (not in D) gives the extent
C_j = C & X[:, j], its intent D_j = AND of the rows of C_j, and the cover s_j = |R & (C_j x D_j)| on the residual R; the
first j with s_j > best replaces (C, D, best).  The factor is (C, D); then R &= ~(C x D).

Here the pass is cut in three:
  seed     the first accepted column of a factor is the first j with a non-zero cover against all rows.  Covers only
           shrink as R loses ones, so the scan resumes where the previous factor's seed was found (`Concepts.p`).  One
           window of 64 columns is scored per step: bmf_concept_intents on this rank's rows, an all-gather of the partial
           intents and row counts, bmf_concept_covers and an all-reduce of the 64 covers.
  extent   every later C is a subset of the seed column's rows: each rank compacts its rows of that column (X and R)
           with bmf_concept_extent, padded to the largest rank share, and one all-gather gives every rank all of them
           in logical row order (extent_layout).
  rounds   on those rows, replicated on every rank with no collective: every candidate after `pos` is scored against
           the current C (bmf_concept_intents + bmf_concept_covers), bmf_concept_decide accepts the first one whose
           cover exceeds `best` or marks the factor done.  Rounds are enqueued in stretches and the state is read once
           per stretch.  The first round starts from pos = seed - 1, best = 0, so it accepts the seed itself.
The residual update (bmf_concept_residual) touches each rank's own rows of C only.  The result does not depend on the
number of ranks: every rank takes the same decisions on the same integers.

Memory: the compact rows take 2 x (ranks x largest share of the seed column) x words x 8 bytes on every rank; a column
that has a one in every row is the bound, two copies of X.  Intents of every column take ceil(n / 64) x 64 x words x 8
bytes (39.5 MB at 17770 columns).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native, device
from .engine import all_reduce_sum, dist_ctx

FIRST_STRETCH = 4                                            # rounds enqueued before the state is first read


def extent_layout(counts):
    """Layout of the all-gathered extent rows for per-rank row counts of the seed column (pure host logic).

    Every rank sends `cap` = max(counts) rows; rank q's rows land at [q cap, q cap + counts[q]) of the `rows` = R cap
    gathered rows, the rest is padding.  `valid` holds the bits of the real rows as int64 words (the first C)."""
    counts = [int(c) for c in counts]
    cap = max(counts) if counts else 0
    rows = cap * len(counts)
    flags = np.zeros((1, max(rows, 1)), np.uint8)
    for q, c in enumerate(counts):
        flags[0, q * cap: q * cap + c] = 1
    return {"cap": cap, "rows": rows, "valid": device.dense_to_words(flags)[0]}


def first_cover(covers, cw, n):
    """The first column of column word cw with a non-zero cover in the 64 seed covers, or -1 (pure host logic)."""
    hit = np.flatnonzero(np.asarray(covers)[: max(0, min(64, n - 64 * cw))] > 0)
    return 64 * cw + int(hit[0]) if len(hit) else -1


def _all_gather(t, world):
    """[world, *t.shape]: every rank's t (t itself when there is one rank)."""
    if world == 1:
        return t.unsqueeze(0)
    import torch.distributed as dist
    out = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t.contiguous())
    return out


class Concepts:
    """The factor loop on this rank's bit rows x [rows r1 - r0][words] of an m x n matrix (all rows with one process).
    Under an initialised process group every method is a collective; every rank gets the same factors."""

    def __init__(self, x_bits, m, n, r0, r1):
        _native.require_gpu()
        self.rank, self.world = dist_ctx()
        self.x, self.res = x_bits, x_bits.clone()
        self.m, self.n, self.r0, self.r1 = int(m), int(n), int(r0), int(r1)
        self.m_loc, self.words = self.r1 - self.r0, x_bits.shape[1]
        self.ncw = (self.n + 63) // 64
        ones = device.zeros((3,), torch.int64)
        if self.m_loc > 0:
            _native.call("bmf_confusion_bits", self.x, self.x, self.m_loc, self.words, -1, ones, None, None)
        self.ones = int(all_reduce_sum(ones)[0])
        self.p = 0                                           # every column before p has a zero cover for good
        self.seed_buf = device.zeros((64 * self.words + 64,), torch.int64)
        self.seed_covers = device.zeros((64,), torch.int64)
        self.intents = device.zeros((self.ncw * 64, self.words), torch.int64)
        self.covers = device.zeros((self.ncw * 64,), torch.int64)

    def seed(self):
        """(first column with a non-zero cover, the per-rank row counts of that column) or (-1, None)."""
        W = self.words
        while self.p < self.n:
            cw = self.p // 64
            _native.call("bmf_concept_intents", self.x, self.m_loc, W, self.n, None, cw, 1, self.p, None, None,
                         self.seed_buf[: 64 * W], self.seed_buf[64 * W:])
            parts = _all_gather(self.seed_buf, self.world)
            _native.call("bmf_concept_covers", self.x, self.res, self.m_loc, W, self.n, None, cw, 1, self.p, None, None,
                         parts, self.world, 64 * W + 64, self.seed_covers)
            j = first_cover(all_reduce_sum(self.seed_covers).cpu().numpy(), cw, self.n)
            if j >= 0:
                self.p = j
                return j, parts[:, 64 * W + j - 64 * cw].cpu().numpy()
            self.p = 64 * (cw + 1)
        return -1, None

    def extent(self, col, counts):
        """The rows of column col from every rank, compacted (extent_layout): (xc, rc, idx, valid c_bits, rows)."""
        L = extent_layout(counts)
        cap, W = L["cap"], self.words
        xc, rc = device.zeros((max(cap, 1), W), torch.int64), device.zeros((max(cap, 1), W), torch.int64)
        idx, fill = device.zeros((max(cap, 1),), torch.int64), device.zeros((1,), torch.int64)
        _native.call("bmf_concept_extent", self.x, self.res, self.m_loc, W, self.r0, col, cap, xc, rc, idx, fill)
        xc, rc, idx = (_all_gather(t, self.world).reshape((-1,) + tuple(t.shape[1:])) for t in (xc, rc, idx))
        c_bits = torch.from_numpy(L["valid"].copy()).to(self.x.device)
        return xc, rc, idx, c_bits, L["rows"]

    def rounds(self, xc, rc, c_bits, d_bits, state, rows, count):
        """Enqueue `count` candidate rounds on the compact rows (no-ops once the factor is done)."""
        W, n = self.words, self.n
        for _ in range(count):
            _native.call("bmf_concept_intents", xc, rows, W, n, c_bits, 0, self.ncw, 0, state, d_bits, self.intents, None)
            _native.call("bmf_concept_covers", xc, rc, rows, W, n, c_bits, 0, self.ncw, 0, state, d_bits, self.intents, 1,
                         0, self.covers)
            _native.call("bmf_concept_decide", xc, rows, W, n, self.covers, self.intents, state, c_bits, d_bits)

    def factor(self):
        """The next factor as (logical rows of C, columns of D, its cover), or None when no column covers a residual
        one.  Updates this rank's rows of the residual."""
        j0, counts = self.seed()
        if j0 < 0:
            return None
        xc, rc, idx, c_bits, rows = self.extent(j0, counts)
        d_bits = device.zeros((self.words,), torch.int64)
        state = torch.tensor([j0 - 1, 0, 0, 0], dtype=torch.int64, device=self.x.device)
        stretch, ran = FIRST_STRETCH, 0
        while True:
            self.rounds(xc, rc, c_bits, d_bits, state, rows, stretch)
            ran += stretch
            st = state.cpu().numpy()
            if st[2] or ran > self.n:
                break
            stretch *= 2
        assert st[2] and st[3] >= 1, "GreConD rounds ended without a decision"
        self.accepted = int(st[3])                           # columns accepted by the rounds (the seed included)
        if self.m_loc > 0:
            _native.call("bmf_concept_residual", self.res, self.r0, self.r1, self.words, idx, rows, c_bits, d_bits)
        members = device.words_to_dense(c_bits.cpu().numpy()[None], rows)[0] != 0
        extent = np.sort(idx.cpu().numpy()[:rows][members])
        intent = np.flatnonzero(device.words_to_dense(d_bits.cpu().numpy()[None], self.n)[0])
        return extent, intent, int(st[1])
