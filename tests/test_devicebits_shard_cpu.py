"""CPU: the slot layout of generate.transpose (one all-to-all of fixed-size slots) for world = 1 .. 8, ragged m and n and
ranks without rows or columns, and a numpy simulation of the whole exchange on dense blocks against X^T."""
import numpy as np
import pytest

from pybmf_b200.engine import ShardPlan
from pybmf_b200.generate import transpose_slots

SHAPES = [(1, 1), (63, 65), (256, 256), (300, 1000), (257, 70), (1000, 300), (2049, 1777), (5000, 130)]


def _simulate(X, world):
    """Every rank packs its slots as transpose() does, the all-to-all is a reshuffle of the slot list, every rank places
    what it received; returns the X^T rows of every rank as dense 0/1 [rows][words_t * 64] blocks."""
    m, n = X.shape
    L = transpose_slots(m, n, world)
    sr, sw, wt = L["slot_rows"], L["slot_words"], L["words_t"]
    send = np.zeros((world, world, sr, sw * 64), np.uint8)               # [from][to] slot, bits unpacked
    for r, (r0, r1) in enumerate(L["rows"]):
        for s, (c0, c1) in enumerate(L["cols"]):
            if r1 > r0 and c1 > c0:
                send[r, s, : c1 - c0, : r1 - r0] = X[r0:r1, L["src_word"][s] * 64:L["src_word"][s] * 64 + (c1 - c0)].T
    out = []
    for s, (c0, c1) in enumerate(L["cols"]):
        recv = send[:, s]                                                # what rank s receives from every rank
        block = np.zeros((max(c1 - c0, 1), wt * 64), np.uint8)
        for r in range(world):
            w0, nw = L["dst_word"][r], L["used_words"][r]
            if nw and c1 > c0:
                block[: c1 - c0, w0 * 64:(w0 + nw) * 64] = recv[r, : c1 - c0, : nw * 64]
        out.append(block)
    return L, out


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("m,n", SHAPES)
def test_every_bit_sent_once_in_whole_words(m, n, world):
    L = transpose_slots(m, n, world)
    assert L["rows"] == ShardPlan(m, world).bounds and L["cols"] == ShardPlan(n, world).bounds
    assert L["words_t"] * 64 >= m and L["words_t"] % 2 == 0
    hits = np.zeros((m, n), np.int64)
    for r, (r0, r1) in enumerate(L["rows"]):
        if r1 > r0:
            assert r0 % 64 == 0 and L["dst_word"][r] * 64 == r0                # whole-word offsets
            assert L["used_words"][r] == -(-(r1 - r0) // 64) <= L["slot_words"]
            assert L["dst_word"][r] + L["used_words"][r] <= L["words_t"]
        else:
            assert L["used_words"][r] == 0
        for s, (c0, c1) in enumerate(L["cols"]):
            if c1 > c0:
                assert c0 % 64 == 0 and L["src_word"][s] * 64 == c0
                assert c1 - c0 <= L["slot_rows"]
            hits[r0:r1, c0:c1] += 1
    assert (hits == 1).all()                                             # every bit of X^T is sent exactly once
    # the receive buffer is world slots, and their used words tile the X^T rows without a gap or an overlap
    spans = [(L["dst_word"][r], L["dst_word"][r] + L["used_words"][r]) for r in range(world) if L["used_words"][r]]
    assert spans[0][0] == 0 and spans[-1][1] == -(-m // 64)
    assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
    assert sum(r1 - r0 for r0, r1 in L["rows"]) == m and sum(c1 - c0 for c0, c1 in L["cols"]) == n
    # the buffers stay about m_loc * n / 8 bytes: slot_words * 64 covers rank 0's rows, slot_rows rank 0's columns
    r0_, r1_ = L["rows"][0]
    c0_, c1_ = L["cols"][0]
    assert L["slot_words"] == -(-(r1_ - r0_) // 64) and L["slot_rows"] == c1_ - c0_


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("m,n", SHAPES)
def test_simulated_exchange_reproduces_transpose(m, n, world):
    rng = np.random.RandomState(m * 31 + n * 7 + world)
    X = (rng.rand(m, n) < 0.3).astype(np.uint8)
    L, out = _simulate(X, world)
    for s, (c0, c1) in enumerate(L["cols"]):
        block = out[s]
        if c1 > c0:
            assert np.array_equal(block[: c1 - c0, :m], X[:, c0:c1].T), (m, n, world, s)
        assert not block[:, m:].any()                                    # pad bits stay zero
    got = np.concatenate([out[s][: c1 - c0, :m] for s, (c0, c1) in enumerate(L["cols"])], axis=0)
    assert np.array_equal(got, X.T)
