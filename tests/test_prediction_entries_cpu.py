"""CPU: the thresholds of generate.ratio_split and their errors, and the numpy restatement of its draws on the ShardPlan
rows of 1 .. 8 ranks against the world-1 result."""
import numpy as np
import pytest

from pybmf_b200.engine import ShardPlan
from pybmf_b200.generate import split_thresholds

from split_reference import draws, ratio_split_rows

T32 = 4294967296.0


def test_thresholds_follow_the_random_bits_conversion():
    m, n, ones = 1000, 701, 70100
    t_v, t_t, q_v, q_t = split_thresholds(ones, m, n, 0.1, 0.2, neg_ratio=1.0)
    assert (t_v, t_t) == (int(0.1 * T32), int(0.2 * T32))
    zeros = m * n - ones
    assert q_v == int(0.1 * ones / zeros * T32) and q_t == int(0.2 * ones / zeros * T32)
    assert split_thresholds(ones, m, n, 0.0, 1.0, 0.0) == (0, 0xFFFFFFFF, 0, 0)
    assert split_thresholds(ones, m, n, 0.5, 0.5, 2.0)[2:] == (int(ones / zeros * T32),) * 2
    assert split_thresholds(0, m, n, 0.1, 0.1, 1.0) == (int(0.1 * T32), int(0.1 * T32), 0, 0)
    assert split_thresholds(m * n, m, n, 0.1, 0.1, 0.0)[2:] == (0, 0)          # no zeros, none asked for


@pytest.mark.parametrize("args", [(-0.1, 0.1, 1.0), (0.1, 1.1, 1.0), (0.6, 0.5, 1.0), (0.1, 0.1, -1.0),
                                  (0.1, 0.1, float("nan")), (float("nan"), 0.1, 1.0)])
def test_threshold_errors(args):
    with pytest.raises(ValueError):
        split_thresholds(100, 100, 100, *args)


def test_too_few_zeros():
    split_thresholds(6000, 100, 100, 0.3, 0.3, 1.0)                          # 3600 negatives from 4000 zeros
    with pytest.raises(ValueError):
        split_thresholds(900, 30, 30, 0.3, 0.3, 1.0)                          # 540 negatives, 0 zeros
    with pytest.raises(ValueError):
        split_thresholds(800, 30, 30, 0.5, 0.5, 1.0)                          # 800 negatives, 100 zeros


def test_draws_are_uniform_and_distinct_per_stream():
    a, b = draws(7, 5, 0, 64, 1000), draws(7, 6, 0, 64, 1000)
    assert a.max() < 2 ** 32 and abs(a.mean() / 2 ** 32 - 0.5) < 0.01
    assert (a != b).mean() > 0.999


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("m,n", [(1000, 701), (257, 65), (3000, 130)])
def test_shard_rows_equal_world_one(m, n, world):
    rng = np.random.default_rng(m + n)
    X = rng.random((m, n)) < 0.2
    th = split_thresholds(int(X.sum()), m, n, 0.1, 0.2, 1.5)
    whole = ratio_split_rows(X, 0, n, 11, th)
    for r0, r1 in ShardPlan(m, world).bounds:
        part = ratio_split_rows(X[r0:r1], r0, n, 11, th)
        for a, b in zip(part, whole):
            assert np.array_equal(a, b[r0:r1])
    train, v1, v0, s1, s0 = whole
    assert np.array_equal(train | v1 | s1, X) and not (train & v1).any() and not (v1 & s1).any()
    assert not ((v0 | s0) & X).any() and not (v0 & s0).any()
