"""GreConD without a GPU: the numpy restatement against the genuine reference run (tests/golden/grecond.npz), the seed
pointer's forward-only scan against the plain scan, and the sharded protocol of pybmf_b200.concept against world 1."""
import os

import numpy as np
import pytest

from grecond_reference import grecond, grecond_packed, metrics, ragged_cases, planted, seed_scan, sharded_grecond
from pybmf_b200.concept import extent_layout, first_cover
from pybmf_b200.engine import ShardPlan

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_restatement_reproduces_golden():
    g = np.load(os.path.join(GOLDEN, "grecond.npz"))
    U, V, covers = grecond(g["X"], k=6)
    assert np.array_equal(U, g["U"]) and np.array_equal(V, g["V"])
    got = metrics(g["X"], covers)
    for i, name in enumerate(("Recall", "Precision", "Accuracy", "F1")):
        assert np.array_equal(got[:, i], g["log_" + name]), name
    # the seed of every factor is column 0 (with best = 0, the first column whose closure touches a residual one wins)
    assert all(V[0, t] == 1 for t in range(6))


@pytest.mark.parametrize("seed", range(12))
def test_seed_pointer_equals_plain_scan(seed):
    """cover1_j never grows while factors are removed, so the first column with cover1 > 0 never moves back."""
    rng = np.random.RandomState(seed)
    m, n = rng.randint(1, 90), rng.randint(1, 150)
    X = planted(m, n, 3, 0.3, 0.05, seed) != 0
    U, V, _covers = grecond(X)
    R, p = X.copy(), 0
    for t in range(U.shape[1]):
        plain = next(j for j in range(n) if seed_scan(R, X, j) > 0)
        assert all(seed_scan(R, X, j) == 0 for j in range(p))
        p = plain
        assert V[p, t] == 1                                            # the seed is in the factor's intent
        R &= ~(U[:, t, None].astype(bool) & V[None, :, t].astype(bool))
    assert U.shape[1] == 0 or all(seed_scan(R, X, j) == 0 for j in range(n))


@pytest.mark.parametrize("world", range(1, 9))
def test_extent_layout(world):
    rng = np.random.RandomState(world)
    for _ in range(20):
        counts = [int(c) for c in rng.randint(0, 40, size=world) * (rng.rand(world) < 0.7)]
        L = extent_layout(counts)
        assert L["cap"] == max(counts) and L["rows"] == world * max(counts)
        bits = np.unpackbits(L["valid"].view(np.uint8), bitorder="little")
        want = np.zeros(len(bits), np.uint8)
        for q, c in enumerate(counts):
            want[q * L["cap"]: q * L["cap"] + c] = 1
        assert np.array_equal(bits, want)


def test_first_cover():
    cov = np.zeros(64, np.int64)
    assert first_cover(cov, 3, 1000) == -1
    cov[[5, 9]] = 1
    assert first_cover(cov, 2, 1000) == 133
    assert first_cover(cov, 2, 133) == -1                              # columns at or past n do not count
    assert first_cover(cov, 0, 6) == 5


@pytest.mark.parametrize("m,n", [(1, 1), (40, 130), (130, 70), (300, 65), (257, 200)])
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_sharded_protocol_equals_reference(m, n, world):
    """Ranks without rows included (ShardPlan aligns shares to whole row blocks, so small m leaves ranks empty)."""
    X = planted(m, n, 3, 0.25, 0.04, m * 7 + n) != 0
    U, V, covers = grecond(X, k=6)
    Us, Vs, cs, _seeds = sharded_grecond(X, k=6, world=world)
    assert np.array_equal(U, Us) and np.array_equal(V, Vs) and covers == cs
    if world > 1 and m <= 256:
        assert any(b == a for a, b in ShardPlan(m, world).bounds)


def test_sharded_protocol_on_golden():
    g = np.load(os.path.join(GOLDEN, "grecond.npz"))
    for world in (1, 2, 4):
        U, V, _c, seeds = sharded_grecond(g["X"], k=6, world=world)
        assert np.array_equal(U, g["U"]) and np.array_equal(V, g["V"]) and seeds == [0] * 6


@pytest.mark.parametrize("case", range(9))
def test_packed_restatement_equals_plain(case):
    name, X, k = ragged_cases()[case]
    U, V, c = grecond(X, k)
    Up, Vp, cp = grecond_packed(X, k)
    assert np.array_equal(U, Up) and np.array_equal(V, Vp) and c == cp, name


def test_fit_without_gpu_fails_loudly():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    from pybmf_b200 import _native, models
    with pytest.raises(_native.NativeError):
        models.GreConD(k=2).fit(np.eye(4), save_model=False, show_logs=False, show_result=False)


def test_tol_and_k_are_checked():
    from pybmf_b200 import models
    with pytest.raises(NotImplementedError):
        models.GreConD(k=3, tol=0.1)
    for k in (0, -1, 1.5, True):
        with pytest.raises(ValueError):
            models.GreConD(k=k)
