"""CPU: the per-iteration exchange of pybmf_b200.expansion (one all-reduce of rank slots plus the words of the row chosen
last) for world = 1 .. 8, and a numpy simulation of the sharded loop over R ranks against the world-1 reference loop."""
import numpy as np
import pytest

from expansion_reference import (STOP, WEIGHTS, block_case, planted_case, random_case, reference_loop, sharded_loop,
                                 tie_case)
from pybmf_b200.engine import ShardPlan
from pybmf_b200.expansion import exchange_layout, merge_slots, pack_slot


def _summed(world, per_rank):
    """The SUM over the ranks of buffers in which every rank fills only its own slot."""
    bufs = []
    for rank in range(world):
        b = np.zeros(exchange_layout(world, 2)["size"], np.int64)
        pack_slot(b, rank, *per_rank[rank])
        bufs.append(b)
    return np.sum(bufs, axis=0)


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("words", [2, 4, 278])
def test_layout_tiles_the_buffer(world, words):
    L = exchange_layout(world, words)
    spans = [L["slots"], L["row_pos"], L["row_neg"]]
    assert spans[0][0] == 0 and spans[-1][1] == L["size"] == 2 * world + 2 * words
    assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
    assert L["row_pos"][1] - L["row_pos"][0] == L["row_neg"][1] - L["row_neg"][0] == words


@pytest.mark.parametrize("world", range(1, 9))
def test_merge_is_the_first_argmax_of_the_concatenation(world):
    rng = np.random.RandomState(world)
    for trial in range(200):
        m = int(rng.choice([1, 100, 256, 300, 513, 2000]))
        bounds = ShardPlan(m, world).bounds
        # few distinct values, so that ties across ranks are common; sometimes every delta is negative except +0.0 in u
        d = rng.choice([-1.5, -0.5, 0.0, 0.25, 0.75], size=m) if trial % 3 else -rng.randint(1, 4, size=m) * 0.5
        if trial % 3 == 0 and trial % 2:
            d[rng.randint(m)] = 0.0
        per_rank = [(d[a:b].max(), a + int(d[a:b].argmax())) if b > a else (0.0, -1) for a, b in bounds]
        score, index = merge_slots(_summed(world, per_rank), world)
        assert (score, index) == (d.max(), int(d.argmax())), (world, m, trial)


def test_merge_ties_ranks_without_rows_and_negative_maxima():
    # equal maxima on ranks 3, 1 and 5: the lowest row wins, whatever the rank order
    s = _summed(6, [(-1.0, 0), (0.5, 300), (0.25, 600), (0.5, 290 + 600), (-1.0, -1), (0.5, 2000)])
    assert merge_slots(s, 6) == (0.5, 300)
    # every delta negative: the max is the maximum negative value, not 0 of an empty rank
    s = _summed(4, [(-2.0, 7), (-0.5, 260), (0.0, -1), (0.0, -1)])
    assert merge_slots(s, 4) == (-0.5, 260)
    # +0.0 of a row in u beats negative deltas of lower rows on other ranks
    s = _summed(3, [(-0.5, 0), (0.0, 256), (0.0, 512)])
    assert merge_slots(s, 3) == (0.0, 256)
    # one rank only
    assert merge_slots(_summed(1, [(3.0, 9)]), 1) == (3.0, 9)


CASES = [("planted_1000x300", lambda w: planted_case(1000, 300, *w, seed=9)),
         ("planted_700x130", lambda w: planted_case(700, 130, *w, seed=4)),
         ("planted_33x1000", lambda w: planted_case(33, 1000, *w, seed=1033)),
         ("block_65", lambda w: block_case(600, 300, 65, *w, seed=3)),
         ("random_u_empty", lambda w: random_case(520, 70, *w, seed=2, u_mode="empty")),
         ("random_u_all", lambda w: random_case(520, 70, *w, seed=2, u_mode="all")),
         ("random_v_all", lambda w: random_case(520, 70, *w, seed=2, v_mode="all"))]


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("name,make", CASES, ids=[c[0] for c in CASES])
def test_sharded_simulation_equals_world_one_loop(name, make, world):
    for w in WEIGHTS:
        X, O, u, v, w_fp, w_fn = make(w)
        want = reference_loop(X, O, u, v, w_fp, w_fn)
        assert want[-1] == (STOP, -1)
        assert sharded_loop(X, O, u, v, w_fp, w_fn, world) == want, (name, world, w)


def test_reference_cases_cover_long_runs_stretch_edges_and_ties():
    """The GPU tests rely on these run lengths: >= 200 iterations, exactly one stretch (64) and one more, and a stop on
    r_score == c_score > 0."""
    assert len(reference_loop(*planted_case(33, 1000, 0.2, 0.8, seed=1033))) >= 200
    assert len(reference_loop(*block_case(600, 4100, 64, 0.5, 0.5, seed=3))) == 64
    assert len(reference_loop(*block_case(600, 4100, 65, 0.5, 0.5, seed=3))) == 65
    X, O, u, v = tie_case(70, 130)
    assert reference_loop(X, O, u, v, 0.3, 0.6) == [(STOP, -1)]
