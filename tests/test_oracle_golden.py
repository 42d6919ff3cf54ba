"""CPU: pin the oracle restatement (oracle/asso_oracle.py) against
 (a) the known-answer table stored in PyBMF's examples/ex01_6_logs.ipynb:253-361,
 (b) outputs of the genuine reference (tests/golden/*.npz, made by oracle/make_golden.py)."""
import numpy as np
import pytest

from conftest import GOLDEN_CASES, LOG_COLS, load_golden
from oracle import asso_oracle as O


def _run_oracle(c):
    try:
        return O.asso_fit(c["X"], c["k"], c["tau"], c["w_fp"], c["w_fn"]), ""
    except O.NoCandidateError as e:
        return e.args[1], "TypeError"


def test_known_answer_table_ex01_6():
    # numbers typed from the notebook's stored output, not from our fixture
    c = load_golden("ex01_6")
    assert int(c["X"].sum()) == 39251                        # ex01_6_logs.ipynb:100
    r, _ = _run_oracle(c)
    logs = r["logs"]
    assert [l["score"] for l in logs] == [817.5, 1564.5, 2182.5, 2797.5, 2953.0]
    assert [l["shape"] for l in logs] == [[71, 151], [63, 152], [24, 226], [24, 223], [23, 189]]
    assert [l["TP"] for l in logs] == [6178, 11713, 15043, 18334, 18938]
    assert [l["FP"] for l in logs] == [4543, 8584, 10678, 12739, 13032]
    assert logs[0]["desc_len"] == 37838.0 and logs[-1]["desc_len"] == 34491.0


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_matches_reference_outputs(name):
    c = load_golden(name)
    g = c["g"]
    r, err = _run_oracle(c)
    assert err == c["error"]
    assert r["U"].shape == g["U"].shape and np.array_equal(r["U"], g["U"])
    assert r["V"].shape == g["V"].shape and np.array_equal(r["V"], g["V"])
    for col in LOG_COLS:                                       # bit-exact, including the fp64 rates
        got = np.array([l[col] for l in r["logs"]], dtype=np.float64)
        assert np.array_equal(got, g["log_" + col]), col
    assert np.array_equal(np.array([l["shape"] for l in r["logs"]]).reshape(-1, 2), g["log_shape"])


@pytest.mark.parametrize("name", ["ex01_6", "c1_noisy", "planted_w02", "planted_w025"])
def test_oracle_assoiter_matches_reference(name):
    c = load_golden(name)
    g = c["g"]
    r, _ = _run_oracle(c)
    it = O.asso_iter_fit(c["X"], r["U"], r["V"], c["k"], c["w_fp"], c["w_fn"])
    trace = np.array([(col, int(acc)) for col, acc in it["trace"]], dtype=np.int64).reshape(-1, 2)
    assert np.array_equal(trace, g["iter_trace"])
    assert np.array_equal(it["U"], g["iter_U"])
    if "iter_score" in g.files:
        assert np.array_equal(np.array([x["score"] for x in it["refinements"]]), g["iter_score"])
        assert np.array_equal(np.array([x["error"] for x in it["refinements"]]), g["iter_error"])
        for col in ["Recall", "Precision", "Accuracy", "F1"]:
            assert np.array_equal(np.array([x[col] for x in it["refinements"]]), g["iter_" + col])
    else:
        assert it["refinements"] == []


def test_d1_truncation_quirk():
    c = load_golden("c1_clean")
    r, _ = _run_oracle(c)
    assert r["U"].shape == (1000, 4) and len(r["logs"]) == 5 and r["logs"][-1]["ERR"] == 0.0


def test_integer_weight_form_equals_float_form():
    rng = np.random.RandomState(3)
    X = (rng.rand(70, 50) < 0.3).astype(np.uint8)
    C = (rng.rand(70, 50) < 0.1).astype(np.uint8)
    B = (rng.rand(20, 50) < 0.3).astype(np.uint8)
    for w_fp, w_fn in [(0.5, None), (0.25, None), (0.375, 0.5), (1.0, 1.0)]:
        a, b, s = O.integer_weights(w_fp, w_fn)
        score, use, P, N, tpo, fpo = O.score_candidates(X, C, B, w_fp, w_fn)
        assert np.array_equal(use, (b * P - a * N) > 0)
        G = O.integer_gains(X, C, B, a, b)
        so = int((b * tpo - a * fpo).sum())
        assert np.array_equal(score, (so + G).astype(np.float64) / (1 << s))
    assert O.integer_weights(0.2, None) is None


# ---- the bit-packed C restatement (oracle/asso_c.c through oracle/asso_oracle_c.py) --------------------------
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_c_restatement_matches_reference_outputs(name):
    """The C restatement that writes the full-size fixtures is pinned against the genuine reference's golden outputs:
    U, V, TP / FP per step, scores (bit for bit for a/2^s weights, rtol 1e-12 otherwise), D1 truncation, D2 error."""
    import scipy.sparse as sp
    from oracle import asso_oracle_c as OC
    c = load_golden(name)
    g = c["g"]
    r = OC.asso_fit(sp.csr_matrix(c["X"]), c["k"], c["tau"], c["w_fp"], c["w_fn"])
    assert r["error"] == c["error"]
    m, n = c["X"].shape
    U = np.stack(r["U_cols"], 1) if r["U_cols"] else np.zeros((m, 0), np.uint8)
    V = np.stack(r["V_cols"], 1) if r["V_cols"] else np.zeros((n, 0), np.uint8)
    assert U.shape == g["U"].shape and np.array_equal(U, g["U"]) and np.array_equal(V, g["V"])
    if "log_TP" in g:
        assert [s["tp"] for s in r["steps"]] == list(g["log_TP"].astype(np.int64))
        assert [s["fp"] for s in r["steps"]] == list(g["log_FP"].astype(np.int64))
        sc = np.array([s["score"] for s in r["steps"]])
        if O.integer_weights(c["w_fp"], c["w_fn"]) is not None:
            assert np.array_equal(sc, g["log_score"])
        else:
            np.testing.assert_allclose(sc, g["log_score"], rtol=1e-12, atol=0)
    if "iter_U" in g:
        it = OC.asso_iter_fit(sp.csr_matrix(c["X"]), g["U"], g["V"], c["k"], c["w_fp"], c["w_fn"])
        assert np.array_equal(it["U"], g["iter_U"])
        assert np.array_equal(np.array([(a, int(b)) for a, b in it["trace"]]).reshape(-1, 2), g["iter_trace"])


@pytest.mark.parametrize("tau", [-0.25, 0.0, 1.0 / 3.0, 0.5, 1.0])
def test_c_restatement_basis_equals_numpy_restatement(tau):
    """Candidate basis of the two restatements, incl. an empty column (its association row is 0, Asso.py:211: every bit is
    set for a negative tau, none otherwise) and ratios exactly equal to tau."""
    import scipy.sparse as sp
    from oracle import asso_oracle_c as OC
    rng = np.random.RandomState(3)
    A = (rng.rand(90, 70) < 0.3).astype(np.uint8)
    A[:, 5] = 0
    A[:, 7] = A[:, 3]
    A[:45, 9] = 1; A[45:, 9] = 0; A[:, 11] = 0; A[:15, 11] = 1     # 15 / 45 = 1 / 3
    st = OC.BitState(sp.csr_matrix(A), tau)
    want = (O.build_assoc(A) > tau).astype(np.uint8)
    got = np.unpackbits(st.basis.view(np.uint8), axis=1, bitorder="little")[:, :70]
    assert np.array_equal(got, want)
    assert np.array_equal(st.pop, want.sum(axis=1)) and np.array_equal(st.alive, (want.sum(axis=1) != 0).astype(np.uint8))


def test_c2_fixture_is_reproduced_and_agrees_with_numpy_restatement():
    """tests/golden/c2_digest.json (BASELINE configs[1], full size, k = 20) is what the C restatement computes today, and
    its first greedy steps equal the dense numpy restatement's (the two share no code; k = 20 was compared once when the
    fixture was made: 82 s of numpy time)."""
    import json
    import os
    from conftest import GOLDEN
    from oracle import asso_oracle_c as OC
    from pybmf_b200 import synth
    X = synth.config_c2()
    want = json.load(open(os.path.join(GOLDEN, "c2_digest.json")))
    r = OC.asso_fit(X, 20, 0.5, 0.5)
    for key in ("winners", "score_bits", "used", "tp", "fp", "u_sha256", "v_sha256"):
        assert r["digest"][key] == want[key], key
    w = O.asso_fit(X, 2, 0.5, 0.5)
    U = np.stack(r["U_cols"], 1)
    assert np.array_equal(U[:, :2], w["U"]) and [l["score"] for l in w["logs"]] == [s["score"] for s in r["steps"][:2]]


def test_c2_general_weights_fixture_is_reproduced():
    """tests/golden/c2w02_digest.json (w_fp = 0.2): what the C restatement computes today; the first factors equal the numpy
    restatement's (whose per-row float sums may differ from the integer-total score in the last ulps, never in U / V here)."""
    import json
    import os
    from conftest import GOLDEN
    from oracle import asso_oracle_c as OC
    from pybmf_b200 import synth
    X = synth.config_c2()
    want = json.load(open(os.path.join(GOLDEN, "c2w02_digest.json")))
    r = OC.asso_fit(X, 20, 0.5, 0.2)
    for key in ("winners", "score_bits", "used", "tp", "fp", "u_sha256", "v_sha256"):
        assert r["digest"][key] == want[key], key
    assert want["winners"][:3] == [57, 20, 9]
    w = O.asso_fit(X, 2, 0.5, 0.2)
    U = np.stack(r["U_cols"], 1)
    assert np.array_equal(U[:, :2], w["U"])
    np.testing.assert_allclose([l["score"] for l in w["logs"]], [s["score"] for s in r["steps"][:2]], rtol=1e-12, atol=0)


def test_c4_fixture_is_self_consistent():
    """tests/golden/c4_digest.json (480189 x 17770, k = 20; 40 min of host time to regenerate): structural checks."""
    import json
    import os
    from conftest import GOLDEN
    d = json.load(open(os.path.join(GOLDEN, "c4_digest.json")))
    assert d["m"] == 480189 and d["n"] == 17770 and d["k"] == 20 and len(d["winners"]) == 20 and d["error"] == ""
    assert len(set(d["winners"])) == 20 and all(0 <= w < d["n"] for w in d["winners"])
    tp, fp = np.array(d["tp"]), np.array(d["fp"])
    assert (np.diff(tp) > 0).all() and (np.diff(fp) >= 0).all() and tp[-1] <= d["sum_x"] == d["nnz"]
    score = np.array([np.frombuffer(bytes.fromhex(h), dtype=np.float64)[0] for h in d["score_bits"]])
    assert np.array_equal(score, 0.5 * tp - 0.5 * fp)                # w = [0.5, 0.5]: score = coverage of the whole cover
    assert (np.diff(score) > 0).all()
