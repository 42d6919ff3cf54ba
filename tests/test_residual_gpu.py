"""GPU: the one-pass residual kernel (bmf_residual_factors), utils.get_residual on host matrices and on generate.DeviceBits,
and generate.prediction -- against numpy on ragged shapes, in every kernel form (BMF_NO_PANEL x BMF_PANEL_DYNAMIC) and
against the two-kernel path (bmf_bool_product + bmf_bits_combine op 2), at c5 scale, through a genuine GreConD run on
the device (tests/golden/grecond.npz), chained into the GreConD+ expansion, and in every error case."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import GOLDEN
from expansion_reference import SHAPES, WEIGHTS, reference_loop

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

# (m, n, k): the copy case (k = 0), the panel-list form (k <= 64), kw = 2 on the row stream (k > 64), the two-chunk panel
# (n = 20010), many panels (n = 33000) and many 32-row blocks (m = 150001)
KERNEL_SHAPES = [(1, 64, 1), (50, 70, 0), (300, 500, 5), (257, 129, 64), (100, 200, 70), (777, 1000, 128),
                 (1501, 20010, 20), (2500, 33000, 17), (150001, 130, 5)]
FORMS = [("0", "0"), ("0", "1"), ("1", "0"), ("1", "1")]              # (BMF_NO_PANEL, BMF_PANEL_DYNAMIC)


@pytest.fixture(scope="module")
def L():
    from pybmf_b200 import _native, device, expansion, generate, models, utils
    _native.require_gpu()
    models.SILENT = True
    return _native, device, generate, utils, expansion


def _dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def _factors(rng, m, n, k):
    """U (m x k) with rows that use no factor, one factor, eight or more (the bit-scan branch of the list kernel) and
    every factor; the other rows use about two.  V (n x k) at density 0.1."""
    U = rng.random((m, k)) < min(1.0, 2.0 / max(k, 1))
    if k:
        special = [np.zeros(k, bool), np.eye(k, dtype=bool)[k // 2], np.arange(k) % max(1, k // 8) == 0,
                   np.ones(k, bool)]
        for i, row in enumerate(special[:m]):
            U[i] = row
    V = rng.random((n, k)) < 0.1
    return U, V


def _residual_np(X, U, V):
    P = (U.astype(np.int64) @ V.T.astype(np.int64)) > 0 if U.shape[1] else np.zeros(X.shape, bool)
    return (X != 0) & ~P


@pytest.mark.parametrize("m,n,k", KERNEL_SHAPES)
def test_kernel_forms_against_numpy_and_two_pass(L, monkeypatch, m, n, k):
    _native, device, _generate, utils, _e = L
    rng = np.random.default_rng(m * 7 + n + k)
    X = rng.random((m, n)) < 0.3
    U, V = _factors(rng, m, n, k)
    uw, kw = utils._factor_words(sp.csr_matrix(U))
    vt = utils._bits_on_device(sp.csr_matrix(V.T))
    x = utils._bits_on_device(sp.csr_matrix(X))
    words = x.shape[1]
    want = device.dense_to_words(_residual_np(X, U, V), words)        # pad words and bits are zero
    pd = device.zeros((m, words), torch.int64)
    _native.call("bmf_bool_product", uw, m, kw, vt, k, words, pd)
    two = device.zeros((m, words), torch.int64)
    _native.call("bmf_bits_combine", x, pd, m, words, 2, two)
    assert np.array_equal(two.cpu().numpy(), want)
    for no_panel, dynamic in FORMS:
        monkeypatch.setenv("BMF_NO_PANEL", no_panel)
        monkeypatch.setenv("BMF_PANEL_DYNAMIC", dynamic)
        out = torch.full((m, words), -1, dtype=torch.int64, device="cuda")  # an unwritten word shows up
        _native.call("bmf_residual_factors", x, m, words, uw, kw, vt, k, out)
        assert torch.equal(out, two), (m, n, k, no_panel, dynamic)


def test_kernel_argument_checks(L):
    _native, device, _generate, _utils, _e = L
    x = device.zeros((4, 2), torch.int64)
    uw = device.zeros((4, 1), torch.int64)
    vt = device.zeros((1, 2), torch.int64)
    out = device.zeros((4, 2), torch.int64)
    for args in ((x, 4, 2, uw, 1, vt, 1, x), (None, 4, 2, uw, 1, vt, 1, out), (x, 4, 3, uw, 1, vt, 1, out),
                 (x, 4, 2, uw, 1, vt, 65, out), (x, 4, 2, uw, 1, None, 1, out), (x, 0, 2, uw, 1, vt, 1, out)):
        with pytest.raises(ValueError):
            _native.call("bmf_residual_factors", *args)


def test_c5_scale_residual_properties(L, monkeypatch):
    """200k x 100k bits, k = 64 (as test_c5_scale_panel_kernels_properties): panel form == row-stream form == product +
    combine, and |residual| = |X| - TP(X, product)."""
    _native, device, _generate, _utils, _e = L
    m, n, k = 200_000, 100_000, 64
    words = device.words_for(n)
    g = torch.Generator(device="cuda"); g.manual_seed(11)

    def rnd(shape, ands):
        w = torch.randint(-2 ** 63, 2 ** 63 - 1, shape, dtype=torch.int64, device="cuda", generator=g)
        for _ in range(ands - 1):
            w &= torch.randint(-2 ** 63, 2 ** 63 - 1, shape, dtype=torch.int64, device="cuda", generator=g)
        return w

    def mask(b):
        b[:, n // 64] &= (1 << (n % 64)) - 1
        b[:, (n + 63) // 64:] = 0
        return b
    uw = rnd((m, 1), 5)
    vt = mask(rnd((k, words), 5))
    pd = device.zeros((m, words), torch.int64)
    _native.call("bmf_bool_product", uw, m, 1, vt, k, words, pd)
    x = mask(pd ^ rnd((m, words), 4))
    two = device.zeros((m, words), torch.int64)
    _native.call("bmf_bits_combine", x, pd, m, words, 2, two)
    c = device.zeros((3,), torch.int64)
    _native.call("bmf_confusion_bits", x, pd, m, words, -1, c, None, None)
    tp, _fp, fn = (int(v) for v in c.cpu().numpy())
    del pd
    out = device.zeros((m, words), torch.int64)
    for env in ("0", "1"):
        monkeypatch.setenv("BMF_NO_PANEL", env)
        out.fill_(-1)
        _native.call("bmf_residual_factors", x, m, words, uw, 1, vt, k, out)
        assert torch.equal(out, two), env
    cr = device.zeros((3,), torch.int64)
    _native.call("bmf_confusion_bits", out, out, m, words, -1, cr, None, None)
    assert int(cr[0].item()) == (tp + fn) - tp


def test_host_get_residual(L):
    _native, device, _generate, utils, _e = L
    rng = np.random.default_rng(3)
    for (m, n) in ((1, 1), (70, 130), (257, 65), (600, 4100)):
        for k in (0, 5, 70):
            X = (rng.random((m, n)) < 0.3).astype(np.int64)
            U, V = _factors(rng, m, n, k)
            want = _residual_np(X, U, V)
            for Xin, dt in ((X, np.int64), (sp.csr_matrix(X.astype(np.float64)), np.float64)):
                R = utils.get_residual(Xin, sp.lil_matrix(U.astype(float)), sp.lil_matrix(V.astype(float)))
                assert sp.isspmatrix_lil(R) and R.dtype == dt and R.shape == (m, n)
                assert np.array_equal(_dense(R), want), (m, n, k)
    X = np.ones((5, 4), np.int64)
    with pytest.raises(AssertionError, match="multiplicable"):
        utils.get_residual(X, np.ones((5, 3)), np.ones((4, 2)))
    with pytest.raises(AssertionError):
        utils.get_residual(X, np.ones((6, 2)), np.ones((4, 2)))


def test_prediction_against_host(L):
    _native, device, generate, utils, _e = L
    rng = np.random.default_rng(4)
    for (m, n, k) in ((1, 1, 1), (70, 130, 0), (257, 65, 5), (600, 4100, 70), (1501, 20010, 20)):
        U, V = _factors(rng, m, n, k)
        want = _dense(utils.get_prediction(sp.csr_matrix(U.astype(np.int64)), sp.csr_matrix(V.astype(np.int64))))
        for conv in (np.asarray, sp.csr_matrix, sp.lil_matrix):
            P = generate.prediction(conv(U.astype(float)), conv(V.astype(float)))
            assert (P.shape, P.r0, P.r1) == ((m, n), 0, m)
            assert np.array_equal(_dense(P.to_csr()), want), (m, n, k)
            assert not device.words_to_dense(P.bits.cpu().numpy(), P.bits.shape[1] * 64)[:, n:].any()
        # a rank's rows are the matching rows of the one-process result, whatever the number of ranks
        for world in (2, 3):
            for rank in range(world):
                S = generate.prediction(U, V, rank=rank, world=world)
                if S.r1 > S.r0:
                    assert np.array_equal(_dense(S.to_csr()), want[S.r0:S.r1])
    S = generate.prediction(np.ones((200, 3)), np.ones((9, 3)), rank=1, world=2)       # m <= 256: rank 1 has no rows
    assert (S.m, S.n, S.r0, S.r1) == (200, 9, 200, 200)


def test_grecond_run_on_device(L):
    """The factors of a genuine GreConD run, pushed through the utils its call sites use, with X a generate.DeviceBits:
    the device counterpart of test_grecond_call_sites_through_routed_utils."""
    _native, device, generate, U_, _e = L
    g = np.load(os.path.join(GOLDEN, "grecond.npz"))
    X = generate.bits_from_host(g["X"])
    U, V = sp.lil_matrix(g["U"].astype(float)), sp.lil_matrix(g["V"].astype(float))
    for t in range(g["U"].shape[1]):
        Ut, Vt = sp.lil_matrix(U[:, : t + 1]), sp.lil_matrix(V[:, : t + 1])
        X_pd = generate.prediction(Ut, Vt)
        X_rs = U_.get_residual(X, Ut, Vt)
        assert isinstance(X_rs, generate.DeviceBits) and (X_rs.shape, X_rs.r0, X_rs.r1) == (X.shape, X.r0, X.r1)
        assert float(U_.ERR(gt=X, pd=X_pd)) == g["step_ERR"][t]
        assert float(U_.weighted_error(gt=X, pd=X_pd, w_fp=0.3, w_fn=0.7)) == g["step_weighted_error"][t]
        assert float(U_.description_length(gt=X, U=Ut, V=Vt, w_model=1.0, w_fp=1.0, w_fn=1.0)) == g["step_desc_len"][t]
        assert float(U_.coverage_score(gt=X, pd=X_pd, w_fp=0.5)) == g["step_coverage"][t]
        assert float(X_rs.to_csr().sum()) == g["step_rs_sum"][t] and float(X_pd.to_csr().sum()) == g["step_pd_sum"][t]
        got = U_.get_metrics(gt=X, pd=X_pd, metrics=["Recall", "Precision", "Accuracy", "F1"])
        assert [float(v) for v in got] == [float(g["log_" + c][t]) for c in ("Recall", "Precision", "Accuracy", "F1")]
    assert np.array_equal(_dense(generate.prediction(U, V).to_csr()), g["X_pd"])
    assert np.array_equal(_dense(U_.get_residual(X, U, V).to_csr()), g["X_rs"])


@pytest.mark.parametrize("m,n", SHAPES)
def test_residual_feeds_expansion(L, m, n):
    """expansion(X, get_residual(X, U, V), u, v) on DeviceBits equals the host chain, and its log equals the numpy loop
    on the numpy residual."""
    _native, _device, generate, utils, E = L
    rng = np.random.RandomState(m * n)
    X = (rng.rand(m, n) < 0.3).astype(np.int64)
    U = (rng.rand(m, 3) < 0.3).astype(np.int64)
    V = (rng.rand(n, 3) < 0.3).astype(np.int64)
    u, v = (rng.rand(m) < 0.3).astype(np.int64), (rng.rand(n) < 0.3).astype(np.int64)
    O = _residual_np(X, U, V).astype(np.int64)
    Xd = generate.bits_from_host(X)
    Rd = utils.get_residual(Xd, U, V)
    Rh = utils.get_residual(sp.csr_matrix(X), U, V)
    assert np.array_equal(_dense(Rd.to_csr()), O) and np.array_equal(_dense(Rh), O)
    for (w_fp, w_fn) in WEIGHTS:
        want = np.array(reference_loop(X, O, u, v, w_fp, w_fn), dtype=np.int64).reshape(-1, 2)
        assert np.array_equal(E.expansion_log(Xd, Rd, u.reshape(-1, 1), v.reshape(-1, 1), w_fp, w_fn), want)
        a, b = (E.expansion(Xg, Og, sp.lil_matrix(u.reshape(-1, 1)), sp.lil_matrix(v.reshape(-1, 1)), w_fp, w_fn)
                for Xg, Og in ((Xd, Rd), (sp.csr_matrix(X), sp.csr_matrix(Rh))))
        assert all(np.array_equal(_dense(p), _dense(q)) for p, q in zip(a, b)), (m, n, w_fp)


def test_error_cases(L):
    _native, _device, generate, utils, _e = L
    m, n = 300, 70
    rng = np.random.default_rng(9)
    X = (rng.random((m, n)) < 0.3).astype(np.int64)
    U, V = np.ones((m, 2)), np.ones((n, 2))
    with pytest.raises(TypeError):
        utils.get_residual(generate.entries_from_host(sp.csr_matrix(X)), U, V)
    Xd = generate.bits_from_host(X)
    for Ub, Vb in ((np.ones((m + 1, 2)), V), (U, np.ones((n - 1, 2))), (U, np.ones((n, 3)))):
        with pytest.raises(ValueError, match="do not fit"):
            utils.get_residual(Xd, Ub, Vb)
    with pytest.raises(ValueError):
        utils.get_residual(generate.DeviceBits(Xd.bits[:256], m, n, 0, 256), U, V)
    with pytest.raises(ValueError):
        generate.prediction(U, np.ones((n, 3)))
