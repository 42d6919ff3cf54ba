"""GPU: prediction-task splits on the device -- generate.DeviceEntries (stored ones and stored zeros), the host packers,
generate.ratio_split, the one-pass stored-entry count kernels, and fits / eval with DeviceEntries splits against the
same entries as host csr with explicitly stored zeros (ragged shapes: n not a multiple of 64, m not a multiple of 256;
weights 0.5 and 0.2)."""
import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp

from split_reference import ratio_split_rows, stored_csr

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

FIT_KW = dict(task="prediction", save_model=False, show_logs=False, show_result=False)
M_, N_ = 1000, 701
WEIGHTS = [0.5, 0.2]
NAMES = ["TP", "FP", "TN", "FN", "TPR", "FPR", "TNR", "FNR", "PPV", "ACC", "ERR", "F1", "Recall", "Precision"]


@pytest.fixture(scope="module")
def env():
    from pybmf_b200 import _native, device, generate, models, utils
    _native.require_gpu()
    models.SILENT = True
    X = generate.planted_bits(M_, N_, 5, 0.2, 0.15, 0.2, 0.03, seed=3)
    train, val, test = generate.ratio_split(X, 0.1, 0.15, neg_ratio=1.0, seed=7)
    d = {"train": train, "val": val, "test": test}
    h = {name: S.to_csr() for name, S in d.items()}
    return generate, models, utils, device, X, d, h


def _dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def _log(df):
    return df.loc[:, [c for c in df.columns if "time" not in c]]


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def _stored(A):
    """(row, col, value != 0) of the stored entries of a csr, in canonical order."""
    A = sp.csr_matrix(A)
    A.sum_duplicates()
    c = A.tocoo()
    return c.row.tolist(), c.col.tolist(), (c.data != 0).tolist()


def _bits(device, dense):
    return torch.from_numpy(device.dense_to_words(dense.astype(np.uint8))).cuda()


def test_host_round_trips(env):
    generate, models, utils, device, X, d, h = env
    rng = np.random.default_rng(1)
    dense = (rng.random((M_, N_)) < 0.1).astype(np.int64)
    H = stored_csr(dense != 0, (dense == 0) & (rng.random((M_, N_)) < 0.05))
    assert H.nnz > (dense != 0).sum()
    E = generate.entries_from_host(H)
    assert (E.shape, E.m, E.n, E.r0, E.r1) == ((M_, N_), M_, N_, 0, M_)
    assert _stored(E.to_csr()) == _stored(H) and E.to_csr().dtype == np.int64
    B = generate.bits_from_host(H)
    assert np.array_equal(_dense(B.to_csr()), dense) and B.to_csr().nnz == (dense != 0).sum()
    assert np.array_equal(_dense(generate.bits_from_host(dense).to_csr()), dense)                # ndarray input
    assert generate.entries_from_host(dense).zeros.to_csr().nnz == 0
    for S in (E.ones, E.zeros, B):
        words = S.bits.cpu().numpy()
        assert not device.words_to_dense(words, words.shape[1] * 64)[:, N_:].any()              # pad bits stay zero


def _entries_case(k, m, n, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((m, n)) < 0.2
    z = ~x & (rng.random((m, n)) < 0.1)
    U = rng.random((m, k)) < 0.08
    U[0] = False                                                   # a row that uses no factor
    U[1] = True                                                    # a row that uses every factor
    V = rng.random((n, k)) < 0.15
    P = (U.astype(np.int64) @ V.T.astype(np.int64)) > 0
    return x, z, U, V, P


@pytest.mark.parametrize("k", [1, 5, 64, 65, 130])
@pytest.mark.parametrize("m,n", [(M_, N_), (300, 20001)])
@pytest.mark.parametrize("with_zeros", [True, False])
def test_entry_count_kernels(env, k, m, n, with_zeros):
    generate, models, utils, device, X, d, h = env
    from pybmf_b200 import _native
    x, z, U, V, P = _entries_case(k, m, n, seed=k + m)
    if not with_zeros:
        z = np.zeros_like(z)
    want = [int((x & P).sum()), int((z & P).sum()), int(x.sum()), int(z.sum())]
    words = device.words_for(n)
    xb, zb = _bits(device, x), (_bits(device, z) if with_zeros else None)
    counts = torch.zeros(4, dtype=torch.int64, device="cuda")
    _native.call("bmf_confusion_entries_bits", xb, zb, _bits(device, P), m, words, counts)
    assert counts.cpu().tolist() == want
    uw, kw = utils._factor_words(sp.csr_matrix(U.astype(np.int64)))
    vt = utils._bits_on_device(sp.csr_matrix(V.T.astype(np.int64)))
    counts.fill_(-1)
    _native.call("bmf_confusion_entries_factors", xb, zb, m, words, uw, kw, vt, k, counts)
    assert counts.cpu().tolist() == want


def _fits(models, X, w, kw=FIT_KW):
    mdl = models.Asso(tau=0.4, k=5, w_fp=w)
    mdl.fit(X["train"], X["val"], X["test"], **kw)
    U0, V0, log0 = _dense(mdl.U), _dense(mdl.V), mdl.logs["updates"]
    it = models.AssoIter(model=mdl, w_fp=w)
    it.fit(X["train"], X["val"], X["test"], **kw)
    return U0, V0, log0, _dense(it.U), it.logs.get("refinements")


def _assert_same_fits(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[3], b[3])
    pd.testing.assert_frame_equal(_log(a[2]), _log(b[2]))
    assert (a[4] is None) == (b[4] is None)
    if a[4] is not None:
        pd.testing.assert_frame_equal(_log(a[4]), _log(b[4]))


@pytest.mark.parametrize("w", WEIGHTS)
def test_fits_with_device_entries_splits(env, w):
    generate, models, utils, device, X, d, h = env
    host_train = dict(h)                                           # same train (host csr), splits on the device or host
    dev_splits = dict(h, val=d["val"], test=d["test"])
    got, want = _fits(models, dev_splits, w), _fits(models, host_train, w)
    _assert_same_fits(got, want)
    assert ("val", 0, "F1") in got[2].columns and ("test", 0, "F1") in got[2].columns
    # the last log row of the fit equals the host triplet path of eval on the final factors
    mdl = models.Asso(tau=0.4, k=5, w_fp=w)
    mdl.fit(dev_splits["train"], d["val"], **FIT_KW)
    last = mdl.logs["updates"].iloc[-1]
    row = utils.eval(["TP", "FP", "FN", "F1"], "prediction", X_gt=h["val"], U=mdl.U, V=mdl.V)
    assert [float(last[("val", 0, c)]) for c in ("TP", "FP", "FN", "F1")] == [float(v) for v in row]


@pytest.mark.parametrize("w", WEIGHTS)
def test_transposed_model_with_device_entries(env, w):
    generate, models, utils, device, X, d, h = env
    got = []
    for val in (d["val"], h["val"]):
        tm = models.TransposedModel(models.Asso(tau=0.4, k=4, w_fp=w))
        tm.fit(h["train"], val, **FIT_KW)
        got.append((_dense(tm.U), _dense(tm.V), tm.model.logs["updates"]))
    assert np.array_equal(got[0][0], got[1][0]) and np.array_equal(got[0][1], got[1][1])
    pd.testing.assert_frame_equal(_log(got[0][2]), _log(got[1][2]))
    tm = models.TransposedModel(models.Asso(tau=0.4, k=4, w_fp=w))
    tm.fit(d["train"], d["val"], d["test"], **FIT_KW)                # all three on the device, transposed there
    ref = models.TransposedModel(models.Asso(tau=0.4, k=4, w_fp=w))
    ref.fit(h["train"], h["val"], h["test"], **FIT_KW)
    assert np.array_equal(_dense(tm.U), _dense(ref.U)) and np.array_equal(_dense(tm.V), _dense(ref.V))
    pd.testing.assert_frame_equal(_log(tm.model.logs["updates"]), _log(ref.model.logs["updates"]))


@pytest.mark.parametrize("w", WEIGHTS)
def test_devicebits_train_under_prediction(env, w):
    """A DeviceBits X_train under task='prediction' counts its ones as its stored entries, like a host csr of them."""
    generate, models, utils, device, X, d, h = env
    got = _fits(models, dict(d), w)
    want = _fits(models, dict(h), w)
    _assert_same_fits(got, want)
    tp_fp = got[2][[("train", 0, "FP")]].to_numpy().astype(np.int64)
    assert (tp_fp == 0).all()                                      # no stored zeros: nothing to predict falsely


@pytest.mark.parametrize("w", WEIGHTS)
def test_device_entries_train(env, w):
    generate, models, utils, device, X, d, h = env
    train = generate.DeviceEntries(d["train"], d["val"].zeros)      # the val negatives stored as zeros of train
    ht = train.to_csr()
    assert ht.nnz > d["train"].to_csr().nnz
    for task in ("prediction", "reconstruction"):
        kw = dict(FIT_KW, task=task)
        _assert_same_fits(_fits(models, dict(d, train=train), w, kw), _fits(models, dict(h, train=ht), w, kw))


def test_eval_both_tasks(env):
    generate, models, utils, device, X, d, h = env
    mdl = models.Asso(tau=0.4, k=5, w_fp=0.5)
    mdl.fit(h["train"], **dict(FIT_KW, task="reconstruction"))
    for task in ("prediction", "reconstruction"):
        for split in ("val", "test"):
            got = utils.eval(NAMES, task, X_gt=d[split], U=mdl.U, V=mdl.V)
            want = utils.eval(NAMES, task, X_gt=h[split], U=mdl.U, V=mdl.V)
            assert all(_same(a, b) for a, b in zip(got, want)), (task, split, got, want)


@pytest.mark.parametrize("m,n,p", [(M_, N_, 0.2), (257, 65, 0.5), (300, 20001, 0.05)])
def test_ratio_split_bit_for_bit(env, m, n, p):
    generate, models, utils, device, X, d, h = env
    Xs = generate.random_bits(m, n, p, seed=m)
    x = _dense(Xs.to_csr()).astype(bool)
    train, val, test = generate.ratio_split(Xs, 0.1, 0.2, neg_ratio=1.5, seed=9)
    th = generate.split_thresholds(int(x.sum()), m, n, 0.1, 0.2, 1.5)
    want = ratio_split_rows(x, 0, n, 9, th)
    got = [train, val.ones, val.zeros, test.ones, test.zeros]
    for g, w_ in zip(got, want):
        assert (g.m, g.n, g.r0, g.r1) == (m, n, 0, m)
        assert np.array_equal(_dense(g.to_csr()).astype(bool), w_)
        words = g.bits.cpu().numpy()
        assert not device.words_to_dense(words, words.shape[1] * 64)[:, n:].any()             # pad bits zero
    tr, v1, v0, s1, s0 = (_dense(g.to_csr()).astype(bool) for g in got)
    assert np.array_equal(tr | v1 | s1, x) and not (tr & v1).any() and not (tr & s1).any() and not (v1 & s1).any()
    assert not ((v0 | s0) & x).any() and not (v0 & s0).any()


def test_ratio_split_negatives_above_l2(env):
    """40000 x 30001 bits (150 MB a matrix, above the 126 MB L2): the counts of the parts lie within six standard
    deviations of their binomial means."""
    generate, models, utils, device, X, d, h = env
    m, n = 40000, 30001
    Xs = generate.random_bits(m, n, 0.01, seed=5)
    train, val, test = generate.ratio_split(Xs, 0.1, 0.1, neg_ratio=2.0, seed=3)
    pop = lambda S: utils.confusion_counts(S, S)[0]
    n1 = pop(train) + pop(val.ones) + pop(test.ones)
    zeros = m * n - n1
    t_v, t_t, q_v, q_t = generate.split_thresholds(n1, m, n, 0.1, 0.1, 2.0)
    for got, trials, thr in ((pop(val.ones), n1, t_v), (pop(test.ones), n1, t_t), (pop(val.zeros), zeros, q_v),
                             (pop(test.zeros), zeros, q_t)):
        p_ = thr / 2.0 ** 32
        mean, sd = trials * p_, (trials * p_ * (1 - p_)) ** 0.5
        assert abs(got - mean) < 6 * sd, (got, mean, sd)
    assert abs(pop(val.zeros) / pop(val.ones) - 2.0) < 0.05


def test_errors(env):
    generate, models, utils, device, X, d, h = env
    for args in ((-0.1, 0.1), (0.1, 1.1), (0.6, 0.5)):
        with pytest.raises(ValueError):
            generate.ratio_split(X, *args)
    with pytest.raises(ValueError):
        generate.ratio_split(X, 0.1, 0.1, neg_ratio=-1.0)
    dense = generate.random_bits(300, 70, 0.9, seed=1)
    with pytest.raises(ValueError):
        generate.ratio_split(dense, 0.3, 0.3, neg_ratio=1.0)        # too few zeros
    other_rows = generate.planted_bits(M_, N_, 5, 0.2, 0.15, 0.2, 0.03, seed=4, rank=1, world=2)
    other_shape = generate.planted_bits(M_, N_ + 1, 5, 0.2, 0.15, 0.2, 0.03, seed=4)
    for bad in (other_rows, other_shape):
        with pytest.raises(ValueError):
            generate.DeviceEntries(d["train"], bad)
    with pytest.raises(ValueError):
        generate.DeviceEntries(other_rows, other_rows)              # rows of rank 1 of 2 in a 1-process run
    wrong_shape = generate.DeviceEntries(other_shape, other_shape)
    with pytest.raises(ValueError):
        models.Asso(tau=0.4, k=3).fit(h["train"], wrong_shape, **FIT_KW)
    with pytest.raises(ValueError):
        models.TransposedModel(models.Asso(tau=0.4, k=3)).fit(d["train"], None, wrong_shape, **FIT_KW)
    with pytest.raises(ValueError):                                 # a plain DeviceBits SPLIT still has no stored zeros
        models.Asso(tau=0.4, k=3).fit(h["train"], d["val"].ones, **FIT_KW)
    mdl = models.Asso(tau=0.4, k=3)
    mdl.fit(h["train"], **FIT_KW)
    with pytest.raises(TypeError):
        utils.eval(["F1"], "prediction", X_gt=d["val"], X_pd=h["val"])
    with pytest.raises(TypeError):
        utils.eval(["F1"], "prediction", X_gt=h["val"], X_pd=d["val"])
    with pytest.raises(TypeError):
        utils.eval(["F1"], "prediction", X_gt=d["val"], X_pd=d["val"], U=mdl.U, V=mdl.V)
    with pytest.raises(ValueError):
        utils.eval(["F1"], "prediction", X_gt=d["val"].ones, U=mdl.U, V=mdl.V)
    E = d["val"]
    for call in (lambda: utils.confusion_counts(E, E), lambda: utils.confusion_counts(E, d["train"]),
                 lambda: utils.TP(E, h["val"]), lambda: utils.F1(E, E), lambda: utils.coverage_score(E, E),
                 lambda: utils.weighted_error(E, E), lambda: utils.get_metrics(E, E, ["F1"]),
                 lambda: utils.get_metrics(h["val"], E, ["F1"]), lambda: utils.description_length(E, mdl.U, mdl.V),
                 lambda: utils.factor_counts(E, mdl.U, mdl.V), lambda: utils.matmul(E, E, boolean=True)):
        with pytest.raises(TypeError):
            call()
