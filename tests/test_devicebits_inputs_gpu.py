"""GPU: device-generated, row-sharded matrices (generate.DeviceBits) as validation and test splits of Asso / AssoIter,
in the evaluation utils, in generate.transpose and in TransposedModel -- each against the same matrices downloaded as
host csr (ragged shapes: n not a multiple of 64, m not a multiple of 256; integer and non-dyadic weights)."""
import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

FIT_KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)
M_, N_ = 1000, 701
WEIGHTS = [0.5, 0.2]


@pytest.fixture(scope="module")
def env():
    from pybmf_b200 import _native, generate, models, utils
    _native.require_gpu()
    models.SILENT = True
    mats = {name: generate.planted_bits(M_, N_, 5, 0.2, 0.15, 0.2, 0.03, seed=seed)
            for name, seed in (("train", 3), ("val", 4), ("test", 5), ("pd", 6))}
    host = {name: X.to_csr() for name, X in mats.items()}
    return generate, models, utils, mats, host


def _dense(A):
    return (np.asarray(A.todense()) != 0).astype(np.uint8)


def _log(df):
    return df.loc[:, [c for c in df.columns if "time" not in c]]


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.mark.parametrize("w", WEIGHTS)
def test_asso_and_assoiter_with_device_splits(env, w):
    generate, models, utils, d, h = env
    fits = []
    for X in (d, h):
        mdl = models.Asso(tau=0.4, k=5, w_fp=w)
        mdl.fit(X["train"], X["val"], X["test"], **FIT_KW)
        U0, V0 = _dense(mdl.U), _dense(mdl.V)
        it = models.AssoIter(model=mdl, w_fp=w)
        it.fit(X["train"], X["val"], X["test"], **FIT_KW)
        fits.append((U0, V0, mdl.logs["updates"], _dense(it.U), it.logs.get("refinements")))
    (Ud, Vd, ld, Uid, rd), (Uh, Vh, lh, Uih, rh) = fits
    assert np.array_equal(Ud, Uh) and np.array_equal(Vd, Vh)
    assert ("val", 0, "F1") in ld.columns and ("test", 0, "F1") in ld.columns
    pd.testing.assert_frame_equal(_log(ld), _log(lh))
    assert np.array_equal(Uid, Uih)
    assert (rd is None) == (rh is None)
    if rd is not None:
        pd.testing.assert_frame_equal(_log(rd), _log(rh))


def test_device_split_with_host_train(env):
    generate, models, utils, d, h = env
    logs = []
    for val in (d["val"], h["val"]):
        mdl = models.Asso(tau=0.4, k=4, w_fp=0.5)
        mdl.fit(h["train"], val, **FIT_KW)
        logs.append(mdl.logs["updates"])
    pd.testing.assert_frame_equal(_log(logs[0]), _log(logs[1]))


@pytest.mark.parametrize("w", WEIGHTS)
def test_utils_counts_and_metrics(env, w):
    generate, models, utils, d, h = env
    mdl = models.Asso(tau=0.4, k=5, w_fp=w)
    mdl.fit(h["train"], **FIT_KW)
    U, V = mdl.U, mdl.V
    names = ["TP", "FP", "TN", "FN", "TPR", "FPR", "TNR", "FNR", "PPV", "ACC", "ERR", "F1", "Recall", "Precision"]
    for split in ("train", "val"):
        got = utils.eval(names, "reconstruction", X_gt=d[split], U=U, V=V)
        want = utils.eval(names, "reconstruction", X_gt=h[split], U=U, V=V)
        assert all(_same(a, b) for a, b in zip(got, want)), (split, got, want)
        assert _same(utils.description_length(d[split], U, V), utils.description_length(h[split], U, V))
    g, p = (d["train"], d["pd"]), (h["train"], h["pd"])
    assert utils.confusion_counts(*g) == utils.confusion_counts(*p)
    for fn in (utils.TP, utils.FP, utils.FN, utils.TN, utils.TPR, utils.TNR, utils.FPR, utils.FNR, utils.PPV, utils.ACC,
               utils.ERR, utils.F1):
        assert _same(fn(*g), fn(*p)), fn.__name__
    for fn in (utils.coverage_score, utils.weighted_error):
        assert _same(fn(*g, w_fp=w), fn(*p, w_fp=w)), fn.__name__
    assert all(_same(a, b) for a, b in zip(utils.get_metrics(*g, names), utils.get_metrics(*p, names)))
    Pd = utils.get_prediction(U, V)
    assert _same(utils.description_length(d["train"], U, V), utils.description_length(h["train"], U, V, pd=Pd))


@pytest.mark.parametrize("m,n", [(M_, N_), (130, 1000), (257, 65)])
def test_transpose(env, m, n):
    generate, models, utils, d, h = env
    from pybmf_b200 import device
    X = generate.planted_bits(m, n, 4, 0.3, 0.2, 0.1, 0.05, seed=9)
    T = generate.transpose(X)
    assert (T.m, T.n, T.r0, T.r1) == (n, m, 0, n)
    assert np.array_equal(_dense(T.to_csr()), _dense(X.to_csr()).T)
    bits = T.bits.cpu().numpy()
    assert bits.shape == (n, device.words_for(m))
    assert not device.words_to_dense(bits, bits.shape[1] * 64)[:, m:].any()      # pad bits stay zero


def test_transpose_bits_row_chunks(env):
    """More rows than one bmf_transpose_bits launch takes (4.19 M): (X^T)^T == X word for word, pad words included."""
    generate, models, utils, d, h = env
    m, n = 4_200_000 + 77, 130
    X = generate.random_bits(m, n, 0.3, seed=2)
    T = generate.transpose(X)
    back = generate.transpose(T)
    assert torch.equal(back.bits, X.bits)
    rows = np.array([0, 1, 4_194_239, 4_194_240, 4_194_303, m - 1])
    x = X.bits[torch.from_numpy(rows).cuda()].cpu().numpy()
    t = T.bits.cpu().numpy()
    for i, r in enumerate(rows):
        for c in (0, 63, 64, 129):
            assert (x[i, c // 64] >> (c % 64)) & 1 == (t[c, r // 64] >> (r % 64)) & 1, (r, c)


@pytest.mark.parametrize("w", WEIGHTS)
def test_transposed_model(env, w):
    generate, models, utils, d, h = env
    got = []
    for X in (d, h):
        mdl = models.TransposedModel(models.Asso(tau=0.4, k=4, w_fp=w))
        mdl.fit(X["train"], X["val"], **FIT_KW)
        got.append((_dense(mdl.U), _dense(mdl.V), mdl.model.logs["updates"]))
    assert got[0][0].shape == (M_, 4) and got[0][1].shape == (N_, 4)
    assert np.array_equal(got[0][0], got[1][0]) and np.array_equal(got[0][1], got[1][1])
    pd.testing.assert_frame_equal(_log(got[0][2]), _log(got[1][2]))


def test_errors(env):
    generate, models, utils, d, h = env
    wrong_shape = generate.planted_bits(M_, N_ + 1, 5, 0.2, 0.15, 0.2, 0.03, seed=4)
    wrong_rows = generate.planted_bits(M_, N_, 5, 0.2, 0.15, 0.2, 0.03, seed=4, rank=1, world=2)
    for bad in (wrong_shape, wrong_rows):
        with pytest.raises(ValueError):
            models.Asso(tau=0.4, k=3).fit(d["train"], bad, **FIT_KW)
        with pytest.raises(ValueError):
            models.TransposedModel(models.Asso(tau=0.4, k=3)).fit(d["train"], None, bad, **FIT_KW)
    with pytest.raises(ValueError):
        models.Asso(tau=0.4, k=3).fit(d["train"], d["val"], **dict(FIT_KW, task="prediction"))
    with pytest.raises(ValueError):
        generate.transpose(wrong_rows)
    with pytest.raises(ValueError):
        utils.confusion_counts(d["train"], wrong_rows)
    mdl = models.Asso(tau=0.4, k=3)
    mdl.fit(h["train"], **FIT_KW)
    with pytest.raises(TypeError):
        utils.confusion_counts(d["train"], h["pd"])
    with pytest.raises(TypeError):
        utils.TP(h["train"], d["pd"])
    with pytest.raises(TypeError):
        utils.eval(["F1"], "reconstruction", X_gt=d["train"], X_pd=h["pd"])
    with pytest.raises(ValueError):
        utils.eval(["F1"], "prediction", X_gt=d["train"], U=mdl.U, V=mdl.V)
    with pytest.raises(TypeError):
        utils.description_length(d["train"], mdl.U, mdl.V, pd=h["pd"])
    for axis in (0, 1):
        with pytest.raises(NotImplementedError):
            utils.confusion_counts(d["train"], d["pd"], axis=axis)
        with pytest.raises(NotImplementedError):
            utils.coverage_score(d["train"], d["pd"], axis=axis)
    for fn in (utils.matmul, utils.add, utils.multiply):
        with pytest.raises(TypeError):
            fn(d["train"], d["pd"], boolean=True)
