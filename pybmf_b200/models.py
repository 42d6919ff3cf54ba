"""`Asso` and `AssoIter` with the reference's constructor / fit() API, computed on a B200.

Host-side mirror of PyBMF/models/{BaseModel,BaseModelTools,Asso,AssoIter}.py: same parameters,
attributes (`U`, `V` lil float64, `X_pd` csr int64, `logs` dict of DataFrames with the
3-level (split, 0, name) columns, `assoc`, `basis`, `name`, `time`), same early-stop
behaviour including the reference's quirks D1/D2 (SURVEY.md section 2), written fresh around the
C-ABI kernels of libbmf_b200.so.  Nothing here falls back to a CPU implementation.
"""
from __future__ import annotations

import os
import pickle
import re
import time
from itertools import product

import numpy as np
import pandas as pd
import scipy.sparse as sp
import torch
from scipy.sparse import csr_matrix, hstack, lil_matrix

from . import _native, device, generate
from . import utils as U_
from .engine import CoverEngine, _Trace, all_reduce_sum, dist_ctx, integer_weights, local_plan

CONFIG_KEYS = ("task", "seed", "display", "verbose", "scaling", "pixels", "show_logs", "save_model", "show_result")
SILENT = bool(int(os.environ.get("PYBMF_B200_SILENT", "0")))


def _say(*a):
    if not SILENT:
        print(*a)


class BaseModel:
    """fit() template of PyBMF/models/BaseModel.py:44-119 + BaseModelTools.py."""

    # ---- parameters / configuration (BaseModelTools.py:16-175) -------------------------------
    def check_params(self, **kwargs):
        self.set_params(**kwargs)
        self.set_config(**kwargs)

    def set_params(self, **kwargs):
        for name, value in kwargs.items():
            if name in CONFIG_KEYS:
                continue
            setattr(self, name, value)
            shown = len(value) if isinstance(value, list) else (value.shape if U_.ismat(value) else value)
            _say("[I] {:<12} : {}".format(name, shown))

    def set_config(self, **kwargs):
        if "task" in kwargs:
            task = kwargs["task"]
            assert task in ["prediction", "reconstruction"], "Eval task must be 'prediction' or 'reconstruction'."
            self.task = task
            _say("[I] task         :", self.task)
        if "seed" in kwargs:
            seed = kwargs["seed"]
            if seed is None and not hasattr(self, "seed"):
                seed = int(time.time())
            if seed is not None:
                self.seed = seed
                self.rng = np.random.RandomState(seed)
                _say("[I] seed         :", self.seed)
        for flag in ("verbose", "display"):
            if not hasattr(self, flag):
                setattr(self, flag, False)
                _say("[I] {:<12} :".format(flag), False)
            if flag in kwargs and kwargs[flag] != getattr(self, flag):
                setattr(self, flag, kwargs[flag])
                _say("[I] {:<12} :".format(flag), kwargs[flag])
        self.scaling = kwargs["scaling"] if ("scaling" in kwargs and self.display) else 1.0
        self.pixels = kwargs["pixels"] if ("pixels" in kwargs and self.display) else 2
        for flag in ("show_logs", "save_model", "show_result"):      # default True, BaseModelTools.py:160-175
            setattr(self, flag, kwargs.get(flag, True))
            if flag in kwargs:
                _say("[I] {:<12} :".format(flag), kwargs[flag])

    def import_model(self, **kwargs):
        """BaseModelTools.py:261-272."""
        for attr, value in kwargs.items():
            setattr(self, attr, value)
            self.print_msg("Overwrote model parameter: {}".format(attr))

    def print_msg(self, msg, type="I"):
        if self.verbose:
            _say("[{}] {}".format(type, msg))

    # ---- data (BaseModel.py:123-150) ---------------------------------------------------------
    def load_dataset(self, X_train, X_val=None, X_test=None):
        if X_train is None:
            raise TypeError("Missing training data.")
        if X_val is None:
            _say("[I] Missing validation data.")
        if X_test is None:
            _say("[W] Missing testing data.")
        # generate.DeviceBits / DeviceEntries (rows already bit-packed on the device) are passed through: Asso packs nothing
        # and uploads nothing
        self.X_train = X_train if hasattr(X_train, "r0") else U_.to_sparse(X_train, "csr")
        self.X_val = _split(self.X_train, X_val, getattr(self, "task", None))
        self.X_test = _split(self.X_train, X_test, getattr(self, "task", None))
        self.m, self.n = self.X_train.shape

    def fit(self, X_train, X_val=None, X_test=None, **kwargs):
        self.check_params(**kwargs)
        self.load_dataset(X_train=X_train, X_val=X_val, X_test=X_test)
        self.init_model()

    def init_model(self):
        self._init_factors()
        self._init_logs()
        self._start_timer()
        self._make_name()

    def _init_factors(self):
        if hasattr(self, "U") or hasattr(self, "V"):
            _say("[I] U, V existed. Skipping initialization.")
            return
        k = self.k if (hasattr(self, "k") and self.k is not None) else 1
        self.U = lil_matrix((self.m, k))
        self.V = lil_matrix((self.n, k))

    def _init_logs(self):
        if not hasattr(self, "logs"):
            self.logs = {}

    def _start_timer(self):
        self.time = time.time()

    def _stop_timer(self):
        if not hasattr(self, "time"):
            _say("[W] Timer not started.")
            return
        self.seconds = time.time() - self.time
        hours, rest = divmod(self.seconds, 3600)
        minutes, seconds = divmod(rest, 60)
        text = ("%dh" % hours if hours > 0 else "") + ("%dm" % minutes if minutes > 0 else "") + "%ds" % seconds
        _say("[I] time elapsed : ", text)
        self.time = text

    def _make_name(self):
        if not hasattr(self, "name"):
            cls = re.split(r"[`\-=~!@#$%^&*()_+\[\]{};'\\:\"|<,./<>?]", str(type(self)))[-3]
            self.name = pd.Timestamp.now().strftime("%Y-%m-%d %H-%M-%S-%f ") + cls
            _say("[I] name         :", self.name)

    # ---- factors (BaseModelTools.py:366-405) --------------------------------------------------
    def set_factors(self, k, u, v):
        if self.U.shape[1] < k + 1:
            self.extend_factors(k + 1)
        self.U[:, k] = u
        self.V[:, k] = v

    def truncate_factors(self, k):
        self.U = self.U[:, :k]
        self.V = self.V[:, :k]

    def extend_factors(self, k):
        self.U = hstack([self.U, lil_matrix((self.m, k - self.U.shape[1]))]).tolil()
        self.V = hstack([self.V, lil_matrix((self.n, k - self.V.shape[1]))]).tolil()

    # ---- early stop (BaseModelTools.py:299-363), defects D1/D2 kept ----------------------------
    def early_stop(self, error=None, diff=None, n_iter=None, n_factor=None, msg=None, k=None, verbose=True):
        is_improving = True
        if error is not None and hasattr(self, "tol") and error <= self.tol:
            self._early_stop(msg="Error <= tolerance", verbose=verbose, k=k)
            is_improving = False
        if n_iter is not None and hasattr(self, "max_iter") and n_iter > self.max_iter:
            self._early_stop(msg="Reach maximum iteration", verbose=verbose, k=k)
            is_improving = False
        if diff is not None and hasattr(self, "min_diff") and diff < self.min_diff:
            self._early_stop(msg="Difference lower than threshold", verbose=verbose, k=k)
            is_improving = False
        if n_factor is not None and (hasattr(self, "k") and self.k is not None) and n_factor >= self.k:
            self._early_stop(msg="Reach requested factor", verbose=verbose)
            is_improving = False
        if msg is not None:
            # the reference calls _early_stop(msg=msg, k=k) without `verbose` here
            # (BaseModelTools.py:338-341 vs :346) and therefore raises TypeError: same behaviour.
            self._early_stop(msg=msg, k=k)
            is_improving = False
        return is_improving

    def _early_stop(self, msg, verbose, k=None):
        if verbose:
            _say("[W] Stopped in advance: " + msg)
        if k is not None:
            if verbose:
                _say("[W] Obtained {} factor(s).".format(k))
            self.truncate_factors(k)

    # ---- evaluation (BaseModel.py:209-277) ----------------------------------------------------
    def evaluate(self, df_name, head_info={}, train_info={}, val_info={}, test_info={},
                 metrics=["Recall", "Precision", "Accuracy", "F1"], train_metrics=None, val_metrics=None,
                 test_metrics=None, verbose=False):
        train_metrics = metrics if train_metrics is None else train_metrics
        val_metrics = metrics if val_metrics is None else val_metrics
        test_metrics = metrics if test_metrics is None else test_metrics
        columns = U_.header(list(head_info.keys()), levels=3)
        results = list(head_info.values())
        for name, info, mets in (("train", train_info, train_metrics), ("val", val_info, val_metrics),
                                 ("test", test_info, test_metrics)):
            if getattr(self, "X_" + name) is None:
                continue
            c, r = self._evaluate(name, info, mets)
            columns += c
            results += r
        batch = self.__dict__.get("_dev_log_batch")
        if batch is not None and not verbose:                  # rows are appended in one go by _flush_logs()
            batch.append((df_name, columns, [pd.Timestamp.now().strftime("%d/%m/%y %I:%M:%S")] + results))
            return
        self._flush_logs()
        U_.record(df_dict=self.logs, df_name=df_name, columns=columns, records=results, verbose=verbose)

    def _flush_logs(self):
        """Turn the batched log rows into DataFrame rows (one construction per table instead of one pandas `.loc`
        assignment per greedy step, which costs ~2 ms each)."""
        batch = self.__dict__.get("_dev_log_batch")
        if not batch:
            return
        by_name = {}
        for df_name, columns, row in batch:
            by_name.setdefault(df_name, (columns, []))[1].append(row)
        del batch[:]
        for df_name, (columns, rows) in by_name.items():
            U_.record_many(self.logs, df_name, columns, rows)

    def _evaluate(self, name, info, metrics):
        counts = self._split_counts(name)
        results = U_.metrics_from_counts(metrics, *counts)
        columns = list(product([name], [0], list(info.keys()) + metrics))
        return columns, list(info.values()) + results

    def _split_counts(self, name):
        """(TP, FP, FN, size) of the current factors against X_<name> under self.task
        (evaluate_utils.py:32-52); counts come from bmf_confusion_factors / _entries_factors / _triplets.  A
        generate.DeviceBits or DeviceEntries split is counted on this rank's rows and summed over the ranks: a collective
        under an initialised process group.  Under 'reconstruction' a DeviceEntries counts as its ones, as a host csr
        with stored zeros does; under 'prediction' a DeviceBits (an X_train) stores its ones and no zeros."""
        X = getattr(self, "X_" + name)
        if self.task == "reconstruction":                     # `self.task` unset -> AttributeError, as D6
            return U_.factor_counts(_ones(X), self.U, self.V)
        if hasattr(X, "r0"):
            return U_.entry_counts(X, self.U, self.V)
        Up, Vp = U_._pattern(self.U), U_._pattern(self.V)
        uw, kw = U_._factor_words(Up)
        r, c, g = U_.to_triplet(X)
        vw, _ = U_._factor_words(Vp)
        counts = device.zeros((4,), torch.int64)
        d = device.dev()
        _native.call("bmf_confusion_triplets", torch.from_numpy(r.astype(np.int32)).to(d),
                     torch.from_numpy(c.astype(np.int32)).to(d), torch.from_numpy((g != 0).astype(np.uint8)).to(d),
                     len(g), uw, kw, vw, counts)
        tp, fp, fn, _tn = (int(v) for v in counts.cpu().numpy())
        return tp, fp, fn, len(g)

    # ---- finish (BaseModel.py:104-119, BaseModelTools.py:217-259) ------------------------------
    def finish(self, show_logs=True, save_model=True, show_result=True):
        self._stop_timer()
        if save_model:
            self._save_model()
        if show_result:
            self._show_result()
        if show_logs:
            self._show_logs()

    def _state_for_pickle(self):
        return {k: v for k, v in self.__dict__.items() if not k.startswith("_dev")}

    def __getstate__(self):
        return self._state_for_pickle()

    def _save_model(self, path=None, name=None):
        name = self.name
        if path is None:
            root = os.path.join(os.path.expanduser("~"), ".pybmf", "saved_models")
            os.makedirs(root, exist_ok=True)
            path = os.path.join(root, name + ".pickle")
        self.pickle_path = path
        _ = self.X_pd                                           # the reference pickles X_pd with the rest
        with open(path, "wb") as handle:
            pickle.dump(self._state_for_pickle(), handle, protocol=pickle.HIGHEST_PROTOCOL)
        _say("[I] model saved as: {}.pickle".format(name))

    def _show_logs(self):
        for log in self.logs.values():
            if isinstance(log, pd.DataFrame):
                with pd.option_context("display.max_rows", None, "display.max_columns", None):
                    _say(log)

    def _show_result(self):
        _say("[W] show_result: matplotlib display is outside the accelerated path; skipped.")

    def show_matrix(self, *a, **k):
        _say("[W] show_matrix: matplotlib display is outside the accelerated path; skipped.")

    # ---- lazily materialised containers --------------------------------------------------------
    def __getattr__(self, name):
        # only called when normal lookup fails: X_pd is produced on demand by the GPU product
        d = self.__dict__
        if name == "X_pd":
            try:
                U, V = self.U, self.V
            except AttributeError:
                raise AttributeError(name) from None
            d["X_pd"] = U_.get_prediction(U=U, V=V, boolean=True)
            return d["X_pd"]
        if name in ("assoc", "basis") and "_dev_keep" in d:
            # `assoc` (Asso.py:207-212) and `basis` (Asso.py:231-234, minus the chosen rows Asso.py:106-107) stay on the
            # device after a fit and come to the host the first time somebody reads them (55 MB of counts at the
            # MovieLens shape: reading them eagerly cost more than the whole fit)
            keep = d["_dev_keep"]
            if name == "basis":
                alive = keep["alive"].cpu().numpy().astype(bool)
                idx = torch.from_numpy(np.flatnonzero(alive)).to(keep["basis_bits"].device)
                rows = U_._bits_to_csr(keep["basis_bits"][idx], int(alive.sum()), keep["n"])
                d["basis"] = _csr_to_lil_fast(rows)
                return d["basis"]
            if keep["cnt"] is None:
                raise AttributeError("assoc: the n x n float64 association matrix is not kept for n > 8192 or when the "
                                     "rows are sharded over several GPUs (%.1f GB at n = %d); use `basis`"
                                     % (8e-9 * keep["n"] ** 2, keep["n"]))
            cnt = keep["cnt"].cpu().numpy().astype(np.float64)
            sdiag = np.diag(cnt).copy()
            out = np.zeros_like(cnt)
            out[sdiag > 0] = cnt[sdiag > 0] / sdiag[sdiag > 0][:, None]
            d["assoc"] = lil_matrix(out)
            keep["cnt"] = None
            return d["assoc"]
        raise AttributeError(name)

    def predict_X(self, U=None, V=None, u=None, v=None, us=None, vs=None, boolean=True):
        """BaseModel.py:153-191 (thresholds then Boolean product)."""
        Um = (self.U if U is None else U).copy()
        Vm = (self.V if V is None else V).copy()
        if us is not None:
            assert len(us) == Um.shape[1]
            for i in range(Um.shape[1]):
                Um[:, i] = U_.binarize(Um[:, i], us[i])
        elif u is not None:
            Um = U_.binarize(Um, u)
        if vs is not None:
            assert len(vs) == Vm.shape[1]
            for i in range(Vm.shape[1]):
                Vm[:, i] = U_.binarize(Vm[:, i], vs[i])
        elif v is not None:
            Vm = U_.binarize(Vm, v)
        self.X_pd = U_.matmul(Um, Vm.T, boolean=boolean, sparse=True)


def _csr_to_lil_fast(A: csr_matrix) -> lil_matrix:
    """csr -> lil for tall matrices.  scipy's `tolil()` / `lil_matrix((m, k))` loop over ALL m rows in Python and, worse,
    create 2 m list objects with the cyclic garbage collector running every few hundred allocations (1.3 s for the
    480189 x 20 usage matrix of the Netflix-shaped config).  Here the per-row lists are created in one comprehension
    with the collector paused, and only non-empty rows are filled."""
    import gc
    A = A.tocsr()
    m, k = A.shape
    out = lil_matrix((1, k), dtype=A.dtype)
    was_on = gc.isenabled()
    gc.disable()
    try:
        rows = np.fromiter([[] for _ in range(m)], dtype=object, count=m)
        data = np.fromiter([[] for _ in range(m)], dtype=object, count=m)
        if A.nnz:
            nz = np.flatnonzero(np.diff(A.indptr))
            big_i, big_d = A.indices.tolist(), A.data.tolist()  # one conversion, then cheap list slices per row
            for r, a, b in zip(nz.tolist(), A.indptr[nz].tolist(), A.indptr[nz + 1].tolist()):
                rows[r] = big_i[a:b]
                data[r] = big_d[a:b]
    finally:
        if was_on:
            gc.enable()
    out._shape = (m, k)
    out.rows, out.data = rows, data
    return out


def _split(X_train, X, task):
    """A validation / test split as fit() keeps it: a host matrix becomes a csr; a generate.DeviceBits or DeviceEntries
    is passed through once it is checked, on every rank and before any collective, to have X_train's shape and this
    rank's ShardPlan rows.  task='prediction' counts stored entries (evaluate_utils.py:32-44), stored zeros included,
    which a DeviceEntries holds and plain bit rows cannot express."""
    if X is None:
        return None
    if not hasattr(X, "r0"):
        return U_.to_sparse(X, "csr")
    if X.shape != X_train.shape:
        raise ValueError("device split of shape %s, X_train is %s" % (X.shape, X_train.shape))
    local_plan(X)
    if task == "prediction" and not hasattr(X, "zeros"):
        raise ValueError("task='prediction' counts stored entries; a DeviceBits split has none, use a DeviceEntries "
                         "or 'reconstruction'")
    return X


def _ones(X):
    """The stored ones of a generate.DeviceEntries (what a fit trains on and 'reconstruction' counts), else X."""
    return X.ones if hasattr(X, "zeros") else X


def _local_rows(X):
    """(plan, r0, r1, bit rows) of this rank's share of the training matrix under ShardPlan.  A generate.DeviceBits is
    used as it is (a DeviceEntries by its ones); of a host csr only the rank's rows are packed (generate.bits_from_host)."""
    X = _ones(X)
    plan, r0, r1 = local_plan(X)
    if not hasattr(X, "bits"):
        X = generate.bits_from_host(X)
    return plan, r0, r1, X.bits


def _gather_rows(local, plan):
    """This rank's row block (device tensor, >= its row count rows) -> the rows of ALL ranks as one host array, in row
    order, on every rank: one all-gather.  Rank r's rows start at r times rank 0's row count (ShardPlan)."""
    rank, world = dist_ctx()
    if world == 1:
        return local[: plan.m].cpu().numpy()
    import torch.distributed as dist
    r0, r1 = plan.rows(rank)
    per = plan.rows(0)[1]
    tail = tuple(local.shape[1:])
    padded = torch.zeros((per,) + tail, dtype=local.dtype, device=local.device)
    padded[: r1 - r0] = local[: r1 - r0]
    gathered = torch.empty((world * per,) + tail, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(gathered, padded)
    return gathered[: plan.m].cpu().numpy()


def replay_sweep(table, k, sum_x, size, w_fp, w_fn, best_error, best_score, n_stop):
    """The host side of one AssoIter sweep (AssoIter.py:55-77) on the per-column table of bmf_refine_sweep summed over
    all rows: row c holds (TP, FP, ...) of the whole matrix after column c was refined.

    Returns (steps, stop, best_error, best_score, n_stop).  `steps` lists the columns the reference visits, in order, as
    dicts {k, accepted, and for accepted columns: tp, fp, fn, score, error, score_before, error_before}; `stop` is the
    column after which the reference stops (n_stop reached k), else None."""
    steps = []
    for c in range(k):
        tp, fp = int(table[c][0]), int(table[c][1])
        score = -w_fp * np.array(fp, dtype=np.int64) + w_fn * np.array(tp, dtype=np.int64)
        fn = sum_x - tp
        error = U_.rates(tp, fp, fn, size)["ERR"]
        if error < best_error:
            steps.append({"k": c, "accepted": True, "tp": tp, "fp": fp, "fn": fn, "score": score, "error": error,
                          "score_before": best_score, "error_before": best_error})
            best_error, best_score = error, score
            n_stop = 0
        else:
            steps.append({"k": c, "accepted": False})
            n_stop += 1
            if n_stop == k:
                return steps, c, best_error, best_score, n_stop
    return steps, None, best_error, best_score, n_stop


def _column(vec, n):
    """uint8 vector -> (n x 1) csr float64, the container set_factors() assigns from."""
    idx = np.flatnonzero(vec)
    return csr_matrix((np.ones(len(idx)), (idx, np.zeros(len(idx), dtype=np.int64))), shape=(n, 1))


class Asso(BaseModel):
    """The Asso algorithm (Miettinen et al., the discrete basis problem) -- PyBMF/models/Asso.py:10-140.

    Parameters are the reference's: `tau`, `k=None`, `tol=0`, `w_fp=0.5`, `w_fn=None` (= 1 - w_fp).
    Extra keyword-only knobs of this build (not in the reference): `scorer` in {'auto', 'tcgen05', 'tcgen05_f4',
    'tcgen05_i8', 'popc'} and `assoc_kernel` in {'auto', 'tcgen05', 'tcgen05_f4', 'tcgen05_i8', 'popc'} choose between
    the tensor-core kernels (FP4 `kind::mxf4` when the operand values are E2M1 numbers -- every a/2^s weight pair with
    a, a+b in {1, 2, 3, 4, 6}, and all non-dyadic weights -- else int8 `kind::i8`) and the bit-packed popcount kernels
    (all sm_100a CUDA; results are identical).
    """

    def __init__(self, tau, k=None, tol=0, w_fp=0.5, w_fn=None, *, scorer="auto", assoc_kernel="auto", rescore="auto"):
        self._scorer, self._assoc_kernel, self._rescore = scorer, assoc_kernel, rescore
        self.check_params(tau=tau, k=k, tol=tol, w_fp=w_fp, w_fn=w_fn)

    def fit(self, X_train, X_val=None, X_test=None, **kwargs):
        self.__dict__.pop("U", None)                           # a fit always starts from empty factors
        self.__dict__.pop("V", None)
        self._dev_t0 = time.perf_counter()
        super().fit(X_train, X_val, X_test, **kwargs)
        self._dev_log_batch = []
        try:
            self._fit()
        finally:
            self._flush_logs()
            self.__dict__.pop("_dev_log_batch", None)
            self._materialize_factors(final=True)
            if "_dev" in self.__dict__:
                self._dev.trace.mark("factors_to_host")
                self._dev.trace.dump(self._dev.rank)
            self._release_device()
        self.__dict__.pop("X_pd", None)                        # recomputed lazily from the final U, V (Asso.py:44)
        self.finish(show_logs=self.show_logs, save_model=self.save_model, show_result=self.show_result)

    # ---- factors are kept as device bit columns during the fit and turned into the reference's
    #      lil float64 containers when somebody reads them (BaseModelTools.py:274-288, 366-405) ----
    def _init_factors(self):
        ncols = self.k if (hasattr(self, "k") and self.k is not None) else 1
        self._dev_kept = [None] * ncols                        # one entry per column of U / V, None = zero column

    def truncate_factors(self, k):
        if "_dev_kept" in self.__dict__:
            self._dev_kept = self._dev_kept[:k]
            for name in ("U", "V", "_host_factors"):
                self.__dict__.pop(name, None)
        else:
            super().truncate_factors(k)

    def _place_factor(self, k, entry):
        kept = self._dev_kept
        while len(kept) < k + 1:                               # extend_factors
            kept.append(None)
        kept[k] = entry
        for name in ("U", "V", "_host_factors"):
            self.__dict__.pop(name, None)

    def _materialize_factors(self, final=False):
        """Device bit columns -> host, still PACKED (one small D2H: k x m/8 bytes + the chosen basis rows).  The csr /
        lil float64 containers of the reference are built from the packed bits the first time `U` / `V` is read
        (unpacking 480189 x 20 bits and csr -> lil costs ~0.05 + 0.5 s on the host, none of it needed by fit())."""
        kept = self.__dict__.get("_dev_kept")
        if kept is None:
            return
        dev = self.__dict__.get("_dev")
        live = [(p, e) for p, e in enumerate(kept) if e is not None]
        packed = None
        if live and dev is not None:
            packed = (dev.gather_used_words([e["ui"] for _p, e in live]),
                      dev.basis_words_host([e["j"] for _p, e in live]),
                      np.array([p for p, _e in live], dtype=np.int64))
        self.__dict__.pop("U", None)
        self.__dict__.pop("V", None)
        self._host_factors = (packed, len(kept))
        if final:
            self.__dict__.pop("_dev_kept", None)

    def _unpack_host_factors(self):
        """(packed bits, ncols) -> (U csr m x ncols, V csr n x ncols), float64 ones."""
        packed, ncols = self._host_factors
        if packed is None:
            return csr_matrix((self.m, ncols)), csr_matrix((self.n, ncols))
        parts, vwords, pos = packed
        cols = CoverEngine.unpack_used(parts, len(pos))                            # [m, live] uint8
        _r, c = np.nonzero(cols)                                                   # row-major order = csr order
        indptr = np.concatenate([[0], np.cumsum(cols.sum(axis=1, dtype=np.int64))])
        Uc = csr_matrix((np.ones(len(c)), pos[c], indptr), shape=(self.m, ncols))
        vr = [np.flatnonzero(row) for row in device.words_to_dense(vwords, self.n)]
        Vc = csr_matrix((np.ones(sum(len(v) for v in vr)),
                         (np.concatenate(vr), np.repeat(pos, [len(v) for v in vr]))), shape=(self.n, ncols))
        return Uc, Vc

    def __getattr__(self, name):
        d = self.__dict__
        if name in ("U", "V"):
            if "_dev_kept" in d and "_dev" in d:
                self._materialize_factors()
            if "_host_factors" in d:
                Uc, Vc = self._unpack_host_factors()
                d["U"], d["V"] = _csr_to_lil_fast(Uc), _csr_to_lil_fast(Vc)
                if "_dev_kept" not in d:
                    del d["_host_factors"]
                return d[name]
        return super().__getattr__(name)

    def _state_for_pickle(self):
        if "_host_factors" in self.__dict__:
            _ = self.U                                          # pickles carry the lil factors like the reference's
        keep = self.__dict__.get("_dev_keep")
        if keep is not None:                                    # ... and `basis` / `assoc` where they are small enough
            _ = self.basis
            if keep["cnt"] is not None:
                _ = self.assoc
        return {k: v for k, v in self.__dict__.items() if not k.startswith("_dev") and k != "_host_factors"}

    # ---- init_model: association matrix and candidate basis (Asso.py:48-59, 191-235) -----------
    def init_model(self):
        super().init_model()
        w_fn = 1 - self.w_fp if self.w_fn is None else self.w_fn
        self._dev = CoverEngine(_ones(self.X_train), self.w_fp, w_fn, scorer=self._scorer, assoc=self._assoc_kernel,
                                rescore=self.__dict__.get("_rescore", "auto"))
        self._dev.trace.rows.insert(0, ("before_engine", self._dev.trace.t0 - self.__dict__.get("_dev_t0", self._dev.trace.t0)))
        self.rescore_ = self._dev.rescore                      # 'incremental' or 'full' (what this fit really runs)
        self._dev_nb = self._dev.build_basis(self.tau, prescore=True)
        self.__dict__.pop("assoc", None)
        self.__dict__.pop("basis", None)

    def _release_device(self):
        dev = self.__dict__.pop("_dev", None)
        if dev is not None:
            # keep what the lazy `assoc` / `basis` attributes need, as host arrays
            self._dev_launches = dev.launches
            self._dev_keep = {"n": dev.n, "basis_bits": dev.basis_bits, "alive": dev.alive,
                              "cnt": dev.counts_full() if (dev.n <= 8192 and dev.cnt is not None) else None}
        self.__dict__.pop("_dev_split_cache", None)
        self.__dict__.pop("_dev_nb", None)

    # ---- the greedy loop (Asso.py:62-140) ------------------------------------------------------
    def _fit(self):
        """The k greedy steps run as ONE device-resident sequence (select -> apply -> re-score -> exchange per step, no
        host round trip: CoverEngine.enqueue_steps); the host then reads the per-step table once and replays the
        reference's bookkeeping on it -- log rows, `early_stop` (incl. quirks D1 / D2), factor placement.  Steps that
        the reference would not have run (everything after a D1 truncation) are rolled back and re-run from the
        truncated factors.  With val / test splits the loop advances one step at a time (their counts are per step)."""
        dev = self._dev
        m, n = self.m, self.n
        size = m * n
        n_basis = self._dev_nb
        stepwise = (self.X_val is not None or self.X_test is not None
                    or os.environ.get("BMF_FIT_TRACE_STEPS", "0") == "1")
        # steps are enqueued speculatively in stretches; what the reference would not have run (after D2 / D1) is wasted
        # work, so a stretch is short when a step is expensive (a full scoring pass) and long when it is cheap
        stretch = 32 if dev.rescore == "incremental" else 8
        chunk = 1 if stepwise else min(self.k if self.k is not None else stretch, stretch)
        k = 0                                                 # next greedy step to book (the reference's `k`)
        enq = 0                                               # steps enqueued so far
        table = None
        base = 0
        best_score = 0
        is_improving = True
        if not dev.prescored:
            dev.first_pass()
        self.fit_steps_ = []                                  # per greedy step: winner, score, used, tp, fp (see digest.py)
        while is_improving:
            best_score = 0 if k == 0 else best_score
            if n_basis == 0:
                is_improving = self.early_stop(msg="Candidate list is empty", k=k)
                break
            if k == enq:                                      # nothing pending: enqueue the next stretch and read it back
                count = chunk if self.k is None else max(1, min(chunk, self.k - enq))
                ends_here = self.k is not None and enq + count >= self.k
                dev.enqueue_steps(enq, count, rescore_last=not ends_here)
                base, enq = enq, enq + count
                table = dev.read_table(base, enq)
                dev.trace.mark("greedy_steps")
            row = table[k - base]
            winner = int(row[0])
            if winner < 0:
                is_improving = self.early_stop(msg="No pattern found.", k=k)
                break
            best_score = float(row[1:2].view(np.float64)[0])
            used, tp, fp = int(row[2]), int(row[5]), int(row[6])
            dev.tp_tot, dev.fp_tot = tp, fp
            rowsum = dev.cand_pop_host(winner)                # |b_winner|; the row itself is fetched once, at the end
            self._place_factor(k, {"ui": k, "j": winner, "used": used, "rowsum": rowsum})
            self.fit_steps_.append({"k": k, "winner": winner, "score": best_score, "used": used, "tp": tp, "fp": fp})
            n_basis -= 1
            fn = dev.sum_x - tp
            tp_a, fp_a, fn_a = (np.array(v, dtype=np.int64) for v in (tp, fp, fn))
            score_05 = -0.5 * fp_a + 0.5 * tp_a                                     # Asso.py:119
            u_sum = np.float64(sum(e["used"] for e in self._dev_kept if e is not None))
            v_sum = np.float64(sum(e["rowsum"] for e in self._dev_kept if e is not None))
            desc_len = 1 * (u_sum + v_sum) + 1 * fp_a + 1 * fn_a                    # Asso.py:120
            self._dev_counts = (tp, fp, fn, size)
            self.evaluate(
                df_name="updates", head_info={"k": k},
                train_info={"score": best_score, "score_0.5": score_05, "desc_len": desc_len,
                            "shape": [used, rowsum]},
                metrics=["TP", "TPR", "FP", "FPR", "FN", "FNR", "ERR", "ACC", "Recall", "Precision", "F1"],
                verbose=self.verbose)
            err = U_.rates(tp, fp, fn, size)["ERR"]
            ncols_before = len(self._dev_kept)
            is_improving = self.early_stop(error=err, k=k)     # Asso.py:135 (0-based k: quirk D1)
            truncated = len(self._dev_kept) != ncols_before
            is_improving = self.early_stop(n_factor=k + 1)     # Asso.py:136 overwrites the flag
            k += 1
            if truncated and is_improving:                     # D1: the cover is U o V^T of the TRUNCATED factors
                dev.rollback(k, [int(r[0]) for r in table[k - base:]],
                             [(e["ui"], e["j"]) for e in self._dev_kept if e is not None], best_score)
                enq = k
        self.__dict__.pop("_dev_counts", None)

    def _split_counts(self, name):
        # the training split's counts are already on the host (integer counters of the cover state)
        if name == "train" and "_dev_counts" in self.__dict__ and self.task == "reconstruction":
            return self._dev_counts
        dev = self.__dict__.get("_dev")
        X = getattr(self, "X_" + name)
        if dev is None or "_dev_counts" not in self.__dict__ or X.shape != (self.m, self.n):
            return super()._split_counts(name)
        # During a fit the cover U o V^T of this rank's rows IS dev.c_bits: the split is packed once per fit and every
        # step costs one streaming pass (no factor materialisation, no re-upload).
        # reconstruction: counts over the whole matrix; prediction: over the STORED entries (evaluate_utils.py:32-44),
        # i.e. ones (TP / FN) and explicitly stored zeros (FP / TN), both in one bmf_confusion_entries_bits pass.
        cache = self.__dict__.setdefault("_dev_split_cache", {})
        key = (name, self.task)
        if key not in cache and hasattr(X, "r0"):           # generate.DeviceBits / DeviceEntries: already bit rows
            ones = _ones(X).bits
            if self.task == "prediction":                    # a DeviceBits (an X_train) stores its ones and no zeros
                cache[key] = {"ones": ones, "zeros": X.zeros.bits if hasattr(X, "zeros") else None}
            else:
                n_ones = device.zeros((3,), torch.int64)
                if dev.m_loc > 0:                             # |split|: TP of the split against itself, once per fit
                    _native.call("bmf_confusion_bits", ones, ones, dev.m_loc, dev.words, -1, n_ones, None, None)
                cache[key] = {"ones": ones, "n_ones": int(n_ones[0])}
        if key not in cache:
            Xl = device.csr_rows_view(X, dev.r0, dev.r1)
            # the common case stores no explicit zeros: then the stored pattern IS the set of ones (no 1e8-entry copies)
            dirty = device.has_stored_zeros(Xl)
            ones = Xl
            if dirty:
                ones = Xl.copy()
                ones.eliminate_zeros()
            entry = {"ones": U_._bits_on_device(ones) if dev.m_loc > 0 else None, "n_ones": int(ones.nnz)}
            if self.task == "prediction":
                entry["zeros"] = None
                if dirty:
                    zeros = Xl.copy()
                    zeros.data = (zeros.data == 0).astype(np.int8)
                    zeros.eliminate_zeros()
                    entry["zeros"] = U_._bits_on_device(zeros) if dev.m_loc > 0 else None
            cache[key] = entry
        e = cache[key]
        counts = device.zeros((4,), torch.int64)
        if dev.m_loc > 0:
            if self.task == "reconstruction":
                _native.call("bmf_confusion_bits", e["ones"], dev.c_bits, dev.m_loc, dev.words, e["n_ones"], counts[:3],
                             None, None)
            else:
                _native.call("bmf_confusion_entries_bits", e["ones"], e["zeros"], dev.c_bits, dev.m_loc, dev.words, counts)
        c = all_reduce_sum(counts).cpu().numpy()
        if self.task == "reconstruction":
            return int(c[0]), int(c[1]), int(c[2]), self.m * self.n
        # (|G1 & C|, |G0 & C|, |G1|, |G0|): TP, FP, FN = |G1| - TP, size = |G1| + |G0|
        return int(c[0]), int(c[1]), int(c[2] - c[0]), int(c[2] + c[3])


class AssoIter(Asso):
    """Asso with iterative refinement of the columns of U -- PyBMF/models/AssoIter.py:12-100."""

    def __init__(self, model, w_fp=0.5, w_fn=None):
        self.check_params(model=model, w_fp=w_fp, w_fn=w_fn)

    def check_params(self, **kwargs):
        super().check_params(**kwargs)
        if "model" in kwargs:
            model = kwargs.get("model")
            self.import_model(k=model.k, U=model.U, V=model.V, logs=model.logs)   # by reference (D7)

    def fit(self, X_train, X_val=None, X_test=None, **kwargs):
        BaseModel.fit(self, X_train, X_val, X_test, **kwargs)
        self.__dict__.pop("X_pd", None)
        self._dev_log_batch = []
        try:
            self._fit()
        finally:
            self._flush_logs()
            self.__dict__.pop("_dev_log_batch", None)
        self.__dict__.pop("X_pd", None)
        self.finish(show_logs=self.show_logs, save_model=self.save_model, show_result=self.show_result)

    def init_model(self):
        BaseModel.init_model(self)

    def _init_factors(self):
        BaseModel._init_factors(self)

    def _fit(self):
        """Rows are sharded like Asso's (ShardPlan over the ranks of an initialised process group): each rank refines
        only its rows, and ONE all-reduce per sweep of the [k][5] per-column table gives every rank the same integers,
        from which every rank replays the same accept / skip / stop decisions (replay_sweep)."""
        _native.require_gpu()
        if self.k > self.U.shape[1]:                                              # U[:, idx] in AssoIter.py:85-86
            raise IndexError("index (%d) out of range" % (self.k - 1))
        trace = _Trace()
        self._dev_trace = trace
        m, n = self.m, self.n
        size = m * n
        w_fp = self.w_fp
        w_fn = 1 - self.w_fp if self.w_fn is None else self.w_fn
        iw = integer_weights(float(w_fp), float(w_fn))
        wa, wb, _s = iw if iw else (0, 0, 0)
        plan, r0, r1, x_bits = _local_rows(self.X_train)
        m_loc = r1 - r0
        words = device.words_for(n)
        trace.mark("upload_pack")
        kU = self.U.shape[1]
        uw, kw = U_._factor_words(U_._pattern(self.U)[r0:r1])
        vt = U_._bits_on_device(U_._pattern(self.V).T.tocsr())
        trace.mark("usage_words")
        counts = device.zeros((3,), torch.int64)                                  # TP, FP, FN of this rank's rows
        if m_loc > 0:
            _native.call("bmf_confusion_factors", x_bits, m_loc, words, uw, kw, vt, kU, -1, counts, None, None)
        tp, fp, fn = (int(v) for v in all_reduce_sum(counts).cpu().numpy())
        sum_x = tp + fn
        best_score = -w_fp * np.array(fp, dtype=np.int64) + w_fn * np.array(tp, dtype=np.int64)   # AssoIter.py:52
        best_error = U_.rates(tp, fp, fn, size)["ERR"]
        n_stop = 0
        is_improving = True
        # A sweep over the k columns is deterministic on the device (U[:, k] is ALWAYS replaced, AssoIter.py:60): one
        # bmf_refine_sweep launch refines every column of the rank's rows and fills the per-column table, which is
        # all-reduced and read with one sync, and the accept / skip / stop bookkeeping is replayed on the host.  If the
        # reference would have stopped in the middle of the sweep, the usage words are restored from the snapshot and
        # the sweep is re-run up to that column.
        table = device.zeros((max(self.k, 1), 5), torch.int64)
        with_splits = self.X_val is not None or self.X_test is not None

        def write_back():                                       # usage words -> the lil U the caller holds (in place: D7)
            # The reference assigns U[:, k] column by column on the SAME lil object the source model holds (AssoIter.py:28,
            # 60); here all columns are rebuilt from the usage words of every rank at once and the object's row lists are
            # replaced in place (a lil column assignment walks every row: 0.3 ms per column at 6040 rows).
            dense = device.words_to_dense(_gather_rows(uw, plan), kU)             # [m, kU] uint8
            new = _csr_to_lil_fast(csr_matrix(dense, dtype=self.U.dtype))
            if sp.isspmatrix_lil(self.U) and self.U.shape == new.shape:
                self.U.rows[:] = new.rows
                self.U.data[:] = new.data
            else:
                for c in range(kU):
                    self.U[:, c] = _column(dense[:, c], m)
            self.__dict__.pop("X_pd", None)

        def run(upto):
            table.zero_()
            if upto > 0 and m_loc > 0:
                _native.call("bmf_refine_sweep", x_bits, m_loc, n, words, uw, kw, vt, kU, 0, upto, wa, wb, float(w_fp),
                             float(w_fn), table)

        while is_improving:
            snapshot = uw.clone()
            run(self.k)
            rows = all_reduce_sum(table).cpu().numpy()
            steps, stop, best_error, best_score, n_stop = replay_sweep(rows, self.k, sum_x, size, w_fp, w_fn, best_error,
                                                                       best_score, n_stop)
            for s in steps:
                k = s["k"]
                if not s["accepted"]:
                    _say("[I] Skipped column i: {}.".format(k))
                    continue
                _say("[I] Refined column i: {}, error: {:.4f} -> {:.4f}, score: {:.2f} -> {:.2f}.".format(
                    k, s["error_before"], s["error"], float(s["score_before"]), float(s["score"])))
                self._dev_counts = (s["tp"], s["fp"], s["fn"], size)
                if with_splits:                                                   # val / test counts read self.U as of now
                    now = uw.clone()
                    uw.copy_(snapshot)
                    run(k + 1)
                    write_back()
                    uw.copy_(now)
                self.evaluate(df_name="refinements", head_info={"k": k},
                              train_info={"score": s["score"], "error": s["error"]})
            if stop is not None:
                _say("[I] Error stops decreasing.")
                is_improving = False
                if stop < self.k - 1:                                             # undo the columns the reference never reached
                    uw.copy_(snapshot)
                    run(stop + 1)
        trace.mark("sweeps")
        write_back()
        trace.mark("write_back")
        trace.dump(dist_ctx()[0])
        self.__dict__.pop("_dev_counts", None)


class TransposedModel(Asso):
    """Column-wise Asso: fit the wrapped model on X^T and swap the factors --
    PyBMF/models/TransposedModel.py:6-23 (SURVEY.md section 8f, rank 1: comes for free once the packer
    handles X^T)."""

    def __init__(self, model, **kwargs):
        self.check_params(model=model, **kwargs)
        assert isinstance(self.model, BaseModel), "The model must be an instance of BaseModel."

    def fit(self, X_train, X_val=None, X_test=None, **kwargs):
        if any(hasattr(X, "r0") for X in (X_train, X_val, X_test)):
            # row-sharded bit rows: their X^T is re-sharded over the ranks by generate.transpose (a collective; both parts
            # of a DeviceEntries); the splits are checked first so that a bad split raises on every rank before any exchange
            task = kwargs.get("task", getattr(self.model, "task", None))
            X_val, X_test = _split(X_train, X_val, task), _split(X_train, X_test, task)
            X_train, X_val, X_test = (_transposed(X) for X in (X_train, X_val, X_test))
        else:
            X_train = X_train.T
            X_val = X_val.T if X_val is not None else None
            X_test = X_test.T if X_test is not None else None
        self.model.fit(X_train, X_val, X_test, **kwargs)
        self.U, self.V = self.model.V, self.model.U


def _transposed(X):
    """X^T of a fit input: generate.transpose of a DeviceBits and of both parts of a DeviceEntries, `.T` of a host matrix."""
    if X is None:
        return None
    if hasattr(X, "zeros"):
        return generate.DeviceEntries(generate.transpose(X.ones), generate.transpose(X.zeros))
    return generate.transpose(X) if hasattr(X, "bits") else X.T


class AssoOpt(Asso):
    """Asso with an exhaustive search over each row of U -- PyBMF/models/AssoOpt.py:12-80 (SURVEY.md section 8f,
    rank 4).  `set_optimal_row(i)` tries all 2^k usage vectors for data row i; here one kernel launch
    (bmf_optimal_rows) does that for every row.  The reference's `_fit` ends in its defect D4
    (`coverage_score(..., w=self.w)`, AssoOpt.py:65: there is no attribute `w`), which is reproduced: U is refined, then
    the same AttributeError surfaces."""

    def __init__(self, model, w_fp=1, w_fn=1):
        self.check_params(model=model, w_fp=w_fp, w_fn=w_fn)

    def check_params(self, **kwargs):
        BaseModel.check_params(self, **kwargs)
        if "model" in kwargs:
            model = kwargs.get("model")
            self.import_model(k=model.k, U=model.U, V=model.V, logs=model.logs)

    def fit(self, X_train, X_val=None, X_test=None, **kwargs):
        BaseModel.fit(self, X_train, X_val, X_test, **kwargs)
        self._fit()
        self.finish(show_logs=self.show_logs, save_model=self.save_model, show_result=self.show_result)

    def init_model(self):
        BaseModel.init_model(self)

    def _init_factors(self):
        BaseModel._init_factors(self)

    def optimal_rows(self, rows=None):
        """argmax trial of every data row (or of `rows`) and its score: int64 [m], float64 [m].

        Without `rows` this is a collective under an initialised process group: each rank searches its ShardPlan rows and
        one all-gather gives every rank all of them.  Explicit `rows` are searched locally, with no collective (of a
        generate.DeviceBits input only this rank's rows can be asked for)."""
        _native.require_gpu()
        vt = U_._bits_on_device(U_._pattern(self.V).T.tocsr())
        if vt.shape[0] != self.k:
            raise ValueError("shapes (1,%d) and (%d,%d) not aligned" % (self.k, vt.shape[0], self.n))   # int2bin(j, k) @ V.T
        X = self.X_train
        plan = None
        if rows is not None:
            idx = np.asarray(rows, dtype=np.int64).reshape(-1)
            if hasattr(X, "bits"):
                assert ((idx >= X.r0) & (idx < X.r1)).all(), "DeviceBits holds rows [%d, %d) only" % (X.r0, X.r1)
                x_bits = X.bits[torch.from_numpy(idx - X.r0).to(X.bits.device)]
            else:
                x_bits = U_._bits_on_device(device.to_csr_pattern(X)[idx])
            m = len(idx)
        else:
            plan, r0, r1, x_bits = _local_rows(X)
            m = r1 - r0
        best = device.zeros((max(m, 1),), torch.int64)
        score = device.zeros((max(m, 1),), torch.float64)
        if m > 0:
            _native.call("bmf_optimal_rows", x_bits, m, x_bits.shape[1], vt, self.k, float(self.w_fp), float(self.w_fn),
                         best, score)
        if plan is not None:
            return _gather_rows(best, plan), _gather_rows(score, plan)
        return best.cpu().numpy()[:m], score.cpu().numpy()[:m]

    def set_optimal_row(self, i):
        """AssoOpt.py:69-80: index of the best of the 2^k usage vectors for row i (np.argmax: first maximum)."""
        idx, _score = self.optimal_rows([i])
        return int(idx[0])

    def _fit(self):
        tic = time.perf_counter()
        results, _scores = self.optimal_rows()
        _say("[I] Exhaustive search finished in {}s.".format(time.perf_counter() - tic))
        k = self.k
        bits = ((results[:, None] >> (k - 1 - np.arange(k))[None, :]) & 1).astype(np.int64)    # int2bin: MSB first
        self.U[:, :] = lil_matrix(bits)
        self.__dict__.pop("X_pd", None)
        self.X_pd = U_.get_prediction(U=self.U, V=self.V, boolean=True)
        score = U_.coverage_score(gt=self.X_train, pd=self.X_pd, w=self.w)         # AssoOpt.py:65 (D4)
        self.evaluate(df_name="refinements", train_info={"score": score})
