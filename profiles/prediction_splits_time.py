"""Prediction-task splits on the device (generate.ratio_split, DeviceEntries, the one-pass stored-entry counts): what
each costs on one GPU.

    python profiles/prediction_splits_time.py [--parts split,bits,factors,fit] [--repeats 10]

  * split: generate.ratio_split(X, 0.05, 0.05, neg_ratio=1) at 480189 x 17770 (the c4 shape, Bernoulli(0.012) bits) by
    CUDA events, best / median of --repeats after one warm-up (the call: |X| count, thresholds, bmf_split_bits, five
    zero-filled outputs), and the kernel alone; GB/s of bytes read + written = 6 * m * words * 8 against a device copy
    of the same bytes timed in the same run.
  * bits: the in-fit count of a prediction split against a cover at the c4 shape: bmf_confusion_entries_bits (one pass
    over ones, zeros and the cover) against the former two bmf_confusion_bits passes (ones vs cover, zeros vs cover).
  * factors: the largest c5 point (1M x 100k, k = 64, U and V ~ Bernoulli(2/64)): bmf_confusion_entries_factors against
    two bmf_confusion_factors passes (ones, then zeros), ones = a 0.5 % Bernoulli matrix, zeros = as many.
  * fit: Asso(tau=0.5, k=20, w=0.5).fit(X, X_val, X_test, task='prediction') at c4 (synth.config_c4(), host csr), with
    val / test splits of 5 % each of X's ones plus as many stored zeros (generate.ratio_split), given once as
    DeviceEntries and once as the same entries as host csr with stored zeros; host clock around fits that end in a
    device synchronise, min / median of --repeats after one warm-up of each.
Counts of the compared forms are checked equal.  The card name and power limit are read in the same run.  Prints one
JSON line per part."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("PYBMF_B200_SILENT", "1")

import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402
import torch  # noqa: E402

KW = dict(task="prediction", save_model=False, show_logs=False, show_result=False)
C4 = (480189, 17770)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def timed(fn, repeats):
    """Event times (s) of fn() after one warm-up."""
    fn()
    out = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) * 1e-3)
    return out


def copy_rate(nbytes, repeats):
    src = torch.empty(int(nbytes // 2), dtype=torch.uint8, device="cuda")         # reads + writes nbytes
    dst = torch.empty_like(src)
    t = min(timed(lambda: dst.copy_(src), repeats))
    return nbytes / t / 1e9


def part_split(args):
    from pybmf_b200 import _native, device, generate, utils
    m, n = C4
    X = generate.random_bits(m, n, 0.012, seed=3)
    words = X.bits.shape[1]
    nbytes = 6 * m * words * 8
    out = device.zeros((5, m, words), torch.int64)
    th = generate.split_thresholds(utils.confusion_counts(X, X)[0], m, n, 0.05, 0.05, 1.0)
    tc = timed(lambda: generate.ratio_split(X, 0.05, 0.05, 1.0, seed=1), args.repeats)
    tk = timed(lambda: _native.call("bmf_split_bits", X.bits, m, n, words, 0, 1, 5, 6, *th, out), args.repeats)
    gbps = copy_rate(nbytes, args.repeats)
    return {"part": "split", "m": m, "n": n, "call_s_best": min(tc), "call_s_median": statistics.median(tc),
            "kernel_s_best": min(tk), "kernel_s_median": statistics.median(tk), "kernel_GBps": nbytes / min(tk) / 1e9,
            "copy_GBps": gbps, "kernel_ratio_to_copy": nbytes / min(tk) / 1e9 / gbps}


def part_bits(args):
    from pybmf_b200 import _native, device, generate
    m, n = C4
    X = generate.random_bits(m, n, 0.012, seed=3)
    cover = generate.random_bits(m, n, 0.01, seed=4)
    _tr, val, _te = generate.ratio_split(X, 0.1, 0.1, 1.0, seed=1)
    ones, zeros, words = val.ones.bits, val.zeros.bits, X.bits.shape[1]
    n1 = device.zeros((3,), torch.int64)
    _native.call("bmf_confusion_bits", ones, ones, m, words, -1, n1, None, None)
    n_ones = int(n1[0])
    c6, c4 = device.zeros((6,), torch.int64), device.zeros((4,), torch.int64)

    def two():
        _native.call("bmf_confusion_bits", ones, cover.bits, m, words, n_ones, c6[:3], None, None)
        _native.call("bmf_confusion_bits", zeros, cover.bits, m, words, -1, c6[3:], None, None)

    def one():
        _native.call("bmf_confusion_entries_bits", ones, zeros, cover.bits, m, words, c4)

    t2, t1 = timed(two, args.repeats), timed(one, args.repeats)
    a, b = c6.cpu().tolist(), c4.cpu().tolist()
    assert [a[0], a[3], a[0] + a[2]] == b[:3], (a, b)
    nbytes = 3 * m * words * 8
    return {"part": "bits", "m": m, "n": n, "two_pass_s_best": min(t2), "two_pass_s_median": statistics.median(t2),
            "one_pass_s_best": min(t1), "one_pass_s_median": statistics.median(t1), "speedup": min(t2) / min(t1),
            "one_pass_GBps": nbytes / min(t1) / 1e9, "copy_GBps": copy_rate(nbytes, args.repeats), "counts": b}


def part_factors(args):
    from pybmf_b200 import _native, device, generate, utils
    m, n, k = 1_000_000, 100_000, 64
    rng = np.random.RandomState(5)
    U = sp.csr_matrix((rng.rand(m, k) < 2 / 64).astype(np.int64))
    V = sp.csr_matrix((rng.rand(n, k) < 2 / 64).astype(np.int64))
    uw, kw = utils._factor_words(U)
    vt = utils._bits_on_device(V.T.tocsr())
    words = device.words_for(n)
    X = generate.random_bits(m, n, 0.01, seed=8)
    _tr, val, _te = generate.ratio_split(X, 0.5, 0.5, 0.98, seed=2)
    del X, _tr, _te
    ones, zeros = val.ones.bits, val.zeros.bits
    c6, c4 = device.zeros((6,), torch.int64), device.zeros((4,), torch.int64)

    def two():
        _native.call("bmf_confusion_factors", ones, m, words, uw, kw, vt, k, -1, c6[:3], None, None)
        _native.call("bmf_confusion_factors", zeros, m, words, uw, kw, vt, k, -1, c6[3:], None, None)

    def one():
        _native.call("bmf_confusion_entries_factors", ones, zeros, m, words, uw, kw, vt, k, c4)

    t2, t1 = timed(two, args.repeats), timed(one, args.repeats)
    a, b = c6.cpu().tolist(), c4.cpu().tolist()
    assert [a[0], a[3], a[0] + a[2], a[3] + a[5]] == b, (a, b)
    nbytes = 2 * m * words * 8
    return {"part": "factors", "m": m, "n": n, "k": k, "two_pass_s_best": min(t2),
            "two_pass_s_median": statistics.median(t2), "one_pass_s_best": min(t1),
            "one_pass_s_median": statistics.median(t1), "speedup": min(t2) / min(t1),
            "one_pass_GBps": nbytes / min(t1) / 1e9, "counts": b}


def part_fit(args):
    from pybmf_b200 import generate, models, synth
    X = synth.config_c4()
    m, n = X.shape
    Xd = generate.bits_from_host(X)
    _tr, val, test = generate.ratio_split(Xd, 0.05, 0.05, 1.0, seed=4)
    out = {"part": "fit", "m": m, "n": n, "val_stored": int(val.to_csr().nnz)}
    arms = (("device_entries", (val, test)), ("host_csr", (val.to_csr(), test.to_csr())))
    f1 = {}
    for label, (v, t) in arms:
        ts = []
        for i in range(args.repeats + 1):
            mdl = models.Asso(tau=0.5, k=20, w_fp=0.5)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mdl.fit(X, v, t, **KW)
            torch.cuda.synchronize()
            if i:
                ts.append(time.perf_counter() - t0)
        out[label + "_s_min"], out[label + "_s_median"] = min(ts), statistics.median(ts)
        f1[label] = [float(x) for x in mdl.logs["updates"][("val", 0, "F1")]]
    out["same_val_F1_column"] = f1["device_entries"] == f1["host_csr"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="split,bits,factors,fit")
    ap.add_argument("--repeats", type=int, default=10)
    args = ap.parse_args()
    from pybmf_b200 import _native, models
    _native.require_gpu()
    models.SILENT = True
    name, q = card()
    for p in args.parts.split(","):
        res = {"split": part_split, "bits": part_bits, "factors": part_factors, "fit": part_fit}[p](args)
        res.update({"card": name, "power_limit_W,max_sm_MHz": q})
        print(json.dumps(res), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
