"""The residual X AND NOT (U o V^T) on one GPU: the one-pass bmf_residual_factors against the two-kernel path it replaces
in utils.get_residual (bmf_bool_product, then bmf_bits_combine op 2), with a device-to-device copy of m * n / 8 bytes
timed in the same run for the copy rate.

    python profiles/residual_time.py [--repeats 20]

Two shapes, both far above the 126 MB L2:
  * c5's largest point, 1M x 100k, k = 64: usage words and V^T rows are ANDs of 5 uniform words (about 2 of 64 factors
    per row), X = the product with about 6 % of its bits flipped, as in test_c5_scale_panel_kernels_properties;
  * the c4 shape 480189 x 17770 with k = 20 factors (two-chunk panel), drawn the same way.
At each shape the three are launched in turn, --repeats times, each between two CUDA events after one warm-up of each,
and with them the fused kernel's static-row-split instance (BMF_PANEL_DYNAMIC=0, the form for more than 64 column panels).
Bytes are the algorithmic ones: fused = m n / 8 read + m n / 8 written + 8 m (usage words) + k n / 8 (V^T); the copy
moves 2 m n / 8 (read + write).  The outputs of both fused forms and the two-kernel path are checked bit-identical.
The card name and power limit are read in the same run.  Prints one JSON line per shape."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SHAPES = {"c5_largest": (1_000_000, 100_000, 64), "c4_k20": (480189, 17770, 20)}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    return q.stdout.strip() or "unknown"


def event_time(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def run_shape(label, m, n, k, repeats):
    from pybmf_b200 import _native, device
    words = device.words_for(n)
    g = torch.Generator(device="cuda")
    g.manual_seed(11)

    def rnd(shape, ands):
        w = torch.randint(-2 ** 63, 2 ** 63 - 1, shape, dtype=torch.int64, device="cuda", generator=g)
        for _ in range(ands - 1):
            w &= torch.randint(-2 ** 63, 2 ** 63 - 1, shape, dtype=torch.int64, device="cuda", generator=g)
        return w

    def mask_cols(b):
        if n % 64:
            b[:, n // 64] &= (1 << (n % 64)) - 1
        b[:, (n + 63) // 64:] = 0
        return b
    uw = rnd((m, 1), 5)
    if k < 64:
        uw &= (1 << k) - 1
    vt = mask_cols(rnd((k, words), 5))
    pd = device.zeros((m, words), torch.int64)
    _native.call("bmf_bool_product", uw, m, 1, vt, k, words, pd)
    x = mask_cols(pd ^ rnd((m, words), 4))
    fused, two, static = (device.zeros((m, words), torch.int64) for _ in range(3))
    src = torch.empty(m * words, dtype=torch.int64, device="cuda")
    dst = torch.empty_like(src)

    def run_fused():
        _native.call("bmf_residual_factors", x, m, words, uw, 1, vt, k, fused)

    def run_static():                                                # the static row split (BMF_PANEL_DYNAMIC=0)
        os.environ["BMF_PANEL_DYNAMIC"] = "0"
        try:
            _native.call("bmf_residual_factors", x, m, words, uw, 1, vt, k, static)
        finally:
            del os.environ["BMF_PANEL_DYNAMIC"]

    def run_two():
        _native.call("bmf_bool_product", uw, m, 1, vt, k, words, pd)
        _native.call("bmf_bits_combine", x, pd, m, words, 2, two)

    def run_copy():
        dst.copy_(src)
    arms = (("fused", run_fused), ("two_pass", run_two), ("copy", run_copy), ("fused_static", run_static))
    times = {name: [] for name, _fn in arms}
    for _name, fn in arms:
        fn()
    torch.cuda.synchronize()
    for _ in range(repeats):
        for name, fn in arms:
            times[name].append(event_time(fn))
    identical = bool(torch.equal(fused, two)) and bool(torch.equal(static, two))
    mat = m * words * 8                                              # m n / 8 bytes, as stored (rows padded to 128 bits)
    alg = 2 * mat + 8 * m + k * words * 8
    copy_tbps = 2 * mat / min(times["copy"]) / 1e12
    fused_tbps = alg / min(times["fused"]) / 1e12
    out = {"shape": label, "m": m, "n": n, "k": k, "repeats": repeats, "bit_identical": identical,
           "algorithmic_bytes": alg}
    for name, ts in times.items():
        out[name + "_s_best"], out[name + "_s_median"] = min(ts), statistics.median(ts)
    out.update({"fused_TBps": fused_tbps, "two_pass_TBps_same_bytes": alg / min(times["two_pass"]) / 1e12,
                "copy_TBps": copy_tbps, "fused_fraction_of_copy": fused_tbps / copy_tbps,
                "fused_static_TBps": alg / min(times["fused_static"]) / 1e12,
                "speedup_vs_two_pass": min(times["two_pass"]) / min(times["fused"])})
    del x, pd, fused, two, static, src, dst
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    args = ap.parse_args()
    from pybmf_b200 import _native
    _native.require_gpu()
    gpu = card()
    for label in args.shapes.split(","):
        res = run_shape(label, *SHAPES[label], args.repeats)
        res["card,power_limit"] = gpu
        print(json.dumps(res), flush=True)
        assert res["bit_identical"], label


if __name__ == "__main__":
    main()
