"""GreConD+'s expansion at the c4 shape (480189 x 17770): the incremental loop against the former one, in one run.

    python profiles/expansion_time.py [--repeats 5] [--m 480189] [--n 17770]

Inputs (generate, one rank): X = planted_bits(m, n, 8 factors, d_u = 0.001, d_v = 0.05, p_fn = 0.05, p_fp = 0.005),
X_old = the cover of its first 3 factors (planted_bits with the same seed, 3 factors, no noise: the factor streams do not
depend on the factor count), and a seed pattern inside factor 5 (its first 32 rows, its first half of columns), which the
loop grows by the rest of that factor: hundreds of iterations.
  * init: bmf_expand_init by CUDA events (best / median of --repeats), GB/s of the 2 m n / 8 bytes it reads, against a
    device copy of X's bit rows (m n / 8 bytes read and written) timed in the same run.
  * new: expansion.expansion_log on the DeviceBits, whole call by events (init, all stretches, the log reads); us per
    iteration = (call - init) / iterations.
  * old: the former loop, kept only here: per iteration two _ExpansionState.score calls (bmf_expand_scores over X / X_old
    and over their transposes, each with its device-to-host read of (score, index)) and the rule; us per iteration.
  * the two loops' iteration logs must be identical.
The card name and power limit are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("PYBMF_B200_SILENT", "1")

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def timed(fn, repeats):
    """Event times (s) of fn() after one warm-up, and the last result."""
    res = fn()
    out = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) * 1e-3)
    return out, res


def old_loop(st, u_bits, v_bits, w_fp, w_fn):
    """The former expansion(): two full score passes and two device-to-host reads per iteration."""
    steps = []
    while True:
        r_score, r_index = st.score(u_bits, v_bits, w_fp, w_fn, axis=1)
        c_score, c_index = st.score(u_bits, v_bits, w_fp, w_fn, axis=0)
        if r_score > c_score and r_score > 0:
            steps.append((0, r_index))
            bits, i = u_bits, r_index
        elif c_score > r_score and c_score > 0:
            steps.append((1, c_index))
            bits, i = v_bits, c_index
        else:
            steps.append((2, -1))
            return np.array(steps, dtype=np.int64)
        b = 1 << (i & 63)
        bits[0, i >> 6] |= b - (1 << 64) if b >= (1 << 63) else b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--m", type=int, default=480189)
    ap.add_argument("--n", type=int, default=17770)
    args = ap.parse_args()
    from pybmf_b200 import _native, device, expansion, generate, models
    torch.cuda.set_device(0)
    _native.require_gpu()
    models.SILENT = True
    m, n, seed, k, k_old, f = args.m, args.n, 5, 8, 3, 5
    d_u, d_v, w_fp, w_fn = 0.001, 0.05, 0.5, 0.5
    X = generate.planted_bits(m, n, k, d_u, d_v, 0.05, 0.005, seed=seed)
    O = generate.planted_bits(m, n, k_old, d_u, d_v, 0.0, 0.0, seed=seed)
    Ufac = device.words_to_dense(generate.random_bits(m, k, d_u, seed, stream_id=1).bits[:, :1].cpu().numpy(), k)
    Vfac = device.words_to_dense(generate.random_bits(k, n, d_v, seed, stream_id=2).bits.cpu().numpy(), n)
    rows, cols = np.flatnonzero(Ufac[:, f]), np.flatnonzero(Vfac[f])
    u, v = np.zeros(m, np.int64), np.zeros(n, np.int64)
    u[rows[:32]] = 1
    v[cols[: len(cols) // 2]] = 1
    words = device.words_for(n)
    byts = 2 * m * n / 8

    # init pass against a device copy of X's bit rows
    u_bits, v_bits = expansion._vec_bits(u, m), expansion._vec_bits(v, n)
    row_cnt = device.zeros((m, 4), torch.int32)
    col_cnt = device.zeros((4, n), torch.int64)
    t_init, _ = timed(lambda: _native.call("bmf_expand_init", X.bits, O.bits, m, n, words, 0, u_bits, v_bits, row_cnt,
                                           col_cnt), args.repeats)
    dst = torch.empty_like(X.bits)
    t_copy, _ = timed(lambda: dst.copy_(X.bits), args.repeats)
    del dst

    # the new loop
    t_new, steps_new = timed(lambda: expansion.expansion_log(X, O, u, v, w_fp, w_fn), args.repeats)
    n_iter = len(steps_new)

    # the former loop on X, X_old and their transposes
    st = expansion._ExpansionState.__new__(expansion._ExpansionState)
    st.m, st.n, st.x, st.o = m, n, X.bits, O.bits
    st.xt, st.ot = generate.transpose_bits(X.bits, m, n), generate.transpose_bits(O.bits, m, n)
    st.delta, st.best = device.zeros((max(m, n),), torch.float64), device.zeros((2,), torch.int64)
    t_old, steps_old = timed(lambda: old_loop(st, expansion._vec_bits(u, m), expansion._vec_bits(v, n), w_fp, w_fn),
                             max(1, args.repeats // 2))

    name, limits = card()
    med = statistics.median
    new_us = (med(t_new) - med(t_init)) / n_iter * 1e6
    old_us = med(t_old) / n_iter * 1e6
    print(json.dumps({
        "card": name, "power_limit,max_sm_clock": limits, "m": m, "n": n, "iterations": n_iter,
        "rows_added": int((steps_new[:, 0] == 0).sum()), "cols_added": int((steps_new[:, 0] == 1).sum()),
        "identical_logs": bool(np.array_equal(steps_new, steps_old)),
        "init_ms_best": 1e3 * min(t_init), "init_ms_median": 1e3 * med(t_init),
        "init_GBps_read": byts / min(t_init) / 1e9,
        "copy_ms_best": 1e3 * min(t_copy), "copy_GBps_read_plus_write": 2 * (m * words * 8) / min(t_copy) / 1e9,
        "init_over_copy_rate": (byts / min(t_init)) / (2 * (m * words * 8) / min(t_copy)),
        "new_call_ms_median": 1e3 * med(t_new), "new_us_per_iter": new_us,
        "old_call_ms_median": 1e3 * med(t_old), "old_us_per_iter": old_us, "speedup_per_iter": old_us / new_us}))


if __name__ == "__main__":
    main()
