"""GreConD at the c4 shape (480189 x 17770) on one GPU, in one run.

    python profiles/grecond_time.py [--repeats 5] [--m 480189] [--n 17770] [--k 20]

Input (generate, one rank): X = planted_bits(m, n, 8 factors, d_u = 0.03, d_v = 0.05, p_fn = 0.05, p_fp = 0.001),
about 1.2 % ones like the Netflix-shaped config.
  * fit: models.GreConD(k).fit on the DeviceBits and on the same matrix as a host csr (which the fit packs), wall clock
    around work that ends in a device synchronise; per-factor times from a separate run of concept.Concepts.factor().
  * seed pass: the window of column word 0 on all rows (bmf_concept_intents + bmf_concept_covers) by CUDA events; its
    bytes = the column word of every row twice, plus the full rows of X and R that have a one in the window.
  * candidate round: bmf_concept_intents + bmf_concept_covers + bmf_concept_decide on the first factor's extent rows,
    from the seed state (every column after the seed scored against all extent rows), by CUDA events; its bytes = for
    every column word, the column word of every extent row twice plus the full X and R rows with a live bit in it (these
    come from L2: the extent rows take 2 |C| words x 8 bytes).
  * both against a device copy of X's bit rows (read + write) timed in the same run.
  * the numpy restatement (tests/grecond_reference.grecond_packed) and the device fit at 20000 x 3000, k = 5, for scale.
The card name and power limit are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ.setdefault("PYBMF_B200_SILENT", "1")

import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402
import torch  # noqa: E402

KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def timed(fn, repeats, before=None):
    """Event times (s) of fn() after one warm-up; before() (untimed) runs ahead of every call."""
    if before:
        before()
    fn()
    out = []
    for _ in range(repeats):
        if before:
            before()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) * 1e-3)
    return out


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    res = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, res


def to_host_csr(bits, m, n, chunk=16384):
    """Bit rows -> host csr int64, unpacked on the device in row chunks."""
    shifts = torch.arange(64, device=bits.device, dtype=torch.int64)
    indptr, indices = [np.zeros(1, np.int64)], []
    base = 0
    for a in range(0, m, chunk):
        b = min(m, a + chunk)
        dense = ((bits[a:b].unsqueeze(-1) >> shifts) & 1).to(torch.uint8).reshape(b - a, -1)[:, :n]
        nz = dense.nonzero()
        cnt = torch.bincount(nz[:, 0], minlength=b - a).cpu().numpy()
        indptr.append(base + np.cumsum(cnt))
        base += int(cnt.sum())
        indices.append(nz[:, 1].cpu().numpy())
    ind = np.concatenate(indices)
    return sp.csr_matrix((np.ones(len(ind), np.int64), ind, np.concatenate(indptr)), shape=(m, n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--m", type=int, default=480189)
    ap.add_argument("--n", type=int, default=17770)
    ap.add_argument("--k", type=int, default=20)
    args = ap.parse_args()
    from pybmf_b200 import _native, concept, device, generate, models
    from grecond_reference import grecond_packed, planted
    torch.cuda.set_device(0)
    _native.require_gpu()
    models.SILENT = True
    m, n, k = args.m, args.n, args.k
    X = generate.planted_bits(m, n, 8, 0.03, 0.05, 0.05, 0.001, seed=4)
    W = X.bits.shape[1]
    out = {"m": m, "n": n, "k": k}

    # whole fits
    mdl = models.GreConD(k=k)
    models.GreConD(k=2).fit(X, **KW)                                    # warm-up (module load, allocator)
    t_dev, _ = wall(lambda: mdl.fit(X, **KW))
    covers = [int(c) for c in mdl.logs["updates"][("train", 0, "cover")]]
    Xh = to_host_csr(X.bits, m, n)
    mdl_h = models.GreConD(k=k)
    t_host, _ = wall(lambda: mdl_h.fit(Xh, **KW))
    same = bool((mdl.U != mdl_h.U).nnz == 0 and (mdl.V != mdl_h.V).nnz == 0)
    out.update({"ones": int(Xh.nnz), "density": Xh.nnz / (m * n), "fit_devicebits_s": t_dev, "fit_host_csr_s": t_host,
                "host_and_device_factors_equal": same, "factors": len(covers), "covers": covers,
                "extent_sizes": [int(v) for v in np.asarray(mdl.U.sum(axis=0)).ravel()],
                "intent_sizes": [int(v) for v in np.asarray(mdl.V.sum(axis=0)).ravel()]})

    # per factor
    search = concept.Concepts(X.bits, m, n, 0, m)
    per, accepted, seeds = [], [], []
    for _ in range(k):
        t, got = wall(search.factor)
        if got is None:
            break
        per.append(t)
        accepted.append(search.accepted)
        seeds.append(search.p)
    out.update({"per_factor_ms": [1e3 * t for t in per], "per_factor_ms_median": 1e3 * statistics.median(per),
                "accepted_columns_per_factor": accepted, "seed_columns": seeds})

    # seed pass over all rows, window 0
    res = X.bits.clone()
    buf = device.zeros((64 * W + 64,), torch.int64)
    cov64 = device.zeros((64,), torch.int64)

    def seed_pass():
        _native.call("bmf_concept_intents", X.bits, m, W, n, None, 0, 1, 0, None, None, buf[: 64 * W], buf[64 * W:])
        _native.call("bmf_concept_covers", X.bits, res, m, W, n, None, 0, 1, 0, None, None, buf.unsqueeze(0), 1,
                     64 * W + 64, cov64)
    t_seed = timed(seed_pass, args.repeats)
    hit_rows = int(((X.bits[:, 0] != 0).sum()).item())
    seed_bytes = 2 * (m * 8 * 4 + hit_rows * W * 8)                  # (32 B sector per column word + full rows) x 2 passes

    # one candidate round from the seed state of the first factor
    search = concept.Concepts(X.bits, m, n, 0, m)
    j0, counts = search.seed()
    xc, rc, idx, c_bits, rows = search.extent(j0, counts)
    c0 = c_bits.clone()
    d_bits = device.zeros((W,), torch.int64)
    state = torch.tensor([j0 - 1, 0, 0, 0], dtype=torch.int64, device=xc.device)

    def reset():
        c_bits.copy_(c0)
        d_bits.zero_()
        state.copy_(torch.tensor([j0 - 1, 0, 0, 0], dtype=torch.int64))
    t_round = timed(lambda: search.rounds(xc, rc, c_bits, d_bits, state, rows, 1), args.repeats, before=reset)
    ncw = (n + 63) // 64
    live_rows = sum(int((xc[:rows, cw] != 0).sum().item()) for cw in range(j0 // 64, ncw))
    round_bytes = 2 * ((ncw - j0 // 64) * rows * 32 + live_rows * W * 8)

    dst = torch.empty_like(X.bits)
    t_copy = timed(lambda: dst.copy_(X.bits), args.repeats)
    copy_rate = 2 * X.bits.numel() * 8 / min(t_copy)
    out.update({"seed_pass_ms_best": 1e3 * min(t_seed), "seed_pass_bytes": seed_bytes,
                "seed_pass_GBps": seed_bytes / min(t_seed) / 1e9, "seed_over_copy_rate": seed_bytes / min(t_seed) / copy_rate,
                "round_extent_rows": rows, "round_seed_column": j0, "round_ms_best": 1e3 * min(t_round),
                "round_bytes": round_bytes, "round_GBps": round_bytes / min(t_round) / 1e9,
                "round_over_copy_rate": round_bytes / min(t_round) / copy_rate,
                "copy_ms_best": 1e3 * min(t_copy), "copy_GBps_read_plus_write": copy_rate / 1e9})

    # the restatement at a smaller shape, for scale
    Xs = planted(20000, 3000, 8, 0.08, 0.004, 99)
    t0 = time.perf_counter()
    Us, Vs, _c = grecond_packed(Xs, 5)
    t_ref = time.perf_counter() - t0
    small = models.GreConD(k=5)
    t_small, _ = wall(lambda: small.fit(sp.csr_matrix(Xs), **KW))
    out.update({"small_shape": [20000, 3000, 5], "restatement_s": t_ref, "small_fit_host_csr_s": t_small,
                "small_equal": bool(np.array_equal((small.U.toarray() != 0), Us != 0)
                                    and np.array_equal((small.V.toarray() != 0), Vs != 0))})
    name, limits = card()
    out = {"card": name, "power_limit,max_sm_clock": limits, **out}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
