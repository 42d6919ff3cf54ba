#!/usr/bin/env python
"""Benchmark of the Asso hot path on B200 (contract: see the task statement / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|c1] [--impl reference] [--dump-outputs DIR]

Metric: Asso cover-score throughput in Gop/s (algorithmic ops = 2*m*n*nb_t per greedy step,
SURVEY.md section 8d) plus fit() seconds, on BASELINE.json's Netflix-shaped config (c4) by default.
One "step" = one greedy Asso step over the whole (row-sharded) matrix: score every live
candidate on the tensor cores -> one integer all-reduce -> argmax -> apply the winner.
Inputs are resident in HBM for `value`; `e2e` is a whole Asso.fit() through the public API from a
host scipy matrix (H2D, packing, association, k steps, D2H of factors and log counters).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (description, tau, w_fp, k of a fit)
    "c4": ("Asso k=20 tau=0.5 w=[0.5,0.5], Netflix-shaped synthetic 480189x17770 @1.2% (BASELINE configs[3])", 0.5, 0.5, 20),
    "c2": ("Asso k=20 tau=0.5 w=[0.5,0.5], MovieLens-1M-shaped synthetic 6040x3706 @4.5% (BASELINE configs[1])", 0.5, 0.5, 20),
    "c1": ("Asso k=5 tau=0.5 w=[0.5,0.5], planted 1000x500 (BASELINE configs[0] shape)", 0.5, 0.5, 5),
}


def make_input(workload):
    from pybmf_b200 import synth
    if workload == "c4":
        return synth.config_c4()
    if workload == "c2":
        return synth.config_c2()
    return synth.planted(1000, 500, 5, 0.2, 0.2, 0.1, 0.02, seed=1000)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return p, "MEASURED_PEAKS.json"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


DUMP_LIMIT = 64 << 20                                           # bytes --dump-outputs may write in all


def dump_rows(out, name, total, row_bytes, budget, take):
    """out[name] = take(rows): every row of a `total`-row output when they fit `budget` bytes, else a fixed seeded sample
    of rows (the same in every run with the same arguments), whose indices go to out[name + '_rows']."""
    keep = min(total, max(1, budget // max(row_bytes, 1)))
    rows = np.arange(total) if keep == total else np.sort(np.random.default_rng(0).choice(total, keep, replace=False))
    out[name] = take(rows)
    if keep < total:
        out[name + "_rows"] = rows.astype(np.float64)


def write_dump(out_dir, arrays):
    """arrays (name -> float32 / float64 array) -> out_dir/<name>.npy."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def loop_outputs(eng, table, n_steps, rank):
    """What the greedy loop computed up to its last step, as its caller receives it: per step the winner, score, #used
    rows and cumulative TP / FP; the factor columns U (m x n_steps) and V (n x n_steps) as 0/1; and the gains of the
    scoring pass that ended the last step (0 for candidates no longer alive: their gains are not computed exactly).
    Every rank must call it (U is gathered over the ranks); rank 0 gets the arrays, the others None."""
    from pybmf_b200 import device
    t = table[:n_steps]
    parts = eng.gather_used_words(list(range(n_steps)))
    if rank != 0:
        return None
    out = {"winner": t[:, 0].astype(np.float64), "score": t[:, 1].copy().view(np.float64),
           "used": t[:, 2].astype(np.float64), "tp": t[:, 5].astype(np.float64), "fp": t[:, 6].astype(np.float64)}
    U = eng.unpack_used(parts, n_steps)
    dump_rows(out, "U", eng.m, 4 * n_steps, 48 << 20, lambda r: U[r].astype(np.float32))
    won = t[:, 0] >= 0
    V = np.zeros((eng.n, n_steps), np.float32)
    if won.any():
        V[:, won] = device.words_to_dense(eng.basis_words_host(t[won, 0]), eng.n).T
    dump_rows(out, "V", eng.n, 4 * n_steps, 12 << 20, lambda r: V[r])
    alive = eng.alive[: eng.n].cpu().numpy() != 0
    out["gain_p"] = np.where(alive, eng.gain_p_red[: eng.n].cpu().numpy(), 0).astype(np.float64)
    if not eng.integer_mode:                                    # general weights: the N sums are the second output
        out["gain_n"] = np.where(alive, eng.gain_n_red[: eng.n].cpu().numpy(), 0).astype(np.float64)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def mark(self, wait_s=4.0):
        """Samples taken from now on belong to the timed region.  nvidia-smi needs a moment to come up (longer when
        eight ranks start one each): wait, outside the timed region, until it has delivered its first sample."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < wait_s:
            time.sleep(0.02)
        self.first = len(self.rows)

    def start(self):
        self.first = 0
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        rows = self.rows[self.first:] or self.rows[-1:]
        sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in rows)]
        busy = [v for v in sm if v > 0.5 * (max(mx) if mx else 1)] or sm
        watts = []
        for r in rows:
            try:
                watts.append(float(r[6]))
            except (IndexError, ValueError):
                pass
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(watts) if watts else None,
                "power_w_median": statistics.median(watts) if watts else None}


# ----------------------------------------------------------------------------------------------
# CPU arm: the bit-packed C restatement (oracle/asso_c.c, AND + POPCNT, OpenMP) on the host cores, on a bounded
# row sample of the same workload.  Thread count is set EXPLICITLY (same at every N; torchrun's OMP_NUM_THREADS=1
# does not apply) and reported.
# ----------------------------------------------------------------------------------------------
CPU_SAMPLE_ROWS = {"c4": 16384, "c2": 6040, "c1": 1000}


def cpu_threads():
    env = os.environ.get("BMF_CPU_THREADS")
    if env:
        return max(1, int(env))
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def run_cpu_arm(args, X, workload, tau, w_fp, standalone):
    """One 'step' = association counts + basis of the row sample (setup, timed separately) and a FULL scoring pass of
    every candidate against the sampled rows (timed): 2 * rows * n * nb algorithmic ops, like the GPU line."""
    from oracle import asso_oracle_c as OC
    threads = cpu_threads()
    rows = min(CPU_SAMPLE_ROWS[workload], X.shape[0])
    Xs = X[:rows]
    t0 = time.perf_counter()
    st = OC.BitState(Xs, tau, threads=threads)
    setup_s = time.perf_counter() - t0
    iw = OC.integer_weights(float(w_fp), float(1 - w_fp))
    nb = int(st.alive.sum())
    steps, warmup = (max(args.steps, 1), args.warmup) if standalone else (2, 1)
    budget = 150.0 if standalone else 25.0                      # seconds of CPU time this arm may take
    done, ops, dt = 0, 0.0, 0.0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        st.score_all(w_fp, 1 - w_fp, iw)
        one = time.perf_counter() - t0
        if i >= warmup or one > budget / 3:
            done += 1
            dt += one
            ops += 2.0 * rows * X.shape[1] * nb
        if dt + setup_s > budget:
            break
    sample = ("first %d of %d data rows x all %d candidates x all %d columns per step; candidates = thresholded X^T X of "
              "the sampled rows" % (rows, X.shape[0], nb, X.shape[1]))
    out = {"value": ops / dt / 1e9, "unit": "Gop/s", "cores": threads, "kind": "port",
           "sample": sample + "; bit-packed AND+POPCNT C restatement oracle/asso_c.c (%s), OpenMP; the Python reference "
                              "cannot travel to the GPU box" % ("AVX-512 VPOPCNTQ" if OC.lib().bmfo_has_avx512() else "scalar POPCNT"),
           "seconds": dt, "steps": done, "setup_seconds": setup_s, "host_cpu_count": os.cpu_count()}
    # context, not measured in this run: the genuine single-threaded reference (BASELINE.md section 2, SURVEY 3.1) and the
    # full-size greedy step of this same port recorded when the c4 fixture was generated
    per_cand = {"c4": 43.0, "c2": 0.096, "c1": 0.011}[workload]
    out["genuine_reference_extrapolated"] = {
        "seconds_per_candidate": per_cand, "source": "SURVEY.md section 3.1 / BASELINE.md section 2 (survey container, 1 core)",
        "fit_seconds_extrapolated": per_cand * X.shape[1] * WORKLOADS[workload][3],
        "gops": 2.0 * X.shape[0] * X.shape[1] / per_cand / 1e9}
    fx = os.path.join(ROOT, "tests", "golden", workload + "_digest.json")
    if os.path.exists(fx):
        with open(fx) as fh:
            d = json.load(fh)
        out["port_full_step_recorded"] = {"seconds_per_full_greedy_step": d.get("oracle_score_seconds_per_step"),
                                          "threads": d.get("oracle_threads"), "fit_seconds": d.get("oracle_seconds"),
                                          "where": "authoring container, oracle/make_digests.py (all %d rows, 20 steps)" % d["m"]}
    return out


def product_sweep(points, steps, warmup, rank, world, dump=None):
    """BASELINE.json configs[4]: bit-packed Boolean product U o V^T and the TP/FP/FN counts behind
    evaluate(), m up to 1M, n up to 100k, k = 64, rows sharded over the ranks (no data-path collective,
    three int64 counters are all-reduced).  One step = one materialised product + one confusion pass
    against the product recomputed on the fly.  Algorithmic bytes: m*n/8 written + m*n/8 read.
    With a `dump` dict, rank 0 adds per point the last step's TP / FP / FN and rows of its product (a seeded
    sample of rank 0's rows where they exceed 8 MB as float32)."""
    import torch
    import torch.distributed as dist
    from pybmf_b200 import _native, device
    from pybmf_b200.engine import ShardPlan, all_reduce_sum

    class _A:
        pass
    args = _A()
    args.steps, args.warmup = steps, warmup
    k = 64
    results = []
    stream = torch.cuda.current_stream()
    for (m, n) in points:
        r0, r1 = ShardPlan(m, world).rows(rank)
        m_loc = max(r1 - r0, 1)
        words = device.words_for(n)
        g = torch.Generator(device="cuda")
        g.manual_seed(5 + rank)

        def bern(shape, ands):                                  # int64 words with bit density 2^-ands
            w = torch.randint(-2 ** 63, 2 ** 63 - 1, shape, dtype=torch.int64, device="cuda", generator=g)
            for _ in range(ands - 1):
                w &= torch.randint(-2 ** 63, 2 ** 63 - 1, shape, dtype=torch.int64, device="cuda", generator=g)
            return w
        uw = bern((m_loc, 1), 5)                                # U ~ Bern(2/64) per bit
        gv = torch.Generator(device="cuda"); gv.manual_seed(77)  # V is replicated: same seed on every rank
        vt = torch.randint(-2 ** 63, 2 ** 63 - 1, (k, words), dtype=torch.int64, device="cuda", generator=gv)
        for _ in range(4):
            vt &= torch.randint(-2 ** 63, 2 ** 63 - 1, (k, words), dtype=torch.int64, device="cuda", generator=gv)
        if n % 64:
            vt[:, (n // 64)] &= (1 << (n % 64)) - 1
        vt[:, (n + 63) // 64:] = 0
        pd = device.zeros((m_loc, words), torch.int64)
        _native.call("bmf_bool_product", uw, m_loc, 1, vt, k, words, pd)
        x = pd.clone()                                           # ground truth = product with ~6 % of the bits flipped
        for c0 in range(0, m_loc, 65536):
            blk = x[c0:c0 + 65536]
            blk ^= bern(blk.shape, 4)
        if n % 64:
            x[:, (n // 64)] &= (1 << (n % 64)) - 1
        x[:, (n + 63) // 64:] = 0
        counts = device.zeros((3,), torch.int64)
        counts2 = device.zeros((3,), torch.int64)
        _native.call("bmf_confusion_bits", x, x, m_loc, words, -1, counts2, None, None)
        x_ones = int(counts2[0].item())                          # |X| of this rank's rows (the csr nnz in real use)

        def step():
            _native.call("bmf_bool_product", uw, m_loc, 1, vt, k, words, pd)
            _native.call("bmf_confusion_factors", x, m_loc, words, uw, 1, vt, k, x_ones, counts, None, None)
        for _ in range(max(args.warmup, 1)):
            step()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev[0].record(stream)
        for _ in range(args.steps):
            _native.call("bmf_bool_product", uw, m_loc, 1, vt, k, words, pd)
        ev[1].record(stream)
        for _ in range(args.steps):
            _native.call("bmf_confusion_factors", x, m_loc, words, uw, 1, vt, k, x_ones, counts, None, None)
        ev[2].record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # size-independent checks: the two confusion kernels agree, and TP + FN = |X|, TP + FP = |product|
        _native.call("bmf_confusion_bits", x, pd, m_loc, words, -1, counts2, None, None)            # counts |gt| itself
        ok = bool(torch.equal(counts, counts2))
        all_reduce_sum(counts)
        tp, fp, fn = (int(v) for v in counts.cpu().numpy())
        if dump is not None and rank == 0:
            key = "c5_%dx%d" % (m, n)
            dump[key + "_counts"] = np.array([tp, fp, fn], dtype=np.float64)
            dump_rows(dump, key + "_product", m_loc, 4 * n, 8 << 20, lambda r: device.words_to_dense(
                pd[torch.as_tensor(r, device=pd.device)].cpu().numpy(), n).astype(np.float32))
        bytes_one = m * words * 8.0                              # one bit matrix, all ranks
        prod_gbs = bytes_one * args.steps / (t[0].item() / 1e3) / 1e9
        conf_gbs = bytes_one * args.steps / (t[1].item() / 1e3) / 1e9
        results.append({"m": m, "n": n, "k": k, "product_ms": t[0].item() / args.steps, "confusion_ms": t[1].item() / args.steps,
                        "product_gbs": prod_gbs, "confusion_gbs": conf_gbs, "tp": tp, "fp": fp, "fn": fn,
                        "kernels_agree": ok})
        del x, pd, uw, vt
        torch.cuda.empty_cache()
    return results


def c5_traffic(last, world):
    """DRAM bytes of one product + one confusion launch from the committed ncu capture (largest point on one GPU only)."""
    if world != 1 or (last["m"], last["n"]) != (1_000_000, 100_000):
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            t = json.load(fh)
        return t["c5:product:1"]["bytes"] + t["c5:confusion:1"]["bytes"]
    except (OSError, ValueError, KeyError):
        return None


C5_POINTS = [(10_000, 1_000), (100_000, 10_000), (1_000_000, 10_000), (100_000, 100_000), (1_000_000, 100_000)]


def run_product_sweep(args, rank, world, local_rank, real_stdout):
    import torch
    import torch.distributed as dist
    from pybmf_b200 import _native, device

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    _native.require_gpu()
    peaks, peak_src = load_peaks()
    points = C5_POINTS
    if args.points > 0:
        points = points[: args.points]
    elif args.points < 0:
        points = points[args.points:]                            # e.g. --points -1: only the largest
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.mark()
    dump = {} if args.dump_outputs else None
    results = product_sweep(points, args.steps, max(args.warmup, 1), rank, world, dump)
    clocks = sampler.stop()
    if dump:
        write_dump(args.dump_outputs, dump)
    ceilings = None
    if rank == 0:
        # context: what a pure write / pure read stream reaches on this box with library kernels
        buf = torch.empty((1 << 30,), dtype=torch.int64, device="cuda")           # 8 GiB
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        buf.zero_(); buf.sum(); torch.cuda.synchronize()
        e[0].record(); buf.zero_(); e[1].record(); buf.sum(); e[2].record(); torch.cuda.synchronize()
        ceilings = {"memset_write_only_gbs": buf.numel() * 8 / (e[0].elapsed_time(e[1]) / 1e3) / 1e9,
                    "sum_read_only_gbs": buf.numel() * 8 / (e[1].elapsed_time(e[2]) / 1e3) / 1e9}
        del buf
    if rank == 0:
        last = results[-1]
        hbm = float(peaks.get("hbm_gbs", 6650.0)) * world
        step_ms = last["product_ms"] + last["confusion_ms"]
        bytes_step = 2.0 * last["m"] * device.words_for(last["n"]) * 8
        value = bytes_step / (step_ms / 1e3) / 1e9
        line = {"metric": "bool_product_confusion_gbs", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u64 bit words", "data": "synthetic",
                "config": {"workload": "Boolean product + TP/FP/FN sweep, k=64 (BASELINE configs[4]); headline = largest point",
                           "m": last["m"], "n": last["n"], "l2": "bit matrices of the large points exceed L2"},
                "roofline": {"bound": "hbm", "achieved": value / world, "peak": hbm / world, "unit": "GB/s",
                             "frac": value / hbm, "traffic": c5_traffic(last, world),
                             "traffic_unit": "bytes per step = one product + one confusion launch (profiles/ncu_traffic.json; largest point, 1 GPU)",
                             "algorithmic_bytes_per_step": bytes_step,
                             "kernel": "bool_product_panel_list_kernel + confusion_panel_list_kernel<false, 3> (V^T panel in shared memory; "
                                       "packed selection lists; TMA ring; carry-save tree + POPC counting; dynamic row blocks)",
                             "frac_product": last["product_gbs"] / hbm, "frac_confusion": last["confusion_gbs"] / hbm,
                             "peak_source": peak_src},
                "sweep": results, "library_stream_ceilings": ceilings, "gpu_launches": 2 * args.steps * len(results),
                "clocks": clocks,
                "e2e": None, "cpu_baseline": None}
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()
    return 0


def measure_cublas_int8(torch, nn=8192, reps=10):
    """Context only: cuBLAS int8 GEMM (torch._int_mm) on this box, best of `reps`, Top/s."""
    try:
        a = torch.randint(-2, 2, (nn, nn), dtype=torch.int8, device="cuda")
        b = torch.randint(-2, 2, (nn, nn), dtype=torch.int8, device="cuda")
        best = float("inf")
        for _ in range(3):
            torch._int_mm(a, b)
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * nn ** 3 / (best / 1e3) / 1e12
    except Exception as e:                                      # pragma: no cover
        return "unavailable: %s" % type(e).__name__


def measure_mma_peak(torch, kind, iters=4096, reps=5):
    """Tensor-pipe ceiling measured live (bmf_probe_mma_rate): back-to-back tcgen05.mma of the production shape on
    operands resident in shared memory.  Returns (burst Top/s = best of reps, sustained Top/s = one long launch)."""
    import ctypes
    from pybmf_b200 import _native
    ops = ctypes.c_double(0.0)
    best = float("inf")
    _native.call("bmf_probe_mma_rate", kind, 256, ctypes.byref(ops))
    torch.cuda.synchronize()
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _native.call("bmf_probe_mma_rate", kind, iters, ctypes.byref(ops))
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    burst = ops.value / (best / 1e3) / 1e12
    long_iters = int(iters * max(1.0, 400.0 / best))            # ~0.4 s back to back
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _native.call("bmf_probe_mma_rate", kind, long_iters, ctypes.byref(ops))
    e1.record()
    torch.cuda.synchronize()
    sustained = ops.value / (e0.elapsed_time(e1) / 1e3) / 1e12
    return burst, sustained


def timed_fits(models, torch, dist, world, X, tau, w_fp, k, scorer, rescore, repeats):
    """`repeats` whole Asso(k).fit() calls through the public API from the host scipy matrix.  Returns the per-run
    seconds (max over ranks), seconds incl. the first read of U / V, the last model and what ended the fit."""
    import gc
    secs, plus, err, mdl = [], [], None, None
    for _ in range(repeats):
        mdl = None                                              # the previous model (a lil U of ~1e6 Python lists at c4) is
        gc.collect()                                            # released BEFORE the timed region, not inside it
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        # the cyclic collector is paused while the clock runs (as `timeit` does): a generation-2 pass walks every live
        # container object, and one lil U of the Netflix-shaped config alone is ~1e6 Python lists -- with a few fitted models
        # alive such passes added 0.1-0.3 s to SOME fits (profiles/r02f_fit_repeat_probe_n2.log, r02k_fit_time_c4*.log)
        gc.disable()
        t0 = time.perf_counter()
        mdl = models.Asso(tau=tau, k=k, w_fp=w_fp, scorer=scorer, rescore=rescore)
        try:
            mdl.fit(X, task="reconstruction", save_model=False, show_logs=False, show_result=False)
        except TypeError as e:                                  # the reference's D2 path ends the fit the same way
            err = str(e)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        gc.enable()
        from pybmf_b200.digest import result_digest
        dg = result_digest(mdl)                                 # from the packed bits, before U / V are unpacked
        t2 = time.perf_counter()
        _ = mdl.U, mdl.V                                        # the reference's lil float64 containers
        t3 = time.perf_counter()
        both = torch.tensor([t1 - t0, (t1 - t0) + (t3 - t2)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(both, op=dist.ReduceOp.MAX)
        secs.append(float(both[0].item()))
        plus.append(float(both[1].item()))
        mdl._bench_digest = dg
    return secs, plus, mdl, err


def load_fixture(workload):
    path = os.path.join(ROOT, "tests", "golden", workload + "_digest.json")
    if not os.path.exists(path):
        return None
    with open(path) as fh:
        return json.load(fh)


def digest_verdict(got, want, steps):
    """True / False against the CPU restatement's fixture (prefix of `steps` greedy steps when the run is shorter than
    the fixture's k; the U / V hashes are compared only for the full-length fit); None when there is no fixture."""
    if want is None:
        return None
    from pybmf_b200.digest import digest_matches
    return bool(digest_matches(got, want, steps=None if steps == want["k"] else steps))


# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("BMF_BENCH_WORKLOAD", "c4"), choices=list(WORKLOADS) + ["c5"])
    ap.add_argument("--points", type=int, default=0, help="c5 only: number of sweep points to run (0 = all)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scorer", default="tcgen05", choices=["tcgen05", "tcgen05_f4", "tcgen05_i8", "popc"],
                    help="tcgen05 = the fastest exact tensor-core path (FP4 kind::mxf4 when the weights allow, else int8); "
                         "popc = the bit-packed AND+POPC comparison variant the north star names")
    ap.add_argument("--w-fp", type=float, default=None,
                    help="override the workload's w_fp (w_fn = 1 - w_fp); a non-dyadic value such as 0.2 runs the "
                         "general-weights scorer (two contractions per element, credited 2*m*n*nb like the others)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip roofline_i8 / popc comparison / other_configs")
    ap.add_argument("--fit-repeats", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed as DIR/<name>.npy (float32 / float64, at most "
                         "64 MB; larger outputs as a seeded row sample), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference does not run it")
    args.warmup = max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "c5" and args.impl != "reference":
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        return run_product_sweep(args, rank, world, local_rank, real_stdout)
    if args.workload == "c5":
        args.workload = "c4"
    desc, tau, w_fp, k_fit = WORKLOADS[args.workload]
    if args.w_fp is not None:
        w_fp = float(args.w_fp)
        desc = desc.replace("w=[0.5,0.5]", "w=[%g,%g]" % (w_fp, 1 - w_fp))

    if args.impl == "reference":
        if rank != 0:
            return 0
        X = make_input(args.workload)
        cpu = run_cpu_arm(args, X, args.workload, tau, w_fp, standalone=True)
        line = {"impl": "reference", "metric": "asso_cover_score_gops", "value": cpu["value"], "unit": "Gop/s",
                "n_gpus": args.gpus, "steps": cpu["steps"], "warmup": args.warmup,
                "ms_per_step": 1e3 * cpu["seconds"] / max(cpu["steps"], 1), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u64 AND + POPCNT counts, int64 gains, f64 score",
                "data": "synthetic",
                "config": {"workload": desc, "m": X.shape[0], "n": X.shape[1], "nnz": int(X.nnz)},
                "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "context": {k: cpu[k] for k in ("genuine_reference_extrapolated", "port_full_step_recorded", "setup_seconds",
                                                 "host_cpu_count") if k in cpu},
                "e2e": {"value": cpu["value"], "unit": "Gop/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # exactly ONE line may reach stdout: libraries (NCCL's version banner, torchrun) write to fd 1 too
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from pybmf_b200 import _native, models
    from pybmf_b200.engine import CoverEngine

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    _native.require_gpu()
    models.SILENT = True
    peaks, peak_src = load_peaks()

    X = make_input(args.workload)
    m, n = X.shape
    fixture = load_fixture(args.workload) if (args.w_fp is None) else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident state: pack, association, basis (setup, timed separately) ---------------
    barrier()
    t0 = time.perf_counter()
    eng = CoverEngine(X, w_fp, 1 - w_fp, scorer=args.scorer, rescore="full")
    nb = eng.build_basis(tau)
    eng.first_pass()
    barrier()
    setup_s = time.perf_counter() - t0

    # ---- `value`: K greedy steps of the device-resident loop with a FULL scoring pass per step ------
    # step = select (argmax of the reduced gains) -> apply the winner -> score every live candidate against every data
    # row on the tensor cores -> ONE all-reduce (gains + the step's three counters).  No host round trip inside.
    stream = torch.cuda.current_stream()
    sampler = ClockSampler(local_rank)
    sampler.start()                                             # nvidia-smi needs ~0.2 s to come up: start it early
    if args.warmup:
        eng.enqueue_steps(0, args.warmup)
    torch.cuda.synchronize()
    launches0 = eng.launches
    eng.score_events = []
    sampler.mark()                                              # may wait for nvidia-smi's first sample: before the barrier
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    eng.enqueue_steps(args.warmup, args.steps)
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    elapsed_ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    elapsed_s = float(elapsed_ms.item()) / 1e3
    launches = eng.launches - launches0
    table = eng.read_table(0, args.warmup + args.steps)
    done = int((table[args.warmup:, 7] == 2).sum())             # steps that really chose and applied a winner
    if args.dump_outputs:
        outputs = loop_outputs(eng, table, args.warmup + args.steps, rank)
        if outputs is not None:
            write_dump(args.dump_outputs, outputs)
    score_ms = [a.elapsed_time(b) for a, b in eng.score_events]
    eng.score_events = None
    # the scoring pass of timed step t sees nb - (warmup + t + 1) live candidates (the winner was just removed)
    ops_per_step = [2.0 * m * n * (nb - (args.warmup + t + 1)) for t in range(done)]
    total_ops = float(sum(ops_per_step))
    value = total_ops / elapsed_s / 1e9
    loop_digest = {"winners": [int(v) for v in table[:, 0]], "tp": [int(v) for v in table[:, 5]],
                   "fp": [int(v) for v in table[:, 6]], "used": [int(v) for v in table[:, 2]],
                   "score_bits": [np.int64(v).tobytes().hex() for v in table[:, 1]]}
    loop_ok = None
    if fixture is not None:
        kk = min(len(loop_digest["winners"]), fixture["k"])
        loop_ok = all(list(loop_digest[key])[:kk] == list(fixture[key])[:kk] for key in loop_digest)

    # ---- roofline of the dominant kernel, this rank's share ---------------------------------------
    kern_ms = statistics.mean(score_ms[:done]) if done else float("nan")
    ops_launch = statistics.mean(ops_per_step) / world if ops_per_step else 0.0     # rows are sharded evenly
    achieved = ops_launch / (kern_ms / 1e3) / 1e12
    bf16 = float(peaks.get("bf16_tflops", 1590.0))
    bf16_sus = float(peaks.get("bf16_tflops_sustained", bf16))
    operand = getattr(eng, "operand", "i8")
    if args.scorer == "popc":
        kernel_name, pipe_mult, pipe = "cover_score_popc_kernel (bit-packed AND + POPC, the comparison variant)", 2.0, "int8"
    elif eng.encoding == "pq":
        kernel_name = ("gemm_%s_kernel<EPI_GAIN2> (general fp64 weights: P and Q contractions = 2x hardware ops)"
                       % ("f4_2sm" if operand == "f4" else "i8_2sm"))
        pipe_mult, pipe = (4.0, "fp4") if operand == "f4" else (2.0, "int8")
    elif operand == "f4":
        kernel_name, pipe_mult, pipe = ("gemm_f4s_2sm_kernel<EPI_GAIN> (tcgen05 kind::mxf4 block-scaled with unit scales, "
                                        "cta_group::2, 256 x 496 super tiles, FP32 accumulate of small integers = exact)"), 4.0, "fp4"
    else:
        kernel_name, pipe_mult, pipe = "gemm_i8_2sm_kernel<EPI_GAIN> (tcgen05 kind::i8, cta_group::2)", 2.0, "int8"
    probe = None
    if args.scorer != "popc":
        try:
            pb, ps = measure_mma_peak(torch, 1 if pipe == "fp4" else 0)
            probe = {"burst_tops": pb, "sustained_tops": ps}
        except Exception as e:                                  # pragma: no cover
            probe = {"error": "%s: %s" % (type(e).__name__, e)}
    hw_mult = 2.0 if eng.encoding == "pq" else 1.0              # P and Q: twice the hardware ops per credited op
    peak_meas = probe["sustained_tops"] if (probe and "sustained_tops" in probe) else pipe_mult * bf16_sus
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak_meas, "unit": "TFLOP/s", "frac": achieved / peak_meas,
                "traffic": None, "kernel": kernel_name, "tensor_pipe": pipe,
                "peak_source": ("measured live on this GPU: bmf_probe_mma_rate, back-to-back tcgen05.mma kind::%s 256x256 "
                                "(cta_group::2) on shared-memory operands, one ~0.4 s launch (sustained; the kernel is timed "
                                "inside a long step loop).  MEASURED_PEAKS.json has no %s figure: its bf16 numbers are listed "
                                "beside it" % ("mxf4" if pipe == "fp4" else "i8", pipe)) if probe and "sustained_tops" in probe
                else "%g x bf16_tflops_sustained of %s (probe unavailable)" % (pipe_mult, peak_src),
                "mma_probe": probe, "hardware_ops_per_credited_op": hw_mult,
                "frac_of_probe_burst": achieved / probe["burst_tops"] if probe and "burst_tops" in probe else None,
                "bf16_based": {"source": peak_src, "mult": pipe_mult, "peak_burst": pipe_mult * bf16,
                               "peak_sustained": pipe_mult * bf16_sus, "frac_burst": achieved / (pipe_mult * bf16),
                               "frac_sustained": achieved / (pipe_mult * bf16_sus),
                               "note": "the driver's bf16 figure was taken at ~1.3 GHz under the 1 kW cap on random data; "
                                       "0/1 operands hold 1.8-1.97 GHz, so these fractions can exceed 1"},
                "kernel_ms": kern_ms, "kernel_share_of_step": kern_ms * done / (elapsed_s * 1e3) if done else None,
                "algorithmic_ops_per_launch": ops_launch,
                "spec_tops_of_pipe": 9000.0 if pipe == "fp4" else 4500.0,
                "frac_of_pipe_spec": achieved / (9000.0 if pipe == "fp4" else 4500.0),
                "int8_spec_tops": 4500.0, "frac_of_int8_spec": achieved / 4500.0}
    variant = ("pq-" if eng.encoding == "pq" else "") + operand if args.scorer != "popc" else "popc"
    try:                                                        # per-launch DRAM bytes from the committed ncu capture
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            hit = json.load(fh).get("%s:%s:%d" % (args.workload, variant, world))
        if hit:
            roofline["traffic"] = hit["bytes"]
            roofline["traffic_unit"] = "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, each scaled by its unit)"
            roofline["traffic_source"] = hit["source"]
            roofline["algorithmic_bytes_per_launch"] = ((m / world) + nb) * (n / 2.0 if operand == "f4" else float(n)) \
                * (2 if variant.startswith("pq") else 1)
    except (OSError, ValueError):
        pass

    # ---- the north star's literal target: the kind::i8 kernel on the same state (rank 0 reports) --------------
    roofline_i8 = popc_cmp = None
    if not args.no_extras and args.scorer == "tcgen05" and eng.integer_mode and operand == "f4":
        del eng
        torch.cuda.empty_cache()
        e8 = CoverEngine(X, w_fp, 1 - w_fp, scorer="tcgen05_i8", assoc="tcgen05_f4", rescore="full")
        e8.build_basis(tau)
        e8.first_pass()
        e8.score_events = []
        barrier()
        e8.enqueue_steps(0, 3)
        barrier()
        ms8 = [a.elapsed_time(b) for a, b in e8.score_events][1:]
        t8 = e8.read_table(0, 3)
        ops8 = statistics.mean([2.0 * m * n * (nb - (t + 1)) for t in range(1, 3)]) / world
        k8 = statistics.mean(ms8)
        try:
            p8b, p8s = measure_mma_peak(torch, 0)
        except Exception:                                       # pragma: no cover
            p8b = p8s = None
        ach8 = ops8 / (k8 / 1e3) / 1e12
        roofline_i8 = {"bound": "tensor", "kernel": "gemm_i8_2sm_kernel<EPI_GAIN> (tcgen05 kind::i8, cta_group::2, 256 x 256 tiles)",
                       "kernel_ms": k8, "achieved": ach8, "unit": "TFLOP/s", "peak": p8s, "frac": ach8 / p8s if p8s else None,
                       "mma_probe": {"burst_tops": p8b, "sustained_tops": p8s},
                       "frac_of_int8_spec": ach8 / 4500.0, "bf16_based_frac_sustained": ach8 / (2.0 * bf16_sus),
                       "same_winners_as_fp4": [int(v) for v in t8[:, 0]] == loop_digest["winners"][:3],
                       "north_star_target": "cover scoring >= 50 % of the int8 tensor-pipe peak on 1 B200"}
        if world == 1:                                          # the mandated AND+POPC comparison, one full pass
            gp = torch.zeros_like(e8.gain_p)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            _native.call("bmf_cover_score_popc", e8.x_bits, e8.c_bits, e8.m_loc, e8.n, e8.words, e8.basis_bits, e8.alive,
                         e8.tp_old, e8.fp_old, e8.wa, e8.wb, e8.w_fp, e8.w_fn, gp, None)
            e1.record(stream)
            torch.cuda.synchronize()
            live = e8.alive.bool()
            popc_ms = e0.elapsed_time(e1)
            # e8.gain_p holds the gains after step 2's scoring pass = the state the popcount kernel just scored
            popc_cmp = {"kernel": "cover_score_popc_kernel (uint64 AND + __popc, 64 x 64 tiles in shared memory)",
                        "ms_per_full_pass": popc_ms, "gops": 2.0 * m * n * (nb - 3) / (popc_ms / 1e3) / 1e9,
                        "tensor_core_speedup": popc_ms / kern_ms,
                        "gains_equal_tensor_core": bool(torch.equal(gp[: e8.n][live], e8.gain_p[: e8.n][live]))}
        del e8
    else:
        del eng
    torch.cuda.empty_cache()
    if rank == 0:
        roofline["cublas_int8_tops_live"] = measure_cublas_int8(torch)

    # ---- end to end: Asso.fit() through the public API from a host scipy matrix ------------------
    e2e = None
    result_digest = None
    if not args.no_e2e:
        k_e2e = min(max(args.steps, 1), k_fit)
        try:                                                    # warm-up: first-use costs of the host side (pandas, scipy)
            models.Asso(tau=tau, k=1, w_fp=w_fp, scorer=args.scorer).fit(
                X, task="reconstruction", save_model=False, show_logs=False, show_result=False)
        except TypeError:
            pass
        reps = max(1, args.fit_repeats)
        secs, plus, mdl, err = timed_fits(models, torch, dist, world, X, tau, w_fp, k_e2e, args.scorer, "auto", reps)
        result_digest = mdl._bench_digest
        steps_done = len(mdl.fit_steps_)
        secs_full, _p, mdl_full, _e = timed_fits(models, torch, dist, world, X, tau, w_fp, k_e2e, args.scorer, "full",
                                                 1 if args.workload == "c4" else reps)
        fit_s = statistics.median(secs)
        ops_fit = sum(2.0 * m * n * (nb - t) for t in range(steps_done))
        h2d = 8 * (X.shape[0] + 1) + 4 * int(X.nnz)             # indptr int64 + indices int32 (all ranks together)
        d2h = steps_done * (8 * 8 + (m + 7) // 8 + 8 * ((n + 63) // 64))
        e2e = {"value": ops_fit / fit_s / 1e9, "unit": "Gop/s", "fit_seconds": fit_s, "fit_seconds_all": secs,
               "fit_seconds_min": min(secs), "fit_seconds_median": fit_s, "repeats": reps,
               "fit_plus_factors_seconds": statistics.median(plus),
               "fit_plus_factors_note": "fit() + the first read of model.U / model.V (unpacking the bit columns into the "
                                        "reference's lil float64 containers on the host)",
               "fit_seconds_full_rescore": statistics.median(secs_full), "rescore": getattr(mdl, "rescore_", None),
               "value_full_rescore": ops_fit / statistics.median(secs_full) / 1e9,
               "greedy_steps": steps_done,
               "value_note": "credited ops = sum_t 2*m*n*nb_t (what the reference's k full candidate sweeps compute).  `value` is the "
                             "default fit, which after the first full pass re-scores only the rows each winner changed -- an exact "
                             "identity, same result_digest; `value_full_rescore` is the same fit EXECUTING a full pass per step",
               "h2d_bytes_per_step": h2d / max(steps_done, 1), "d2h_bytes_per_step": d2h / max(steps_done, 1),
               "includes": "csr H2D, bit packing, association X^T X + basis, %d greedy steps, U/V D2H (bit-packed), log rows" % steps_done,
               "ended_with": err,
               "full_rescore_digest_equal": mdl_full._bench_digest == result_digest}

    # ---- the other BASELINE configs, driver-run in the same line (rank 0's view; every rank takes part) -----------
    other = None
    if not args.no_extras and not args.no_e2e and args.workload == "c4" and args.w_fp is None:
        other = {}
        X2 = make_input("c2")
        fx2, fx3 = load_fixture("c2"), load_fixture("c3")
        s2, p2, m2, _e2 = timed_fits(models, torch, dist, world, X2, 0.5, 0.5, 20, args.scorer, "auto", 3)
        other["c2_asso_k20"] = {"fit_seconds_median": statistics.median(s2), "fit_seconds_all": s2,
                                "fit_plus_factors_seconds": statistics.median(p2),
                                "digest_ok": digest_verdict(m2._bench_digest, fx2, 20)}
        it_secs = []
        for _ in range(3):
            src = models.Asso(tau=0.5, k=20, w_fp=0.5, scorer=args.scorer)
            src.fit(X2, task="reconstruction", save_model=False, show_logs=False, show_result=False)
            barrier()
            t0 = time.perf_counter()
            it = models.AssoIter(model=src, w_fp=0.5)
            it.fit(X2, task="reconstruction", save_model=False, show_logs=False, show_result=False)
            torch.cuda.synchronize()
            it_secs.append(time.perf_counter() - t0)
        import hashlib
        h = hashlib.sha256()
        Uc = it.U.tocsc()
        for c in range(Uc.shape[1]):
            h.update(np.packbits((Uc[:, c].toarray().ravel() != 0).astype(np.uint8), bitorder="little").tobytes())
        other["c3_assoiter_k20"] = {"fit_seconds_median": statistics.median(it_secs), "fit_seconds_all": it_secs,
                                    "u_hash_ok": None if fx3 is None else h.hexdigest() == fx3["u_sha256"],
                                    "note": "AssoIter.fit() on the fitted k=20 model (runs on every rank independently)"}
        pts = product_sweep(C5_POINTS[-1:], 3, 1, rank, world)
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        other["c5_largest_point"] = dict(pts[0], frac_product=pts[0]["product_gbs"] / (hbm * world),
                                         frac_confusion=pts[0]["confusion_gbs"] / (hbm * world),
                                         note="1M x 100k, k=64, rows sharded over the ranks; GB/s are whole-job algorithmic")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = run_cpu_arm(args, X, args.workload, tau, w_fp, standalone=False)

    dtype_desc = ("e2m1 x e2m1 -> f32 accumulate of integers (exact) -> int32 counts, int64 gains, f64 score" if operand == "f4"
                  else "int8 x int8 -> int32 (counts), int64 gains, f64 score")
    if rank == 0:
        line = {"metric": "asso_cover_score_gops", "value": value, "unit": "Gop/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * elapsed_s / max(args.steps, 1), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": dtype_desc,
                "data": "synthetic",
                "config": {"workload": desc, "m": m, "n": n, "nnz": int(X.nnz), "candidates": nb, "scorer": args.scorer,
                           "parallelism": "rows sharded over %d rank(s), ONE int64 all-reduce per greedy step (gains + counters)" % world,
                           "step": "device-resident greedy step with a FULL scoring pass (rescore='full'); no host sync inside the timed region",
                           "l2": "operand planes (%.1f GB) exceed L2; no flush needed" % (m * float(n) / (2e9 if operand == "f4" else 1e9))},
                "clocks": clocks, "gpu_launches": launches, "setup_seconds": setup_s, "timed_steps_completed": done,
                "roofline": roofline, "roofline_i8": roofline_i8, "popc_comparison": popc_cmp,
                "e2e": e2e, "cpu_baseline": cpu,
                "result_digest": result_digest,
                "digest_ok": digest_verdict(result_digest, fixture, len(result_digest["winners"])) if result_digest else None,
                "timed_loop_matches_fixture": loop_ok,
                "digest_fixture": "tests/golden/%s_digest.json (CPU restatement, oracle/make_digests.py)" % args.workload if fixture else None,
                "other_configs": other,
                "fit_seconds": e2e["fit_seconds"] if e2e else None}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
