"""AssoIter wall time and the one-pass sweep kernel against per-column launches, at c3 and c4.

    python profiles/assoiter_time.py [--configs c3,c4,c4dev] [--repeats 3]
    torchrun --nproc-per-node N profiles/assoiter_time.py ...

For each config the k = 20 Asso model is fitted first (not timed), then:
  * fit seconds of AssoIter(model).fit(X): min / median of --repeats fits after one warm-up, each ending in a device
    synchronise, the max over ranks (every fit starts from the Asso model's U: AssoIter refines it in place);
  * the phase split of one more fit with BMF_FIT_TRACE=1 (upload / pack, usage words, sweeps, write-back) and the number
    of sweep launches;
  * per-sweep kernel time by CUDA events: ONE bmf_refine_sweep(0, k) launch against k bmf_refine_column launches on the
    same state (and both at one column), on this rank's rows; the two tables must be equal;
  * algorithmic bytes of a sweep: m·words·8 (x) + 8·m·kw (usage words read) + 8·m·kw (written) + k·words·8 (V^T),
    and 64-bit popcounts (fused: m·words·(2 + 2k), per column: 4·k·m·words), as rates against the D2D copy rate
    measured in the same run.
c3 = synth.config_c2() (x is 2.8 MB: L2-resident after the first pass); c4 = synth.config_c4() (1.07 GB of x per
GPU at N = 1: DRAM); c4dev = the same shape and densities generated on the device (generate.planted_bits).
Prints one JSON line per config (rank 0)."""
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


def copy_rate(nbytes=2 << 30, reps=10):
    """Device-to-device copy: (read + write bytes) / time, best of `reps`."""
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        t = e0.elapsed_time(e1) * 1e-3
        best = t if best is None else min(best, t)
    return 2 * nbytes / best


def max_over_ranks(v):
    import torch.distributed as dist
    t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def load(name):
    from pybmf_b200 import generate, synth
    if name == "c3":
        return synth.config_c2()
    if name == "c4":
        return synth.config_c4()
    if name == "c4dev":
        return generate.planted_bits(480189, 17770, 40, 0.0175, 0.0175, 0.10, 0.001, seed=20240)
    raise SystemExit("unknown config " + name)


def kernel_times(models, X, U, V, k, reps):
    """Events around one fused sweep and around k per-column launches, on this rank's rows (medians, seconds)."""
    from pybmf_b200 import _native, device
    from pybmf_b200 import utils as U_
    plan, r0, r1, x_bits = models._local_rows(X)
    m_loc = r1 - r0
    n = X.shape[1]
    words = device.words_for(n)
    uw, kw = U_._factor_words(U_._pattern(U)[r0:r1])
    vt = U_._bits_on_device(U_._pattern(V).T.tocsr())
    kU = U.shape[1]
    snap = uw.clone()
    t_f = device.zeros((k, 5), torch.int64)
    t_c = device.zeros((k, 5), torch.int64)
    args = (0.5, 0.5)

    def fused(ncols, table):
        _native.call("bmf_refine_sweep", x_bits, m_loc, n, words, uw, kw, vt, kU, 0, ncols, 1, 1, *args, table)

    def columns(ncols, table):
        for c in range(ncols):
            _native.call("bmf_refine_column", x_bits, m_loc, n, words, uw, kw, vt, kU, c, 1, 1, *args, table[c])

    res = {}
    for label, fn, ncols, table in (("sweep", fused, k, t_f), ("columns", columns, k, t_c),
                                    ("sweep_1col", fused, 1, t_f), ("column_1", columns, 1, t_c)):
        ts = []
        for _ in range(reps + 1):
            uw.copy_(snap)
            table.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(ncols, table)
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        res[label] = statistics.median(ts[1:])
        if label == "columns":
            assert torch.equal(t_f, t_c), "fused and per-column tables differ"
    uw.copy_(snap)
    byts = m_loc * words * 8 + 16 * m_loc * kw + k * words * 8
    res.update(m_loc=m_loc, words=words, kw=kw, sweep_bytes=byts, popc_fused=m_loc * words * (2 + 2 * k),
               popc_columns=4 * k * m_loc * words)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c3,c4,c4dev")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--kernel-reps", type=int, default=5)
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch.distributed as dist
        local = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from pybmf_b200 import _native, models
    from pybmf_b200.engine import dist_ctx
    _native.require_gpu()
    rank, world = dist_ctx()
    name, limits = card()
    peak = copy_rate()
    calls = {"n": 0}
    real_call = _native.call

    def counting_call(fn, *args):
        if fn == "bmf_refine_sweep":
            calls["n"] += 1
        return real_call(fn, *args)

    for cfg in a.configs.split(","):
        X = load(cfg)
        mdl = models.Asso(tau=0.5, k=20, w_fp=0.5)
        mdl.fit(X, **KW)
        U0, V0, logs0 = mdl.U.copy(), mdl.V.copy(), dict(mdl.logs)
        times = []
        for r in range(a.repeats + 1):
            mdl.U, mdl.logs = U0.copy(), dict(logs0)
            it = models.AssoIter(model=mdl, w_fp=0.5)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            it.fit(X, **KW)
            torch.cuda.synchronize()
            dt = max_over_ranks(time.perf_counter() - t0)
            if r > 0:
                times.append(dt)
        accepted = len(it.logs["refinements"]) if "refinements" in it.logs else 0
        mdl.U, mdl.logs = U0.copy(), dict(logs0)
        os.environ["BMF_FIT_TRACE"] = "1"
        models._native.call = counting_call
        try:
            it = models.AssoIter(model=mdl, w_fp=0.5)
            it.fit(X, **KW)
        finally:
            models._native.call = real_call
            os.environ.pop("BMF_FIT_TRACE")
        phases = {}
        for ph, dt in it._dev_trace.rows:
            phases[ph] = phases.get(ph, 0.0) + dt
        phases = {ph: max_over_ranks(v) for ph, v in phases.items()}
        kt = kernel_times(models, X, U0, V0, 20, a.kernel_reps)
        t_sweep = max_over_ranks(kt["sweep"])
        t_cols = max_over_ranks(kt["columns"])
        rec = {"config": cfg, "world": world, "card": name, "power_limit_and_max_sm_clock": limits,
               "m": X.shape[0], "n": X.shape[1], "k": 20, "accepted": accepted, "sweep_launches": calls["n"],
               "fit_s_min": min(times), "fit_s_median": statistics.median(times), "fit_s_all": times,
               "phases_s": phases,
               "sweep_kernel_s": t_sweep, "k_refine_column_s": t_cols, "fused_speedup": t_cols / t_sweep,
               "sweep_1col_s": max_over_ranks(kt["sweep_1col"]), "refine_column_1_s": max_over_ranks(kt["column_1"]),
               "rank0_rows": kt["m_loc"], "sweep_bytes_rank0": kt["sweep_bytes"],
               "sweep_GBps_rank0": kt["sweep_bytes"] / kt["sweep"] / 1e9,
               "columns_bytes_rank0": 20 * kt["sweep_bytes"],
               "columns_GBps_rank0": 20 * kt["sweep_bytes"] / kt["columns"] / 1e9,
               "copy_peak_GBps": peak / 1e9, "sweep_fraction_of_copy_peak": kt["sweep_bytes"] / kt["sweep"] / peak,
               "popc64_per_s_fused": kt["popc_fused"] / kt["sweep"],
               "popc64_per_s_columns": kt["popc_columns"] / kt["columns"]}
        if rank == 0:
            print(json.dumps(rec), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
