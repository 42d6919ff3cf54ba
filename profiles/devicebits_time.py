"""Device-generated, row-sharded inputs (generate.DeviceBits) through the public API: what each costs.

    python profiles/devicebits_time.py [--parts transpose,eval,fit] [--repeats 10]
    torchrun --nproc-per-node N profiles/devicebits_time.py --parts transpose

  * transpose: generate.transpose at 480189 x 17770 (the c4 shape, Bernoulli(0.012) bits) by CUDA events, best and
    median of --repeats calls after one warm-up, and GB/s of (bytes read + bytes written) = 2 * m * n / 8 against a
    device copy of the same bytes timed in the same run.  With N ranks the time is the max over ranks of the whole call
    (transposes into the slots, the all_to_all_single, the placement) and the rate is over the summed bytes of all ranks.
  * eval: utils.eval(..., 'reconstruction', X_gt=<DeviceBits>, U, V) at the largest c5 point (1M x 100k, k = 64, U and V
    ~ Bernoulli(2/64) as lil float64, X = the product with 6 % of its bits flipped, as bench.py builds it) against the
    same bmf_confusion_factors launch called directly on already-packed operands.  The difference is the public API:
    packing U and V on the host, the uploads, the all-reduce and the read-back (3 calls of eval: each takes seconds).
  * fit: Asso(tau=0.5, k=20, w=0.5).fit(X, X_val) at c4 (synth.config_c4(), host csr) with a 10 % validation split (X's
    ones kept with probability 0.1) given once as a DeviceBits and once as the same matrix downloaded as a host csr;
    host clock around fits that end in a device synchronise, min / median of --repeats after one warm-up of each.
The card name and power limit are read in the same run.  Prints one JSON line per part (rank 0)."""
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

KW = dict(task="reconstruction", save_model=False, show_logs=False, show_result=False)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def timed(fn, repeats, world):
    """Event times (s) of fn() after one warm-up; the max over ranks of each call."""
    import torch.distributed as dist
    fn()
    out = []
    for _ in range(repeats):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out.append(float(t))
    return out


def part_transpose(args, rank, world):
    from pybmf_b200 import generate
    m, n = 480189, 17770
    X = generate.random_bits(m, n, 0.012, seed=3)
    m_loc = X.r1 - X.r0
    nbytes = max(m_loc, 1) * n / 8                              # this rank's share of X (and of X^T)
    src = torch.empty(int(2 * nbytes), dtype=torch.uint8, device="cuda")  # a copy reading + writing 2 * nbytes
    dst = torch.empty_like(src)
    tt = timed(lambda: generate.transpose(X), args.repeats, world)
    tc = timed(lambda: dst.copy_(src), args.repeats, world)
    total = 2 * m * n / 8                                       # bytes read + written by all ranks
    return {"part": "transpose", "m": m, "n": n, "world": world, "transpose_s_best": min(tt),
            "transpose_s_median": statistics.median(tt), "transpose_GBps": total / min(tt) / 1e9,
            "copy_s_best": min(tc), "copy_GBps": world * 2 * 2 * nbytes / min(tc) / 1e9,
            "ratio_to_copy": (total / min(tt)) / (world * 2 * 2 * nbytes / min(tc))}


def part_eval(args, rank, world):
    from pybmf_b200 import _native, device, generate, utils
    from pybmf_b200.engine import ShardPlan
    m, n, k = 1_000_000, 100_000, 64
    rng = np.random.RandomState(5)
    U = (rng.rand(m, k) < 2 / 64).astype(np.uint8)
    V = (rng.rand(n, k) < 2 / 64).astype(np.uint8)
    Ul, Vl = sp.lil_matrix(U.astype(np.float64)), sp.lil_matrix(V.astype(np.float64))
    r0, r1 = ShardPlan(m, world).rows(rank)
    uw, kw = utils._factor_words(utils._pattern(Ul)[r0:r1])
    vt = utils._bits_on_device(utils._pattern(Vl).T.tocsr())
    words = device.words_for(n)
    bits = device.zeros((max(r1 - r0, 1), words), torch.int64)
    if r1 > r0:
        _native.call("bmf_bool_product", uw, r1 - r0, kw, vt, k, words, bits)
        flip = generate.random_bits(m, n, 0.06, seed=8)
        bits ^= flip.bits
        del flip
    X = generate.DeviceBits(bits, m, n, r0, r1)
    counts = device.zeros((3,), torch.int64)
    names = ["TP", "FP", "FN", "F1"]

    def direct():
        if r1 > r0:
            _native.call("bmf_confusion_factors", X.bits, r1 - r0, words, uw, kw, vt, k, -1, counts, None, None)

    te = timed(lambda: utils.eval(names, "reconstruction", X_gt=X, U=Ul, V=Vl), min(args.repeats, 3), world)
    td = timed(direct, args.repeats, world)
    res = utils.eval(names, "reconstruction", X_gt=X, U=Ul, V=Vl)
    return {"part": "eval", "m": m, "n": n, "k": k, "world": world, "eval_s_best": min(te),
            "eval_s_median": statistics.median(te), "direct_s_best": min(td), "direct_s_median": statistics.median(td),
            "api_cost_s": min(te) - min(td), "counts": [int(v) for v in res[:3]],
            "direct_GBps": (r1 - r0) * n / 8 / min(td) / 1e9}


def part_fit(args, rank, world):
    from pybmf_b200 import generate, models, synth, utils
    from pybmf_b200.engine import ShardPlan
    X = synth.config_c4()
    m, n = X.shape
    r0, r1 = ShardPlan(m, world).rows(rank)
    xb = utils._bits_on_device(sp.csr_matrix(X)[r0:r1]) if r1 > r0 else None
    keep = generate.random_bits(m, n, 0.1, seed=12)
    if xb is not None:
        keep.bits[: r1 - r0] &= xb[: r1 - r0, : keep.bits.shape[1]]
    val_d = keep
    val_h = keep.to_csr() if world == 1 else None             # the host arm needs the whole split on one rank
    out = {"part": "fit", "m": m, "n": n, "world": world, "val_nnz": int(val_h.nnz) if val_h is not None else None}
    for label, val in (("devicebits", val_d), ("host_csr", val_h)):
        if val is None:
            continue
        ts = []
        logs = None
        for i in range(args.repeats + 1):
            mdl = models.Asso(tau=0.5, k=20, w_fp=0.5)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mdl.fit(X, val, **KW)
            torch.cuda.synchronize()
            if i:
                ts.append(time.perf_counter() - t0)
            logs = mdl.logs["updates"]
        out[label + "_s_min"], out[label + "_s_median"] = min(ts), statistics.median(ts)
        out[label + "_val_F1_last"] = float(logs[("val", 0, "F1")].iloc[-1])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="transpose,eval,fit")
    ap.add_argument("--repeats", type=int, default=10)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from pybmf_b200 import _native, models
    _native.require_gpu()
    models.SILENT = True
    name, q = card()
    for p in args.parts.split(","):
        res = {"transpose": part_transpose, "eval": part_eval, "fit": part_fit}[p](args, rank, world)
        res.update({"card": name, "power_limit_W,max_sm_MHz": q})
        if rank == 0:
            print(json.dumps(res), flush=True)
        torch.cuda.empty_cache()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
