"""Block-sparse against dense FP4 cover scoring at the c4 workload (480189 x 17770, tau = 0.5), one GPU.

    python profiles/block_sparse_time.py [--reps 20]

Times with CUDA events (mean over --reps launches after a warm-up):
  * a full scoring pass: bmf_cover_score_f4 on natural-order planes (dense walk) and bmf_cover_score_f4_blocks on the
    engine's reordered planes (K-block lists, cost-balanced super-tile-outer walk);
  * one re-score over the first 1 % of the data rows (the size of a typical winner's used rows), both ways;
and prints, per kernel, the executed MMA operations / time against the live kind::mxf4 probe rate, and the operand bytes
the kernel must read (rows plane once + the nonzero candidate blocks once) / time against a device copy measured in the
same run.  Both passes must produce identical gains."""
import argparse
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from pybmf_b200 import _native, device, synth  # noqa: E402
from pybmf_b200.engine import F4_ROW_PAD, CoverEngine  # noqa: E402


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    _native.require_gpu()
    X = synth.config_c4()
    eng = CoverEngine(X, 0.5, 0.5, scorer="tcgen05", rescore="full")
    eng.build_basis(0.5)
    assert eng.kb_table is not None, "the c4 basis should select the block-sparse scorer"
    n, m, words, ld4, cp = eng.n, eng.m_loc, eng.words, eng.ld4, eng.cand_pad
    rows_pad = eng.rows_plane.shape[0]
    lib = _native.load()
    one, cov = lib.bmf_e2m1_code(eng.wa + eng.wb), lib.bmf_e2m1_code(eng.wa)
    nat_rows = device.empty((rows_pad, ld4), torch.uint8)
    _native.call("bmf_expand_bits_f4", eng.x_bits, eng.c_bits, m, n, words, one, 0, cov, nat_rows, rows_pad, ld4)
    nat_cand = device.empty((cp, ld4), torch.uint8)
    _native.call("bmf_expand_bits_f4", eng.basis_bits, None, n, n, words, 2, 0, 0, nat_cand, cp, ld4)
    g_dense = device.zeros((cp,), torch.int64)
    g_sparse = device.zeros((cp,), torch.int64)

    def dense():
        _native.call("bmf_cover_score_f4", nat_cand, cp, nat_rows, rows_pad, ld4, eng.cand_pop, eng.wa, g_dense)

    def sparse():
        _native.call("bmf_cover_score_f4_blocks", eng.cand_plane, cp, eng.rows_plane, rows_pad, ld4, eng.cand_pop, eng.wa,
                     eng.kb_table, eng.cand_id, g_sparse)

    sub_rows = max(1, m // 100)
    dyn = torch.tensor([sub_rows], dtype=torch.int32, device=device.dev())

    def re_dense():
        _native.call("bmf_cover_rescore_f4", nat_cand, cp, nat_rows, rows_pad, ld4, eng.cand_pop, eng.wa, dyn, 1, g_dense)

    def re_sparse():
        _native.call("bmf_cover_rescore_f4_blocks", eng.cand_plane, cp, eng.rows_plane, rows_pad, ld4, eng.cand_pop,
                     eng.wa, eng.kb_table, eng.cand_id, dyn, 1, g_sparse)

    out = {"gpu": torch.cuda.get_device_name(), "m": m, "n": n}
    dense()
    sparse()
    torch.cuda.synchronize()
    out["gains_identical"] = bool(torch.equal(g_dense, g_sparse))
    mt, kb = cp // 256, ld4 // 128
    nnz_blocks = int(eng.kb_table[mt].item())
    out["nonzero_blocks"], out["all_blocks"] = nnz_blocks, mt * kb
    ms = {"full_dense": timed(dense, args.reps), "full_sparse": timed(sparse, args.reps),
          "rescore_1pct_dense": timed(re_dense, args.reps), "rescore_1pct_sparse": timed(re_sparse, args.reps)}
    out["ms"] = ms
    # live ceilings measured in this run
    o = ctypes.c_double()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _native.call("bmf_probe_mma_rate", 1, 4096, None)
    e0.record()
    _native.call("bmf_probe_mma_rate", 1, 4096, ctypes.byref(o))
    e1.record()
    torch.cuda.synchronize()
    probe_tops = o.value / (e0.elapsed_time(e1) / 1e3) / 1e12
    src = torch.empty((1 << 31,), dtype=torch.uint8, device=device.dev())
    dst = torch.empty_like(src)
    copy_ms = timed(lambda: dst.copy_(src), 5)
    copy_gbs = 2 * src.numel() / (copy_ms / 1e3) / 1e9                             # read + write
    del src, dst
    st_total = rows_pad // F4_ROW_PAD
    per_block = 2.0 * 256 * F4_ROW_PAD * 256                                       # both sub-tiles, 256 K elements
    for name, blocks, t in (("full_dense", mt * kb, ms["full_dense"]), ("full_sparse", nnz_blocks, ms["full_sparse"])):
        mma_tops = st_total * blocks * per_block / (t / 1e3) / 1e12
        need = rows_pad * ld4 + blocks * 256 * 128                                # rows plane once + the candidate blocks
        out[name] = {"executed_mma_tops": mma_tops, "frac_of_probe": mma_tops / probe_tops,
                     "operand_gbs": need / (t / 1e3) / 1e9, "frac_of_copy": need / (t / 1e3) / 1e9 / copy_gbs}
    out["probe_mxf4_tops"], out["copy_gbs"] = probe_tops, copy_gbs
    out["speedup_full"] = ms["full_dense"] / ms["full_sparse"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
