"""Device-resident state of one Asso fit: bit-packed X and cover, candidate basis, packed-E2M1 / int8 operand
planes, and the greedy loop as ONE enqueued sequence  select -> apply (+ compaction) -> re-score -> all-reduce  per step
(`enqueue_steps`; the step-wise `score_all` / `select_and_apply` pair remains for callers that want every step).

After the first full scoring pass only the rows a winner changed are re-scored (`rescore='incremental'`, exact);
`rescore='full'` runs a whole contraction per step.

Rows of X are sharded across ranks when torch.distributed is initialised (one process per
GPU); the candidate basis, V and the greedy decisions are replicated.  Integer partial
gains (and the step's three counters, in the tail of the same buffer) are summed with ONE all-reduce per greedy step,
so every rank sees identical totals and takes the identical lowest-index strict argmax (SURVEY.md section 8e).
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import scipy.sparse as sp
import torch

from . import _native, device

ROW_ALIGN = 256        # shard boundaries are multiples of the MMA N tile (and of 64-bit u words)
F4_ROW_PAD = 496       # BMF_F4_SUPER_ROWS: data rows of the FP4 planes are padded to whole super tiles (256 + 240)


def integer_weights(w_fp, w_fn, max_int=127, max_shift=30):
    """(a, b, s) with w_fp = a/2^s and w_fn = b/2^s exactly and 0 <= a, b <= 127, else None.

    When it exists, every product and sum of the reference's fp64 score expression
    (PyBMF/utils/metrics.py:201) is exact, so `s_new > s_old` <=> b*P - a*N > 0 and the
    score is 2^-s times an integer: one signed int8 contraction decides everything."""
    for s in range(max_shift + 1):
        a, b = w_fp * (1 << s), w_fn * (1 << s)
        if a == int(a) and b == int(b):
            a, b = int(a), int(b)
            if 0 <= a <= max_int and 0 <= b <= max_int and (a | b):
                return a, b, s
            return None
    return None


class ShardPlan:
    """Contiguous row ranges per rank, aligned to ROW_ALIGN (pure host logic, CPU-testable)."""

    def __init__(self, m: int, world: int):
        per = device.round_up(-(-m // max(world, 1)), ROW_ALIGN)
        self.m, self.world = m, world
        self.bounds = [(min(r * per, m), min((r + 1) * per, m)) for r in range(world)]

    def rows(self, rank: int):
        return self.bounds[rank]


def dist_ctx():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def local_plan(X):
    """(plan, r0, r1): ShardPlan of X's rows over the ranks of the process group and this rank's rows.  A
    generate.DeviceBits or DeviceEntries must hold exactly those rows, else ValueError (raised before any collective)."""
    rank, world = dist_ctx()
    plan = ShardPlan(X.shape[0], world)
    r0, r1 = plan.rows(rank)
    if hasattr(X, "r0") and (X.r0, X.r1) != (r0, r1):
        raise ValueError("device rows [%d, %d) must follow ShardPlan(m, world).rows(rank) = [%d, %d)"
                         % (X.r0, X.r1, r0, r1))
    return plan, r0, r1


def all_reduce_sum(t):
    """In-place integer SUM across ranks (NCCL on GPU tensors, gloo on CPU tensors in tests)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


class _Trace:
    """BMF_FIT_TRACE=1: wall-clock phases of a fit (with a device sync at every mark), printed by rank 0."""

    def __init__(self):
        self.on = os.environ.get("BMF_FIT_TRACE", "0") == "1"
        self.t = self.t0 = time.perf_counter()
        self.rows = []

    def mark(self, name):
        if not self.on:
            return
        torch.cuda.synchronize()
        now = time.perf_counter()
        self.rows.append((name, now - self.t))
        self.t = now

    def dump(self, rank):
        if self.on and rank == 0:
            agg = {}
            for name, dt in self.rows:
                agg[name] = agg.get(name, 0.0) + dt
            print("[fit trace] " + "  ".join("%s=%.1fms" % (k, 1e3 * v) for k, v in agg.items()), file=sys.stderr)


class CoverEngine:
    """All device buffers and kernel launches behind Asso.init_model / Asso._fit."""

    def __init__(self, X: sp.csr_matrix, w_fp: float, w_fn: float, scorer: str = "auto", assoc: str = "auto",
                 rescore: str = "auto"):
        _native.require_gpu()
        self.trace = _Trace()
        self.rank, self.world = dist_ctx()
        self.m, self.n = X.shape
        self.plan, r0, r1 = local_plan(X)
        self.r0, self.r1 = r0, r1
        self.m_loc = r1 - r0
        # Each rank takes only ITS rows (a view, no copy).  The packer ORs bits, so unsorted or duplicate column
        # indices need no host-side canonicalisation; explicitly stored zeros do matter, but scanning 1e8 values
        # takes the host ~0.1 s, so the scan runs in build_basis() WHILE the GPU packs and computes X^T X, and only
        # a matrix that really stores zeros (rare) is cleaned and rebuilt.  |X| is counted on the device.
        self._ctor_args = (w_fp, w_fn, scorer, assoc, rescore)
        on_device = hasattr(X, "bits") and hasattr(X, "r0")     # generate.DeviceBits: this rank's rows are already bit rows
        if on_device:
            Xl = None
        else:
            Xl = device.csr_rows_view(X, r0, r1)
        self._host_rows = Xl
        self.trace.mark("host_csr")
        self.w_fp, self.w_fn = float(w_fp), float(w_fn)
        iw = integer_weights(self.w_fp, self.w_fn)
        self.wa, self.wb, self.shift = iw if iw else (0, 0, 0)
        self.integer_mode = iw is not None
        # scorer: 'auto' / 'tcgen05' pick the fastest exact tensor-core path (FP4 when the operand values are E2M1
        # numbers, else int8); 'tcgen05_i8' / 'tcgen05_f4' force one; 'popc' is the bit-packed AND+POPC variant
        operand = os.environ.get("BMF_OPERAND", "auto")
        if scorer in ("tcgen05_i8", "tcgen05_f4"):
            operand, scorer = scorer[-2:], "tcgen05"
        if scorer == "auto":
            scorer = "tcgen05"
        assert scorer in ("tcgen05", "popc") and assoc in ("auto", "tcgen05", "tcgen05_i8", "tcgen05_f4", "popc")
        assert operand in ("auto", "i8", "f4")
        self.scorer = scorer
        # operand encoding of the rows plane (see include/pybmf_b200.h):
        #   integer mode, all give D = wb*P - wa*N exactly:
        #   "zero"  : uncovered one -> wa+wb, uncovered zero -> 0, covered -> wa, bias wa*|b_j| in the epilogue
        #   "signed": uncovered one -> +wb,   uncovered zero -> -wa, covered -> 0
        #   general (non-dyadic) weights:
        #   "pq"    : interleaved 0/1 planes P = x & ~c and Q = c per 128 rows; the epilogue gets P and
        #             N = |b_j| - Q - P per element and evaluates the reference's fp64 row test literally
        enc = os.environ.get("BMF_PLANE_ENCODING", "zero")
        if enc == "zero" and self.wa + self.wb > 127:
            enc = "signed"
        if not self.integer_mode:
            enc = "pq"
        self.encoding = enc
        self.plane_sign = -1 if enc == "signed-" else 1
        self.cand_pop = None
        self._cand_pop_host = None
        # FP4 (tcgen05 kind::mxf4, twice the int8 rate): exact when the plane values 0 / wa / wa+wb are E2M1 numbers
        lib = _native.load()
        f4_ok = (enc == "pq") or (self.integer_mode and enc == "zero" and lib.bmf_e2m1_code(self.wa) >= 0
                                  and lib.bmf_e2m1_code(self.wa + self.wb) >= 0)       # the P/Q planes are 0/1: always fine
        if max(self.wa + self.wb, 1) * self.n >= (1 << 24):    # every partial sum must stay an exact FP32 integer
            f4_ok = False
        if operand == "f4" and scorer == "tcgen05" and not f4_ok:
            raise ValueError("the FP4 scorer needs integer weights whose values wa=%d and wa+wb=%d are E2M1 numbers "
                             "(0, 1, 2, 3, 4, 6) and (wa+wb)*n < 2^24" % (self.wa, self.wa + self.wb))
        self.operand = "f4" if (scorer == "tcgen05" and f4_ok and operand in ("auto", "f4")) else "i8"
        if assoc in ("tcgen05_i8", "tcgen05_f4"):
            self.assoc_operand, assoc = assoc[-2:], "tcgen05"
        else:
            self.assoc_operand = "i8" if operand == "i8" else "f4"
        if max(self.r1 - self.r0, 1) >= (1 << 24):             # co-occurrence counts must stay below 2^24 for FP32
            self.assoc_operand = "i8"
        self.assoc_kind = "tcgen05" if assoc == "auto" else assoc
        # rescore: how the gain vector of step t+1 is obtained.  'full' = one whole contraction per greedy step;
        # 'incremental' = only the rows the winner used are re-scored, before and after the update (exact: no other row
        # changed state) -- integer weights on the tensor-core scorers; 'auto' picks incremental where it exists.
        rescore = os.environ.get("BMF_RESCORE", rescore)
        assert rescore in ("auto", "full", "incremental")
        can_inc = scorer == "tcgen05"                          # integer weights and general weights (P/Q planes) alike
        if rescore == "incremental" and not can_inc:
            raise ValueError("incremental rescoring needs a tensor-core scorer")
        self.rescore = "incremental" if (can_inc and rescore != "full") else "full"
        # X^T X is symmetric: on one GPU the FP4 association skips the tiles below the diagonal (with sharded rows every
        # rank needs complete row blocks for the reduce-scatter, and its share of the GEMM is 1/world anyway)
        self.assoc_symmetric = (self.world == 1 and os.environ.get("BMF_ASSOC_SYMMETRIC", "1") == "1")
        self.cnt_is_upper = False

        self.words = device.words_for(self.n)
        self.words_m = device.words_for(max(self.m_loc, 1))
        self.ld = device.round_up(self.n, 128)                  # K extent of the int8 cover planes (bytes)
        self.ld4 = device.round_up(self.n, 256) // 2            # ... of the packed FP4 planes (bytes)
        m_alloc = max(self.m_loc, 1)
        self.cnt = None
        self.launches = 0
        self._ip = self._ix = None
        if on_device:
            self.x_bits = X.bits
        elif self.assoc_kind == "tcgen05" and self.assoc_operand == "f4" and self.m_loc > 0:
            self._upload_pack_associate(Xl)                     # chunked: H2D of chunk c+1 overlaps X^T X of chunk c
        else:
            self._ip, self._ix = device.upload_csr(Xl)
            self.x_bits = device.pack_csr(self._ip, self._ix, self.m_loc, self.n)
        ones = device.zeros((3,), torch.int64)
        if self.m_loc > 0:                                      # |X| of this rank's rows: TP of X against itself
            _native.call("bmf_confusion_bits", self.x_bits, self.x_bits, self.m_loc, self.words, -1, ones, None, None)
        all_reduce_sum(ones)
        self._ones = ones                                       # read (one sync) at the end of build_basis()
        self.sum_x = None
        self.trace.mark("h2d_pack")
        self.c_bits = device.zeros((m_alloc, self.words), torch.int64)
        self.tp_old = device.zeros((m_alloc,), torch.int32)
        self.fp_old = device.zeros((m_alloc,), torch.int32)
        self.alive = device.zeros((self.n,), torch.uint8)
        self.basis_bits = device.zeros((self.n, self.words), torch.int64)
        self.cand_pad = device.round_up(self.n, 256)           # multiple of 256 -> the 2-SM (cta_group::2) kernel
        self.cand_plane = None
        self.rows_plane = None
        # gain buffer [gain_p | tail (8) | gain_n]: the tail carries (#used, sum P, sum N) of the last apply, so ONE
        # all-reduce per greedy step moves the gains and the counters (integer mode reduces only gain_p + tail)
        cp = self.cand_pad
        self.gbuf = device.zeros((2 * cp + 8,), torch.int64)
        self.gain_p, self.tail, self.gain_n = self.gbuf[:cp], self.gbuf[cp:cp + 8], self.gbuf[cp + 8:]
        self.red_len = cp + 8 if self.integer_mode else 2 * cp + 8
        if self.world > 1:                                      # reduced copy (select reads it; gbuf keeps the local sums)
            self.gred = device.zeros((2 * cp + 8,), torch.int64)
            self.gain_p_red, self.tail_red, self.gain_n_red = self.gred[:cp], self.gred[cp:cp + 8], self.gred[cp + 8:]
        else:
            self.gred, self.gain_p_red, self.tail_red, self.gain_n_red = self.gbuf, self.gain_p, self.tail, self.gain_n
        self.record = device.zeros((8,), torch.int64)           # [winner, score bits, used, sumP, sumN]
        self.state = device.zeros((8,), torch.int64)            # device-resident loop state (see bmf_greedy_select)
        self.nused = device.zeros((2,), torch.int32)
        self.table = None                                       # [kcap + 1, 8] per-step results
        self.u_all = None                                       # [kcap, words_m] usage bit columns
        self.comp_old = self.comp_new = self.comp_counts = None
        self.plane_stale = False
        self.score_events = None                                # bench: list of (start, end) CUDA events per scoring pass
        self.u_cols = []                                        # device bit vectors, one per chosen factor
        self.tp_tot = 0
        self.fp_tot = 0
        self.prescored = False

    # ---- association + basis (Asso.py:191-235) -------------------------------------------------
    def build_basis(self, tau: float, prescore: bool = False):
        """Association + basis (+ operand planes).  prescore=True also enqueues the first greedy step's scoring pass
        before the host-side stored-zero scan, so that the scan (35 ms for 1e8 values on 8 threads) hides behind the
        first full pass (35 ms at c4); the caller must then skip its own first pass (`self.prescored`)."""
        self._build_basis(tau)                                 # enqueued, not waited for
        if prescore:
            self.score_all()
        self.prescored = bool(prescore)
        Xl, self._host_rows = self._host_rows, None
        dirty = torch.tensor([1 if (Xl is not None and device.has_stored_zeros(Xl)) else 0], dtype=torch.int64,
                             device=device.dev())
        self.trace.mark("host_zero_scan")
        all_reduce_sum(dirty)                                  # every rank must take the same branch
        if int(dirty.item()):
            launches = self.launches
            clean = device.drop_stored_zeros(Xl)
            full = sp.csr_matrix((self.m, self.n), dtype=clean.dtype)      # this rank's rows in place, others empty
            ip = np.zeros(self.m + 1, dtype=np.int64)
            ip[self.r0 + 1:self.r1 + 1] = clean.indptr[1:]
            ip[self.r1 + 1:] = clean.indptr[-1]
            full.indptr, full.indices, full.data = ip, clean.indices, clean.data
            self.__init__(full, *self._ctor_args)
            self._host_rows = None
            self.launches += launches
            self._build_basis(tau)
            if prescore:
                self.score_all()
            self.prescored = bool(prescore)
        nb = int(self.alive.sum().item())
        self.sum_x = int(self._ones[0].item())
        self.trace.mark("basis_wait")
        return nb

    def _cnt_shape(self):
        n_pad = device.round_up(self.n, 256)
        return n_pad, max(n_pad, device.round_up(self.n, F4_ROW_PAD))   # the FP4 kernel walks data rows in super tiles of 496

    def _upload_pack_associate(self, Xl: sp.csr_matrix):
        """FP4 association path: the csr rows go up in a few chunks on a copy stream; as soon as a chunk has landed the
        main stream packs its bit rows, packs / expands its slice of X^T (K = the chunk's rows) and ACCUMULATES that
        slice's X^T X into cnt, while the copy of the next chunk is in flight (large index arrays go through
        device.stager(): threaded memcpy into a pinned ring + async DMA, ~4x the driver's single-thread pageable staging).
        At c4 the copy (38 ms pageable) and the association (36 ms) used to run back to back."""
        n, m_loc = self.n, self.m_loc
        n_pad, ldc = self._cnt_shape()
        d = device.dev()
        self.x_bits = device.zeros((m_loc, self.words), torch.int64)
        cnt = device.zeros((self._cnt_rows(n_pad), ldc), torch.int32)
        self.cnt_is_upper = self.assoc_symmetric
        nchunks = 3 if Xl.nnz >= (1 << 24) else 1
        step = device.round_up(-(-m_loc // nchunks), 256)      # chunk boundaries: multiples of 256 rows (K tiles, bit words)
        main = torch.cuda.current_stream()
        copy = device.copy_stream() if nchunks > 1 else main   # ONE copy stream per process: the caching allocator keeps a
        indptr, indices = Xl.indptr, Xl.indices                # block pool per stream, a new stream per fit strands ~0.4 GB each
        first = True
        self.trace.mark("upload_alloc")
        for a in range(0, m_loc, step):
            b = min(a + step, m_loc)
            ia, ib = int(indptr[a]), int(indptr[b])
            ip_h = torch.from_numpy(np.ascontiguousarray((indptr[a:b + 1] - indptr[a]).astype(np.int64, copy=False)))
            ix_h = torch.from_numpy(np.ascontiguousarray(indices[ia:ib].astype(np.int32, copy=False)))
            st = device.stager(self.world) if ix_h.numel() >= (1 << 22) else None     # >= 16 MB of indices
            with torch.cuda.stream(copy):
                ip_d = ip_h.to(d, non_blocking=True)
                if st is None:
                    ix_d = ix_h.to(d, non_blocking=True)       # pageable: staged by the driver on one thread (11 GB/s)
                else:
                    ix_d = torch.empty(ix_h.shape, dtype=torch.int32, device=d)
            if st is not None:
                st.upload(ix_h.numpy(), ix_d, copy)            # threaded memcpy into a pinned ring + async DMA
            self.trace.mark("upload_stage")
            with torch.cuda.stream(copy):
                landed = torch.cuda.Event()
                landed.record(copy)
            main.wait_event(landed)
            ip_d.record_stream(main)
            ix_d.record_stream(main)
            rows = b - a
            if ib > ia:
                _native.call("bmf_pack_csr", ip_d, ix_d, rows, n, 0, self.x_bits[a:b], self.words)
                xt_bits = device.pack_csr(ip_d, ix_d, rows, n, transposed=True)            # [n, words(rows)]
                ldk = device.round_up(rows, 256) // 2
                xt_plane = device.empty((max(n_pad, ldc), ldk), torch.uint8)
                _native.call("bmf_expand_bits_f4", xt_bits, None, n, rows, xt_bits.shape[1], 2, 0, 0, xt_plane,
                             xt_plane.shape[0], ldk)
                _native.call("bmf_gemm_f4_nt", xt_plane, n_pad, xt_plane, device.round_up(n, F4_ROW_PAD), ldk, cnt, ldc,
                             (0 if first else 1) | (2 if self.assoc_symmetric else 0))
                first = False
                self.launches += 4
                del xt_plane, xt_bits
        self.cnt = cnt

    def _cnt_rows(self, n_pad):
        """Rows of the count matrix: with sharded rows it is reduce-scattered in `world` equal row blocks."""
        if self.world == 1:
            return n_pad
        return self.world * (-(-n_pad // self.world))

    def counts_full(self):
        """X^T X as a full n x n int32 tensor (the symmetric GEMM leaves the part below the diagonal unwritten)."""
        c = self.cnt[: self.n, : self.n]
        if not self.cnt_is_upper:
            return c
        up = torch.triu(c)
        return up + torch.triu(c, 1).T

    def _build_basis(self, tau: float):
        n, m_loc = self.n, self.m_loc
        n_pad, ldc = self._cnt_shape()
        cnt = self.cnt if self.cnt is not None else device.zeros((self._cnt_rows(n_pad), ldc), torch.int32)
        if m_loc > 0 and self.cnt is None:
            if self._ip is None:                                # the input never was a csr (generate.DeviceBits)
                from .generate import transpose_bits
                xt_bits = transpose_bits(self.x_bits, m_loc, n)
            else:
                xt_bits = device.pack_csr(self._ip, self._ix, m_loc, n, transposed=True)
            if self.assoc_kind == "tcgen05" and self.assoc_operand == "f4":
                # X^T as packed E2M1 0/1; A operand = rows padded to 256, B operand = the same plane padded to 496
                ldk = device.round_up(m_loc, 256) // 2
                xt_plane = device.empty((max(n_pad, ldc), ldk), torch.uint8)
                _native.call("bmf_expand_bits_f4", xt_bits, None, n, m_loc, xt_bits.shape[1], 2, 0, 0, xt_plane,
                             xt_plane.shape[0], ldk)
                _native.call("bmf_gemm_f4_nt", xt_plane, n_pad, xt_plane, device.round_up(n, F4_ROW_PAD), ldk, cnt, ldc,
                             2 if self.assoc_symmetric else 0)
                self.cnt_is_upper = self.assoc_symmetric
                del xt_plane
            elif self.assoc_kind == "tcgen05":
                xt_plane = device.expand_bits_i8(xt_bits, n, m_loc, 1, 0, 256)
                _native.call("bmf_assoc_counts_i8", xt_plane, n, n_pad, xt_plane.shape[1], cnt, ldc)
                del xt_plane
            else:
                _native.call("bmf_assoc_counts_popc", xt_bits, n, xt_bits.shape[1], cnt, ldc)
            self.launches += 3
            del xt_bits
        self.trace.mark("assoc_counts")
        self.cnt = cnt
        self.cand_pop = device.zeros((max(self.cand_pad, self._cnt_rows(n_pad)),), torch.int32)
        if self.scorer == "tcgen05" and self.operand == "i8":
            self.cand_plane = device.zeros((self.cand_pad, self.ld), torch.int8)
        if self.world > 1:
            # SURVEY 8(e): partial counts -> reduce-scatter by row blocks -> every rank thresholds ITS n/R rows ->
            # all-gather of the bit rows (39.5 MB at c4 instead of all-reducing 1.28 GB of int32)
            import torch.distributed as dist
            per = cnt.shape[0] // self.world
            mine = device.empty((per, ldc), torch.int32)
            dist.reduce_scatter_tensor(mine, cnt, op=dist.ReduceOp.SUM)
            self.trace.mark("assoc_reduce_scatter")
            row0 = self.rank * per
            nrows = max(0, min(n, row0 + per) - row0)
            blk_bits = device.zeros((per, self.words), torch.int64)
            blk_alive = device.zeros((per,), torch.uint8)
            blk_pop = device.zeros((per,), torch.int32)
            if nrows > 0:
                _native.call("bmf_basis_threshold_rows", mine, ldc, n, row0, nrows, 0, float(tau), blk_bits, self.words,
                             blk_alive, blk_pop)
            all_bits = device.empty((per * self.world, self.words), torch.int64)
            all_alive = device.empty((per * self.world,), torch.uint8)
            all_pop = device.empty((per * self.world,), torch.int32)
            dist.all_gather_into_tensor(all_bits, blk_bits)
            dist.all_gather_into_tensor(all_alive, blk_alive)
            dist.all_gather_into_tensor(all_pop, blk_pop)
            self.basis_bits = all_bits[:n]
            self.alive = all_alive[:n].contiguous()
            self.cand_pop[: all_pop.shape[0]] = all_pop
            self.cnt = None                                   # only this rank's row block is complete: not kept
            self._cnt_block = (mine, row0, nrows)
            if self.cand_plane is not None:                   # int8 candidate rows from the gathered bits
                self.cand_plane = device.expand_bits_i8(self.basis_bits, n, n, 1, 0, 256, out=self.cand_plane)
            self.launches += 1
        else:
            _native.call("bmf_basis_threshold_rows", cnt, ldc, n, 0, n, 1 if self.cnt_is_upper else 0, float(tau),
                         self.basis_bits, self.words, self.alive, self.cand_pop)
            if self.cand_plane is not None:
                self.cand_plane = device.expand_bits_i8(self.basis_bits, n, n, 1, 0, 256, out=self.cand_plane)
            self.launches += 1
        if self.scorer == "tcgen05" and self.operand == "f4":   # candidate rows as packed E2M1 0/1
            self.cand_plane = device.empty((self.cand_pad, self.ld4), torch.uint8)
            _native.call("bmf_expand_bits_f4", self.basis_bits, None, n, n, self.words, 2, 0, 0, self.cand_plane,
                         self.cand_pad, self.ld4)
            self.launches += 1
        if self.scorer == "tcgen05":
            self._rebuild_rows_plane()
        self.trace.mark("basis_planes")

    def _rebuild_rows_plane(self):
        """rows_plane[i][k] = 0 if covered, +wb if x, -wa otherwise (the signed operand of D = wb*P - wa*N)."""
        self.plane_stale = False
        if self.encoding == "pq" and self.operand == "f4":
            if self.rows_plane is None:
                self.rows_plane = device.empty((2 * device.round_up(max(self.m_loc, 1), 120), self.ld4), torch.uint8)
            if self.m_loc > 0:
                _native.call("bmf_expand_bits_pq_f4", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                             self.rows_plane, self.ld4)
            self.launches += 1
            return
        if self.encoding == "pq":
            if self.rows_plane is None:
                self.rows_plane = device.empty((2 * device.round_up(max(self.m_loc, 1), 128), self.ld), torch.int8)
            if self.m_loc > 0:
                _native.call("bmf_expand_bits_pq", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                             self.rows_plane, self.ld)
            self.launches += 1
            return
        one, zero, covered = self._plane_values()
        if self.operand == "f4":
            lib = _native.load()
            rows_pad = device.round_up(max(self.m_loc, 1), F4_ROW_PAD)
            if self.rows_plane is None:
                self.rows_plane = device.empty((rows_pad, self.ld4), torch.uint8)
            _native.call("bmf_expand_bits_f4", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         lib.bmf_e2m1_code(one), 0, lib.bmf_e2m1_code(covered), self.rows_plane, rows_pad, self.ld4)
            self.launches += 1
            return
        self.rows_plane = device.expand_bits_i8(self.x_bits, self.m_loc, self.n, one, zero, 256,
                                                mask=self.c_bits, out=self.rows_plane, masked=covered)
        self.launches += 1

    def _plane_values(self):
        """(uncovered one, uncovered zero, covered) byte values of the rows plane."""
        if self.encoding == "zero":
            return self.wa + self.wb, 0, self.wa
        sg = self.plane_sign
        return sg * self.wb, -sg * self.wa, 0

    def assoc_host(self):
        """The reference's `assoc` attribute (n x n float64) from the device counts."""
        cnt = self.counts_full().cpu().numpy().astype(np.float64)
        s = np.diag(cnt).copy()
        out = np.zeros_like(cnt)
        nz = s > 0
        out[nz] = cnt[nz] / s[nz][:, None]
        return out

    def basis_host(self):
        """Remaining candidate rows (alive only, original order) as uint8 [nb, n]."""
        B = device.bits_to_host(self.basis_bits, self.n)
        return B[self.alive.cpu().numpy().astype(bool)]

    # ---- one greedy step (Asso.py:62-110) ------------------------------------------------------
    def score_all(self):
        """One full scoring pass + the exchange (step-wise API: tests, bench `value` loop, rescore='full')."""
        self._score_into_gains()
        self._reduce_gains()

    def _reduce_gains(self, tail_only=False):
        """Local gains (+ the three counters of the last apply) -> sums over all ranks: ONE all-reduce per greedy step."""
        if self.world == 1:
            return
        if tail_only:
            self.tail_red.copy_(self.tail)
            all_reduce_sum(self.tail_red)
            return
        self.gred[: self.red_len].copy_(self.gbuf[: self.red_len])
        all_reduce_sum(self.gred[: self.red_len])

    def select_and_apply(self, best_score: float):
        """argmax + apply without a host round trip in between; one small D2H read at the end.
        Returns (winner, score, n_used, sum_p, sum_n) with winner = -1 when nothing beats best_score."""
        base_int = self.wb * self.tp_tot - self.wa * self.fp_tot
        scale = 1.0 / float(1 << self.shift)
        self.record.zero_()
        _native.call("bmf_select_first_max", self.gain_p_red, self.gain_n_red if not self.integer_mode else None,
                     self.alive, self.n, self.wa, self.wb, base_int, scale, self.w_fp, self.w_fn, self.tp_tot,
                     self.fp_tot, float(best_score), self.record)
        u_bits = device.zeros((self.words_m,), torch.int64)
        if self.m_loc > 0 and self.scorer == "tcgen05" and self.encoding == "pq" and self.operand == "f4":
            _native.call("bmf_cover_apply_f4_general", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.w_fp, self.w_fn,
                         self.rows_plane, self.ld4, u_bits, self.record[2:5])
        elif self.m_loc > 0 and self.scorer == "tcgen05" and self.encoding == "pq":
            _native.call("bmf_cover_apply_general", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.w_fp, self.w_fn,
                         self.rows_plane, self.ld, u_bits, self.record[2:5])
        elif self.m_loc > 0 and self.scorer == "tcgen05" and self.operand == "f4":
            _native.call("bmf_cover_apply_f4", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.wa, self.wb,
                         self.rows_plane, self.ld4, _native.load().bmf_e2m1_code(self.wa), u_bits, self.record[2:5])
        elif self.m_loc > 0:
            _native.call("bmf_cover_apply", self.x_bits, self.c_bits, self.m_loc, self.n, self.words, self.basis_bits,
                         self.alive, self.record, self.tp_old, self.fp_old, self.wa, self.wb, self.w_fp, self.w_fn,
                         self.rows_plane, self.ld, self._plane_values()[2] if self.scorer == "tcgen05" else 0,
                         u_bits, self.record[2:5])
        self.launches += 2
        if self.world > 1:
            all_reduce_sum(self.record[2:5])
        rec = self.record.cpu().numpy()
        winner = int(rec[0])
        if winner < 0:
            return -1, float(best_score), 0, 0, 0
        if self.m_loc == 0:
            self.alive[winner] = 0                            # bmf_cover_apply does this on ranks that own rows
        score = float(rec[1:2].view(np.float64)[0])
        used, sp_, sn_ = int(rec[2]), int(rec[3]), int(rec[4])
        self.u_cols.append(u_bits)
        self.tp_tot += sp_
        self.fp_tot += sn_
        return winner, score, used, sp_, sn_

    # ---- the device-resident greedy loop (Asso.py:62-110 without a host round trip per step) -----------------
    def ensure_capacity(self, kcap: int):
        """Per-step result table and usage bit columns for `kcap` greedy steps (+ compact planes when incremental)."""
        if self.table is None or self.table.shape[0] < kcap + 1:
            table = device.zeros((kcap + 1, 8), torch.int64)
            u_all = device.zeros((kcap, self.words_m), torch.int64)
            if self.table is not None:
                table[: self.table.shape[0]] = self.table
                u_all[: self.u_all.shape[0]] = self.u_all
            self.table, self.u_all = table, u_all
        if self.rescore == "incremental" and self.comp_old is None and self.m_loc > 0:
            rows, ld = self.rows_plane.shape
            dt = self.rows_plane.dtype
            self.comp_old = device.empty((rows, ld), dt)           # capacity = every row: a winner can use them all;
            self.comp_new = device.empty((rows, ld), dt)           # bmf_cover_apply_compact writes whole rows incl. K padding
            if self.encoding == "pq":                              # general weights: the used rows' TP / FP before / after
                self.comp_counts = device.zeros((4, self.m_loc), torch.int32)

    def _score_into_gains(self):
        """One FULL scoring pass of the current cover into the local gain vector(s) (kernel only, no exchange)."""
        ev = None
        if self.score_events is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record(torch.cuda.current_stream())
        if self.m_loc == 0:
            _native.call("bmf_fill_zero", self.gbuf, 8 * self.cand_pad)
            if not self.integer_mode:
                _native.call("bmf_fill_zero", self.gain_n, 8 * self.cand_pad)
        else:
            if self.scorer == "tcgen05" and self.plane_stale:
                self._rebuild_rows_plane()
            self._launch_scorer()
        if ev is not None:
            ev[1].record(torch.cuda.current_stream())
            self.score_events.append(ev)

    def _launch_scorer(self):
        if self.scorer == "tcgen05" and self.encoding == "pq" and self.operand == "f4":
            _native.call("bmf_cover_score_f4_general", self.cand_plane, self.cand_pad, self.rows_plane, self.m_loc,
                         self.ld4, self.cand_pop, self.tp_old, self.fp_old, self.w_fp, self.w_fn, self.gain_p,
                         self.gain_n)
        elif self.scorer == "tcgen05" and self.encoding == "pq":
            _native.call("bmf_cover_score_i8_general", self.cand_plane, self.cand_pad, self.rows_plane, self.m_loc,
                         self.ld, self.cand_pop, self.tp_old, self.fp_old, self.w_fp, self.w_fn, self.gain_p,
                         self.gain_n)
        elif self.scorer == "tcgen05" and self.operand == "f4":
            _native.call("bmf_cover_score_f4", self.cand_plane, self.cand_pad, self.rows_plane,
                         self.rows_plane.shape[0], self.ld4, self.cand_pop, self.wa, self.gain_p)
        elif self.scorer == "tcgen05":
            _native.call("bmf_cover_score_i8", self.cand_plane, self.cand_pad, self.rows_plane,
                         self.rows_plane.shape[0], self.ld, self.plane_sign,
                         self.cand_pop if self.encoding == "zero" else None, self.wa, self.gain_p)
        else:
            _native.call("bmf_cover_score_popc", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.tp_old, self.fp_old, self.wa, self.wb, self.w_fp,
                         self.w_fn, self.gain_p, self.gain_n)
        self.launches += 1

    def first_pass(self):
        """Gains of the empty cover (enqueued by init_model so that host work hides behind it)."""
        self._score_into_gains()
        self._reduce_gains()

    def enqueue_steps(self, t0: int, count: int, rescore_last: bool = True):
        """Enqueue greedy steps t0 .. t0+count-1: select -> apply -> re-score -> exchange, all on the device.
        Precondition: the (reduced) gain vector describes the cover before step t0.  rescore_last=False skips the
        re-scoring after the final step (the caller knows the loop ends there)."""
        self.ensure_capacity(t0 + count)
        scale = 1.0 / float(1 << self.shift)
        gn_red = None if self.integer_mode else self.gain_n_red
        for t in range(t0, t0 + count):
            _native.call("bmf_greedy_select", self.gain_p_red, gn_red, self.tail_red, self.tail, self.alive, self.n,
                         self.wa, self.wb, scale, self.w_fp, self.w_fn, 1 if t == 0 else 0, self.state, self.table[t],
                         self.table[t - 1] if t > 0 else None, self.record, self.nused)
            self.launches += 1
            last = (t == t0 + count - 1) and not rescore_last
            self._apply_winner(t, compact=(self.rescore == "incremental" and not last))
            if last:
                self._reduce_gains(tail_only=True)
            else:
                if self.rescore == "incremental":
                    self._rescore_used_rows()
                else:
                    self._score_into_gains()
                self._reduce_gains()
            if len(self.u_cols) <= t:
                self.u_cols.extend([None] * (t + 1 - len(self.u_cols)))
            self.u_cols[t] = self.u_all[t]
        # fold the last step's counters into the state and its table row
        _native.call("bmf_greedy_select", self.gain_p_red, gn_red, self.tail_red, self.tail, self.alive, self.n, self.wa,
                     self.wb, scale, self.w_fp, self.w_fn, 0, self.state, None, self.table[t0 + count - 1], self.record,
                     self.nused)
        self.launches += 1

    def _apply_winner(self, t: int, compact: bool):
        """bmf_cover_apply* for the winner in self.record: usage column t, cover, per-row counters, counters into the
        gain tail; incremental mode also compacts the used rows' operand rows before / after the update."""
        if self.m_loc == 0:
            return
        u_bits = self.u_all[t]
        lib = _native.load()
        if self.rescore == "incremental" and self.encoding == "pq":
            kind = 3 if self.operand == "f4" else 4
            cc = self.comp_counts
            _native.call("bmf_cover_apply_compact_general", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.w_fp, self.w_fn,
                         kind if compact else 0, self.comp_old, self.comp_new, self.comp_old.shape[1], self.m_loc,
                         self.nused, cc[0], cc[1], cc[2], cc[3], u_bits, self.tail)
            self.plane_stale = True
            self.launches += 2 if compact else 1
            return
        if self.rescore == "incremental":
            if self.operand == "f4":
                kind, (one, zero, cov) = 1, [lib.bmf_e2m1_code(v) for v in self._plane_values()]
                tile = F4_ROW_PAD
            else:
                kind, (one, zero, cov) = 2, self._plane_values()
                tile = 256
            _native.call("bmf_cover_apply_compact", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.wa, self.wb,
                         kind if compact else 0, one, zero, cov, self.comp_old, self.comp_new,
                         self.comp_old.shape[1], self.comp_old.shape[0], tile, self.nused, u_bits, None, 0, 0, None,
                         self.tail)
            self.plane_stale = True                            # the big plane is no longer patched
            self.launches += 2 if compact else 1
            return
        if self.scorer == "tcgen05" and self.encoding == "pq" and self.operand == "f4":
            _native.call("bmf_cover_apply_f4_general", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.w_fp, self.w_fn,
                         self.rows_plane, self.ld4, u_bits, self.tail)
        elif self.scorer == "tcgen05" and self.encoding == "pq":
            _native.call("bmf_cover_apply_general", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.w_fp, self.w_fn,
                         self.rows_plane, self.ld, u_bits, self.tail)
        elif self.scorer == "tcgen05" and self.operand == "f4":
            _native.call("bmf_cover_apply_f4", self.x_bits, self.c_bits, self.m_loc, self.n, self.words,
                         self.basis_bits, self.alive, self.record, self.tp_old, self.fp_old, self.wa, self.wb,
                         self.rows_plane, self.ld4, lib.bmf_e2m1_code(self.wa), u_bits, self.tail)
        else:
            _native.call("bmf_cover_apply", self.x_bits, self.c_bits, self.m_loc, self.n, self.words, self.basis_bits,
                         self.alive, self.record, self.tp_old, self.fp_old, self.wa, self.wb, self.w_fp, self.w_fn,
                         self.rows_plane if self.scorer == "tcgen05" else None, self.ld,
                         self._plane_values()[2] if self.scorer == "tcgen05" else 0, u_bits, self.tail)
        self.launches += 1

    def _rescore_used_rows(self):
        """gain += sum_{used rows} relu(D after) - relu(D before): two small scoring GEMMs over the compacted rows."""
        if self.m_loc == 0:
            return
        cap = self.comp_old.shape[0]
        if self.encoding == "pq":
            cc = self.comp_counts
            fn = "bmf_cover_rescore_f4_general" if self.operand == "f4" else "bmf_cover_rescore_i8_general"
            ld = self.ld4 if self.operand == "f4" else self.ld
            for plane, tp, fp, sign in ((self.comp_old, cc[0], cc[1], -1), (self.comp_new, cc[2], cc[3], 1)):
                _native.call(fn, self.cand_plane, self.cand_pad, plane, self.m_loc, ld, self.cand_pop, tp, fp, self.w_fp,
                             self.w_fn, self.nused, sign, self.gain_p, self.gain_n)
            self.launches += 2
            return
        for plane, sign in ((self.comp_old, -1), (self.comp_new, 1)):
            if self.operand == "f4":
                _native.call("bmf_cover_rescore_f4", self.cand_plane, self.cand_pad, plane, cap, self.ld4, self.cand_pop,
                             self.wa, self.nused, sign, self.gain_p)
            else:
                _native.call("bmf_cover_rescore_i8", self.cand_plane, self.cand_pad, plane, cap, self.ld, self.plane_sign,
                             self.cand_pop if self.encoding == "zero" else None, self.wa, self.nused, sign, self.gain_p)
        self.launches += 2

    def read_table(self, t0: int, t1: int) -> np.ndarray:
        """Rows t0..t1-1 of the per-step table (one D2H, the only sync of the loop)."""
        return self.table[t0:t1].cpu().numpy()

    def rollback(self, t_keep: int, discarded_winners, kept, best_score: float):
        """After the reference's truncation quirk D1 at step t_keep-1: speculative steps >= t_keep are void.  Their
        winners return to the candidate list, the cover is rebuilt from the factors in `kept` (Asso.py:80 recomputes
        X_pd from the truncated U, V), the inherited threshold is `best_score`, and the gains are re-scored in full."""
        for w in discarded_winners:
            if w >= 0:
                self.alive[int(w)] = 1
        if self.u_all is not None and t_keep < self.u_all.shape[0]:
            self.u_all[t_keep:].zero_()
            self.table[t_keep:].zero_()
        self.reset_cover(kept)
        st = np.zeros(8, dtype=np.int64)
        st[0] = np.float64(best_score).view(np.int64)
        st[1], st[2], st[4] = self.tp_tot, self.fp_tot, t_keep
        self.state.copy_(torch.from_numpy(st).to(self.state.device))
        self.tail.zero_()
        if self.world > 1:
            self.tail_red.zero_()
        self._score_into_gains()
        self._reduce_gains()

    def basis_row_host(self, j: int) -> np.ndarray:
        return device.words_to_dense(self.basis_bits[j:j + 1].cpu().numpy(), self.n)[0]

    def basis_rows_host(self, js) -> np.ndarray:
        idx = torch.as_tensor(list(js), dtype=torch.int64, device=device.dev())
        return device.words_to_dense(self.basis_bits[idx].cpu().numpy(), self.n)

    def cand_pop_host(self, j: int) -> int:
        """|b_j| from a host copy of the per-candidate popcounts (one D2H per fit instead of one per greedy step)."""
        if self._cand_pop_host is None:
            self._cand_pop_host = self.cand_pop[: self.n].cpu().numpy()
        return int(self._cand_pop_host[j])

    def gather_used_words(self, ids):
        """Bit columns `ids` of U over ALL ranks' rows, still packed: a list of (uint64 words [len(ids), w_r], rows_r),
        one entry per rank in row order (one device all-gather + D2H; unpacking is host work, see unpack_used)."""
        if not ids:
            return []
        local = torch.stack([self.u_cols[i] for i in ids])                       # [c, words_m]
        if self.world == 1:
            return [(local.cpu().numpy(), self.m_loc)]
        import torch.distributed as dist
        wmax = device.words_for(self.plan.rows(0)[1] - self.plan.rows(0)[0])
        padded = device.zeros((len(ids), wmax), torch.int64)
        padded[:, : local.shape[1]] = local
        gathered = device.empty((self.world, len(ids), wmax), torch.int64)
        dist.all_gather_into_tensor(gathered, padded)
        both = gathered.cpu().numpy()                                            # one D2H
        return [(both[r], self.plan.rows(r)[1] - self.plan.rows(r)[0]) for r in range(self.world)]

    @staticmethod
    def unpack_used(parts, ncols_live) -> np.ndarray:
        """Packed parts of gather_used_words -> uint8 [m, ncols_live]."""
        if not parts:
            return np.zeros((0, ncols_live), np.uint8)
        return np.ascontiguousarray(np.concatenate([device.words_to_dense(w, rows).T for w, rows in parts], axis=0))

    def gather_used_columns(self, ids) -> np.ndarray:
        """Columns `ids` of U over ALL ranks' rows as uint8 [m, len(ids)]."""
        if not ids:
            return np.zeros((self.m, 0), np.uint8)
        return self.unpack_used(self.gather_used_words(ids), len(ids))

    def basis_words_host(self, js) -> np.ndarray:
        idx = torch.as_tensor(list(js), dtype=torch.int64, device=device.dev())
        return self.basis_bits[idx].cpu().numpy()

    # ---- cover rebuilt from a factor list (after the reference's truncation quirk D1) -----------
    def reset_cover(self, kept):
        """Recompute c_bits / tp_old / fp_old / rows_plane from the factors in `kept`, a list of
        (u_col index, basis row index): the reference recomputes X_pd from the (possibly
        truncated) U, V at the top of every step (Asso.py:80, BaseModelTools.py:392-393)."""
        self.c_bits.zero_()
        self.tp_old.zero_()
        self.fp_old.zero_()
        self.tp_tot = self.fp_tot = 0
        if kept:
            counts = device.zeros((3,), torch.int64)
            if self.m_loc > 0:                                 # only ranks that own rows launch kernels ...
                k = len(kept)
                kw = (k + 63) // 64
                cols = [device.words_to_dense(self.u_cols[ui].cpu().numpy().reshape(1, -1), self.m_loc)[0]
                        for (ui, _j) in kept]
                uw = torch.from_numpy(device.dense_to_words(np.stack(cols, axis=1), words=kw)).to(device.dev())
                vt = torch.stack([self.basis_bits[j] for (_ui, j) in kept]).contiguous()
                _native.call("bmf_bool_product", uw, self.m_loc, kw, vt, k, self.words, self.c_bits)
                _native.call("bmf_confusion_bits", self.x_bits, self.c_bits, self.m_loc, self.words, -1, counts,
                             self.tp_old, self.fp_old)
                self.launches += 2
            all_reduce_sum(counts)                             # ... but EVERY rank joins the exchange
            c = counts.cpu().numpy()
            self.tp_tot, self.fp_tot = int(c[0]), int(c[1])
        if self.scorer == "tcgen05":
            self._rebuild_rows_plane()
