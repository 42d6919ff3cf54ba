// Dense 0/1 contractions of the Asso hot path on the 5th-generation tensor cores (sm_100a):
//   D[j][i] = sum_k cand[j][k] * rows[i][k]      (int8 x int8 -> int32, tcgen05.mma kind::i8)
// Both operands are K-major int8 planes in HBM, moved by TMA (SWIZZLE_128B) into a 4-stage
// shared-memory ring, multiplied by a single elected thread into TMEM accumulators
// (2 x 256 columns, double buffered) and drained by four epilogue warps that apply the fused
// epilogue without writing D to HBM:
//   EPI_GAIN : gain[j] += sum_i relu(D[j][i])           (cover-gain scoring, Asso.py:83-95/144-188)
//   EPI_STORE: cnt[j][i] = D[j][i]                      (association counts X^T X, Asso.py:207)
//   EPI_GAIN2: general (non-dyadic) weights.  The data-row operand interleaves, per 128 rows, a
//              P plane (x & ~c) and a Q plane (c), so a tile's 256 accumulator columns hold
//              P[j][i] = |b_j & x_i & ~c_i| (columns 0..127) and Q[j][i] = |b_j & c_i| (128..255) for
//              the same 128 rows; N = |b_j| - Q - P, the row test is the reference's literal fp64
//              expression (metrics.py:201) and gain_p[j] += sum_use P, gain_n[j] += sum_use N.
// Candidates sit on the MMA M axis (TMEM lanes): each epilogue thread owns one candidate and
// reduces over its tile columns in registers -- no cross-lane traffic.
//
// Warp roles (192 threads, 1 CTA/SM, persistent over a grouped tile raster):
//   warp 0: TMA producer (one lane)      warp 1: TMEM allocator + MMA issuer (one lane)
//   warps 2-5: epilogue (TMEM lane quadrant = warp_id % 4)
#include <cuda.h>
#include <math.h>
#include <stdlib.h>

#include "bmf_common.cuh"

namespace bmf {
namespace tc {

constexpr int BM = BMF_I8_CAND_TILE;   // 128 candidates per tile (MMA M)
constexpr int BN = BMF_I8_ROW_TILE;    // 256 data rows per tile (MMA N)
constexpr int BK = BMF_I8_K_TILE;      // 128 bytes of K per stage = one swizzle row
constexpr int UMMA_K = 32;             // K per tcgen05.mma kind::i8
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * BK;       // 16 KB
constexpr int B_BYTES = BN * BK;       // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int NUM_THREADS = 192;
constexpr int TMEM_COLS = 512;         // 2 accumulators x 256 columns x 128 lanes x int32
constexpr int ROWSTATE_BYTES = 2 * 128 * 16;  // EPI_GAIN2: per-row (s_old, tp_old, fp_old), double buffered
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + ROWSTATE_BYTES;

enum { EPI_GAIN = 0, EPI_STORE = 1, EPI_GAIN2 = 2 };

// everything the fused epilogues need (passed by value)
struct EpiArgs {
  int sign;                        // EPI_GAIN
  const int32_t* cand_pop;         // EPI_GAIN (zero-dominant bias, nullable), EPI_GAIN2 (|b_j|, required)
  int bias_scale;                  // EPI_GAIN
  unsigned long long* gain;        // EPI_GAIN: sum relu; EPI_GAIN2: sum_use P
  unsigned long long* gain_n;      // EPI_GAIN2: sum_use N
  int32_t* C;                      // EPI_STORE
  int64_t ldc;
  int accumulate;                  // EPI_STORE (FP4 super-tile kernel): C += D instead of C = D (K split over launches)
  const int32_t* tp_old;           // EPI_GAIN2: per data row counts of the current cover
  const int32_t* fp_old;
  int64_t m_rows;                  // EPI_GAIN2: true number of data rows (the rest is padding)
  double neg_w_fp, w_fn;           // EPI_GAIN2
  uint64_t policy_a, policy_b;     // L2 eviction policy of the candidate (A) and data-row (B) TMA loads
  long long w_fn_fix, w_fp_fix;    // EPI_GAIN2 (FP4): round(w * 2^20) for the fixed-point pre-decision of the row test
  int fix_ok;                      // ... usable: weights finite and |w| < 1024
  const int32_t* dyn_rows;         // EPI_GAIN (incremental rescoring): device-side count of valid data rows; the tile grid
                                   // shrinks to ceil(*dyn_rows / tile) row tiles (nullable: all rows_pad rows are walked)
  int gain_sign;                   // EPI_GAIN: gain[j] += gain_sign * sum relu (-1 retracts the used rows' old contribution)
  int symmetric;                   // EPI_STORE (X^T X): row tiles entirely below the diagonal are skipped (C = C^T)
  const int32_t* kb_table;         // EPI_GAIN, FP4 super tiles (nullable): per candidate tile the K blocks that hold a nonzero
                                   // (layout in include/pybmf_b200.h, bmf_cover_score_f4_blocks)
  const int32_t* cand_id;          // EPI_GAIN (nullable): candidate plane row -> index of its gain and cand_pop entry
};
struct __align__(16) RowState { double s_old; int tpo; int fpo; };

// instruction descriptor (cute::UMMA::InstrDescriptor layout): dense, no saturate,
// C = S32 (2) at [4,6), A = S8 (1) at [7,10), B = S8 (1) at [10,13), K-major both,
// N>>3 at [17,23), M>>4 at [24,29)
constexpr uint32_t IDESC_I8 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) |
                              ((uint32_t)(BM >> 4) << 24);

// L2 eviction policies for the operand streams (createpolicy encodings, as in cute::TMA::CacheHintSm90),
// selectable with BMF_L2_HINT for experiments; see dispatch_gemm for what was measured.
constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull;
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull;
constexpr uint64_t L2_EVICT_LAST = 0x14F0000000000000ull;

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                            uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
// elect_one() / warp_uniform(): see bmf_common.cuh (issue discipline of the producer and MMA warps)
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tcgen05_mma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): K-major, SWIZZLE_128B,
// rows 128 B apart, 8-row groups 1024 B apart (SBO), version 1
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr) {
  uint64_t d = (uint64_t)((addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// 32 lanes x 32 consecutive columns of int32: thread t of the warp gets lane (quadrant*32 + t)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Grouped raster: GROUP_M candidate tiles share the L2-resident candidate panel while the
// row tiles sweep; a wave of CTAs covers a near-square block of the tile grid.
__device__ __forceinline__ void tile_coords(int64_t t, int mt_total, int nt_total, int group_m, int& mt, int& nt) {
  const int64_t per_group = (int64_t)group_m * nt_total;
  const int g = (int)(t / per_group);
  const int64_t r = t - (int64_t)g * per_group;
  const int first = g * group_m;
  const int gsize = min(group_m, mt_total - first);
  mt = first + (int)(r % gsize);
  nt = (int)(r / gsize);
}


// two 32-column chunks in flight, one wait
__device__ __forceinline__ void tmem_ld_32x32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// EPI_GAIN2 on compacted rows (incremental re-scoring): the number of valid data rows comes from the device counter
__device__ __forceinline__ int64_t dyn_m_rows(const EpiArgs& ea) {
  return ea.dyn_rows != nullptr ? (int64_t)*reinterpret_cast<const volatile int32_t*>(ea.dyn_rows) : ea.m_rows;
}

// EPI_GAIN2, before the accumulator is waited for: the 128 epilogue threads of a CTA stage the state of the
// tile's 128 data rows (et = 0..127) into buffer `acc` and meet on named barrier 1.  With two buffers one
// barrier per tile is enough: a thread that passes the barrier of tile t+1 has finished reading tile t.
__device__ __forceinline__ void stage_row_state(RowState* rs, int acc, int et, int nt, const EpiArgs& ea) {
  const int64_t i = (int64_t)nt * 128 + et;
  RowState r;
  if (i < dyn_m_rows(ea)) {
    r.tpo = ea.tp_old[i];
    r.fpo = ea.fp_old[i];
    r.s_old = cover_score_f64(ea.neg_w_fp, ea.w_fn, r.fpo, r.tpo);
  } else {                                                // padding row: never used
    r.tpo = 0;
    r.fpo = 0;
    r.s_old = __longlong_as_double(0x7ff0000000000000ll);
  }
  rs[acc * 128 + et] = r;
  asm volatile("bar.sync 1, 128;" ::: "memory");
}

// One accumulator tile (this thread's TMEM lane = candidate `row`, BN columns) through the fused epilogue.
template <int EPI>
__device__ __forceinline__ void epilogue_tile(uint32_t taddr, int64_t row, int nt, const RowState* rs, const EpiArgs& ea) {
  if (EPI == EPI_GAIN2) {
    const int pop = ea.cand_pop[row];
    long long sum_p = 0, sum_n = 0;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t vp[32], vq[32];
      tmem_ld_32x32_nowait(taddr + (uint32_t)(c * 32), vp);
      tmem_ld_32x32_nowait(taddr + (uint32_t)(128 + c * 32), vq);
      tmem_ld_wait();
      int part_p = 0, part_n = 0;
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const RowState r = rs[c * 32 + q];                // same address for the whole warp: broadcast
        const int P = (int)vp[q];
        const int N = pop - (int)vq[q] - P;
        const bool use = cover_score_f64(ea.neg_w_fp, ea.w_fn, r.fpo + N, r.tpo + P) > r.s_old;
        part_p += use ? P : 0;
        part_n += use ? N : 0;
      }
      sum_p += part_p;
      sum_n += part_n;
    }
    if (sum_p | sum_n) {
      atomicAdd(ea.gain + row, (unsigned long long)(ea.gain_sign < 0 ? -sum_p : sum_p));
      atomicAdd(ea.gain_n + row, (unsigned long long)(ea.gain_sign < 0 ? -sum_n : sum_n));
    }
  } else {
    const int bias = (EPI == EPI_GAIN && ea.cand_pop != nullptr) ? ea.bias_scale * ea.cand_pop[row] : 0;
    const int sign = ea.sign;
    long long relu_sum = 0;
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + (uint32_t)(c * 32), v);
      if (EPI == EPI_GAIN) {
        int part = 0;                                     // 32 * 127 * K fits int32 for K < 5e5
#pragma unroll
        for (int q = 0; q < 32; ++q) part += max(sign * (int)v[q] - bias, 0);
        relu_sum += part;
      } else {
        int4* dst = reinterpret_cast<int4*>(ea.C + row * ea.ldc + (int64_t)nt * BN + c * 32);
#pragma unroll
        for (int q = 0; q < 8; ++q)
          dst[q] = make_int4((int)v[4 * q], (int)v[4 * q + 1], (int)v[4 * q + 2], (int)v[4 * q + 3]);
      }
    }
    if (EPI == EPI_GAIN && relu_sum != 0)
      atomicAdd(ea.gain + row, (unsigned long long)(ea.gain_sign < 0 ? -relu_sum : relu_sum));   // two's complement: exact
  }
}

// incremental rescoring: the number of row tiles comes from a device counter written by bmf_cover_apply_compact
__device__ __forceinline__ int dyn_row_tiles(const EpiArgs& ea, int nt_total, int tile_rows) {
  if (ea.dyn_rows == nullptr) return nt_total;
  const int rows = *reinterpret_cast<const volatile int32_t*>(ea.dyn_rows);
  const int nt = (rows + tile_rows - 1) / tile_rows;
  return nt < nt_total ? nt : nt_total;
}

template <int EPI>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_i8_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               int mt_total, int nt_total_in, int kb_total, int group_m, const EpiArgs ea) {
  extern __shared__ uint8_t smem_raw[];
  const int nt_total = dyn_row_tiles(ea, nt_total_in, EPI == EPI_GAIN2 ? 128 : BN);   // GAIN2: a tile = 128 P + 128 Q rows
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  // bars[0..S) full, [S..2S) empty, [2S..2S+2) tmem_full, [2S+2..2S+4) tmem_empty, then tmem base
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  RowState* row_state = reinterpret_cast<RowState*>(smem + STAGES * STAGE_BYTES + 256);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t total_tiles = (int64_t)mt_total * nt_total;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_base_slot);

  if (warp == 0) {
    // ===== TMA producer (whole warp, one elected lane issues) =====
    {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t sb = warp_uniform(smem_base);
      for (int64_t t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        int mt, nt;
        tile_coords(t, mt_total, nt_total, group_m, mt, nt);
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t a_dst = sb + stage * STAGE_BYTES;
          if (elect_one()) {
            mbar_expect_tx(full_bar(stage), STAGE_BYTES);
            tma_load_2d(a_dst, &tmap_a, full_bar(stage), kb * BK, mt * BM, ea.policy_a);
            tma_load_2d(a_dst + A_BYTES, &tmap_b, full_bar(stage), kb * BK, nt * BN, ea.policy_b);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer (whole warp, converged -- see elect_one) =====
    {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint32_t tb = warp_uniform(tmem_base), sb = warp_uniform(smem_base);
      for (int64_t t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);       // epilogue has drained this accumulator
        tcgen05_fence_after();
        const uint32_t d_tmem = tb + (uint32_t)(acc * BN);
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(full_bar(stage), phase);              // TMA bytes have landed
          tcgen05_fence_after();
          const uint32_t a_addr = sb + stage * STAGE_BYTES;
          const uint64_t da = make_smem_desc(a_addr), db = make_smem_desc(a_addr + A_BYTES);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k)
              tcgen05_mma_i8(d_tmem, da + (uint64_t)(k * (UMMA_K >> 4)), db + (uint64_t)(k * (UMMA_K >> 4)),
                             IDESC_I8, (uint32_t)((kb | k) != 0));
            tcgen05_commit(empty_bar(stage));             // smem slot free once these MMAs retire
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) tcgen05_commit(tfull_bar(acc));  // accumulator complete -> epilogue
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue warps =====
    const int quad = warp & 3;                            // TMEM lanes [32*quad, 32*quad+32)
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int64_t t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      int mt, nt;
      tile_coords(t, mt_total, nt_total, group_m, mt, nt);
      if (EPI == EPI_GAIN2) stage_row_state(row_state, acc, (int)threadIdx.x - 64, nt, ea);
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN);
      const int64_t row = (int64_t)mt * BM + quad * 32 + lane;
      epilogue_tile<EPI>(taddr, row, nt, row_state + acc * 128, ea);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));        // 4 arrivals free the accumulator
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

// ---- host side ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess || p == nullptr)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// plane[rows][ld] int8, box = box_rows x 128 bytes, 128-byte swizzle
static int make_plane_map(CUtensorMap* map, const int8_t* plane, int64_t rows, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available from the driver");
    return BMF_E_DRIVER;
  }
  cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<int8_t*>(plane), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld ld=%lld)", (int)r, (long long)rows,
              (long long)ld);
    return BMF_E_DRIVER;
  }
  return 0;
}

template <int EPI>
static int launch_gemm(const int8_t* a, int64_t a_rows, const int8_t* b, int64_t b_rows, int64_t ld,
                       const EpiArgs& ea, cudaStream_t stream) {
  CUtensorMap ma, mb;
  int rc = make_plane_map(&ma, a, a_rows, ld, BM);
  if (rc) return rc;
  rc = make_plane_map(&mb, b, b_rows, ld, BN);
  if (rc) return rc;
  static bool attr_set[3] = {false, false, false};
  if (!attr_set[EPI]) {
    rc = check_cuda(cudaFuncSetAttribute(gemm_i8_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES),
                    "cudaFuncSetAttribute(gemm_i8_kernel)");
    if (rc) return rc;
    attr_set[EPI] = true;
  }
  const int mt = (int)(a_rows / BM), nt = (int)(b_rows / BN), kb = (int)(ld / BK);
  const int64_t tiles = (int64_t)mt * nt;
  const int grid = (int)(tiles < num_sms() ? tiles : num_sms());
  int group_m = 16;                                       // candidate tiles per raster group (L2 reuse)
  if (const char* e = getenv("BMF_GROUP_M")) { int v = atoi(e); if (v >= 1 && v <= 64) group_m = v; }
  gemm_i8_kernel<EPI><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(ma, mb, mt, nt, kb, group_m, ea);
  return check_cuda(cudaGetLastError(), "gemm_i8_kernel launch");
}


// =================================================================================================
// 2-SM variant: a CTA pair (cluster 2x1x1 on one TPC) computes a 256 x 256 tile with
// tcgen05.mma.cta_group::2 (UMMA M = 256).  Each CTA stages ITS 128 candidate rows and ITS half
// (128) of the tile's data rows, so every operand byte is fetched from L2 once per pair instead of
// once per CTA, the per-CTA stage shrinks to 32 KB and the ring deepens to 6 stages.  Only the
// leader CTA issues MMAs; TMA transactions of both CTAs complete on the leader's "full" barrier,
// tcgen05.commit multicasts "empty"/"accumulator full" to both CTAs, and the epilogue warps of both
// CTAs (each draining its own 128 TMEM lanes) arrive remotely on the leader's "accumulator empty".
// =================================================================================================
namespace sm2 {
constexpr int BM2 = 256;                 // candidates per pair tile
constexpr int HALF = 128;                // rows each CTA stages per operand
constexpr int STAGES2 = 6;
constexpr int OP_BYTES = HALF * BK;      // 16 KB
constexpr int STAGE_BYTES2 = 2 * OP_BYTES;
constexpr int SMEM_BYTES2 = STAGES2 * STAGE_BYTES2 + 1024 + 256 + ROWSTATE_BYTES;
constexpr uint32_t IDESC_I8_2SM = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) |
                                  ((uint32_t)(BM2 >> 4) << 24);
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;   // clears the CTA-pair bit of a shared::cluster address

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1,
                                                uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tcgen05_commit_2sm(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void tcgen05_mma_i8_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                   uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t local_bar) {
  // arrive on the barrier at the same offset in CTA rank 0 of the pair
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(remote) : "r"(local_bar));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_i8_2sm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   int mt_total, int nt_total_in, int kb_total, int group_m, const EpiArgs ea) {
  extern __shared__ uint8_t smem_raw[];
  const int nt_total = dyn_row_tiles(ea, nt_total_in, EPI == EPI_GAIN2 ? 128 : BN);
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES2 * STAGE_BYTES2);
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES2 + 4);
  RowState* row_state = reinterpret_cast<RowState*>(smem + STAGES2 * STAGE_BYTES2 + 256);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES2 + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES2 + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES2 + 2 + a); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int64_t pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int64_t total_tiles = (int64_t)mt_total * nt_total;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES2; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();                                     // barriers of BOTH CTAs are initialised and visible
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_base_slot);

  if (warp == 0) {
    // ===== TMA producer (both CTAs: own 128 candidate rows + own 128 data rows; whole warp, one elected lane issues) =====
    {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t sb = warp_uniform(smem_base);
      for (int64_t t = pair; t < total_tiles; t += num_pairs) {
        int mt, nt;
        tile_coords(t, mt_total, nt_total, group_m, mt, nt);
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t leader_full = full_bar(stage) & PEER_MASK;
          const uint32_t a_dst = sb + stage * STAGE_BYTES2;
          if (elect_one()) {
            if (leader) mbar_expect_tx(full_bar(stage), 2 * STAGE_BYTES2);     // bytes of both CTAs
            tma_load_2d_2sm(a_dst, &tmap_a, leader_full, kb * BK, mt * BM2 + (int)rank * HALF, ea.policy_a);
            tma_load_2d_2sm(a_dst + OP_BYTES, &tmap_b, leader_full, kb * BK, nt * BN + (int)rank * HALF, ea.policy_b);
          }
          __syncwarp();
          if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA only; whole warp, converged -- see elect_one) =====
    if (leader) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint32_t tb = warp_uniform(tmem_base), sb = warp_uniform(smem_base);
      for (int64_t t = pair; t < total_tiles; t += num_pairs) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tb + (uint32_t)(acc * BN);
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t a_addr = sb + stage * STAGE_BYTES2;
          const uint64_t da = make_smem_desc(a_addr), db = make_smem_desc(a_addr + OP_BYTES);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k)
              tcgen05_mma_i8_2sm(d_tmem, da + (uint64_t)(k * (UMMA_K >> 4)), db + (uint64_t)(k * (UMMA_K >> 4)),
                                 IDESC_I8_2SM, (uint32_t)((kb | k) != 0));
            tcgen05_commit_2sm(empty_bar(stage));         // frees the slot in BOTH CTAs
          }
          __syncwarp();
          if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) tcgen05_commit_2sm(tfull_bar(acc));   // accumulator halves ready in BOTH CTAs
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue warps (both CTAs; CTA r owns candidates [r*128, r*128+128) of the tile) =====
    const int quad = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int64_t t = pair; t < total_tiles; t += num_pairs) {
      int mt, nt;
      tile_coords(t, mt_total, nt_total, group_m, mt, nt);
      if (EPI == EPI_GAIN2) stage_row_state(row_state, acc, (int)threadIdx.x - 64, nt, ea);
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN);
      const int64_t row = (int64_t)mt * BM2 + (int64_t)rank * HALF + quad * 32 + lane;
      epilogue_tile<EPI>(taddr, row, nt, row_state + acc * 128, ea);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tempty_bar(acc)); // 8 arrivals (4 warps x 2 CTAs) free the accumulator
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();                                     // nobody leaves while the pair still shares smem / TMEM
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

template <int EPI>
static int launch_gemm_2sm(const int8_t* a, int64_t a_rows, const int8_t* b, int64_t b_rows, int64_t ld,
                           const EpiArgs& ea, cudaStream_t stream) {
  CUtensorMap ma, mb;
  int rc = make_plane_map(&ma, a, a_rows, ld, HALF);
  if (rc) return rc;
  rc = make_plane_map(&mb, b, b_rows, ld, HALF);
  if (rc) return rc;
  static bool attr_set[3] = {false, false, false};
  if (!attr_set[EPI]) {
    rc = check_cuda(cudaFuncSetAttribute(gemm_i8_2sm_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES2),
                    "cudaFuncSetAttribute(gemm_i8_2sm_kernel)");
    if (rc) return rc;
    attr_set[EPI] = true;
  }
  const int mt = (int)(a_rows / BM2), nt = (int)(b_rows / BN), kb = (int)(ld / BK);
  const int64_t tiles = (int64_t)mt * nt;
  const int pairs_max = num_sms() / 2;
  const int pairs = (int)(tiles < pairs_max ? tiles : pairs_max);
  int group_m = 16;                                       // 256-row candidate tiles per raster group
  if (const char* e = getenv("BMF_GROUP_M2")) { int v = atoi(e); if (v >= 1 && v <= 64) group_m = v; }
  gemm_i8_2sm_kernel<EPI><<<2 * pairs, NUM_THREADS, SMEM_BYTES2, stream>>>(ma, mb, mt, nt, kb, group_m, ea);
  return check_cuda(cudaGetLastError(), "gemm_i8_2sm_kernel launch");
}
}  // namespace sm2


// =================================================================================================
// FP4 variant of the pair kernel: tcgen05.mma kind::mxf4 (packed E2M1 operands, block-32 UE8M0 scale factors,
// FP32 accumulators) runs at TWICE the kind::i8 rate and moves half the operand bytes.  The operands of this path
// are tiny non-negative integers -- candidate rows {0,1}, data rows {0, wa, wa+wb} -- which E2M1 represents exactly
// ({0, .5, 1, 1.5, 2, 3, 4, 6}); every product is an integer <= 6 and every partial sum an integer < 2^24, so the
// FP32 accumulation is EXACT and the epilogue converts back to the same int32 the kind::i8 kernel produces
// (tests compare the two bit for bit, also at the full Netflix-shaped size).  All scale factors are 1.0: the 32 TMEM
// columns behind the accumulators are filled once with the UE8M0 byte 0x7F, so any scale-factor layout reads 1.0.
// Tile: 256 candidates x 240 data rows (two 240-column FP32 accumulators + 32 scale columns = 512 TMEM columns),
// K = 256 elements (128 bytes) per stage, four K=64 MMAs per stage.
// =================================================================================================
namespace f4 {
using sm2::cluster_ctarank;
using sm2::cluster_sync_all;
using sm2::tma_load_2d_2sm;
using sm2::tcgen05_commit_2sm;
using sm2::mbar_arrive_leader;
using sm2::PEER_MASK;
constexpr int BM4 = 256, HALFM = 128;    // candidates per pair tile / per CTA
#ifdef BMF_F4_PROBE_BN                   /* timing experiment only (accumulator 1 overlaps the scale columns) */
constexpr int BN4 = BMF_F4_PROBE_BN;
#else
constexpr int BN4 = BMF_F4_ROW_TILE;     // 240 data rows per pair tile
#endif
constexpr int HALFN = BN4 / 2;           // 120 per CTA
#ifndef BMF_F4_STAGES
#define BMF_F4_STAGES 7
#endif
constexpr int STAGES4 = BMF_F4_STAGES;
constexpr int A_OP = HALFM * BK;         // 16 KB
constexpr int B_OP = HALFN * BK;         // 15 KB
constexpr int STAGE_BYTES4 = A_OP + B_OP;   // 31 KB, a multiple of 1024 (swizzle atom alignment)
constexpr int SMEM_BYTES4 = STAGES4 * STAGE_BYTES4 + 1024 + 256 + ROWSTATE_BYTES;
constexpr int SF_COL = 480;              // scale-factor columns [480, 512)
constexpr uint32_t SF_ONE = 0x7F7F7F7Fu; // UE8M0 1.0 in every byte
// cute::UMMA::InstrDescriptorBlockScaled: a/b format E2M1 (MXF4Format 1) at [7,10)/[10,13), K-major both,
// N>>3 at [17,23), scale format UE8M0 (1) at bit 23, M>>4 at [24,29), K = 64 (bit 31 = 0), scale-factor ids 0
constexpr uint32_t IDESC_F4 = (1u << 7) | (1u << 10) | ((uint32_t)(BN4 >> 3) << 17) | (1u << 23) |
                              ((uint32_t)(BM4 >> 4) << 24);

__device__ __forceinline__ void tcgen05_mma_f4_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                   uint32_t accumulate, uint32_t sfa, uint32_t sfb) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%6], p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(sfa), "r"(sfb)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32_x8(uint32_t taddr, uint32_t v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(v)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32_x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ int f32_bits_to_int(uint32_t bits) { return __float2int_rn(__uint_as_float(bits)); }

// The general-weights epilogue does ~20 dependent instructions per element (F2I, I2F.F64, DMUL, DADD, DSETP) and, with
// one epilogue warp per scheduler, ran at IPC ~0.2: it -- not the tensor pipe -- bounded EPI_GAIN2 (168 instead of 128
// cycles per MMA).  EPI_GAIN2 therefore runs EIGHT epilogue warps (two per TMEM lane quadrant, each taking half of the
// tile's data rows), so every scheduler has two warps to hide those latencies with.
template <int EPI> struct F4Threads { static constexpr int value = (EPI == EPI_GAIN2) ? 320 : NUM_THREADS; };

// One FP32 accumulator tile (this thread's TMEM lane = candidate `row`, 240 columns) through the fused epilogue.
// EPI_GAIN2 on FP4 tiles: 120 data rows per tile, P in columns [0, 120), Q in [120, 240)
template <int NEPI>
__device__ __forceinline__ void stage_row_state_f4(RowState* rs, int acc, int et, int nt, const EpiArgs& ea) {
  if (et < HALFN) {
    const int64_t i = (int64_t)nt * HALFN + et;
    RowState r;
    if (i < dyn_m_rows(ea)) {
      r.tpo = ea.tp_old[i];
      r.fpo = ea.fp_old[i];
      r.s_old = cover_score_f64(ea.neg_w_fp, ea.w_fn, r.fpo, r.tpo);
    } else {
      r.tpo = 0;
      r.fpo = 0;
      r.s_old = __longlong_as_double(0x7ff0000000000000ll);
    }
    rs[acc * 128 + et] = r;
  }
  asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory");
}

// `half` (EPI_GAIN2 only): which half of the tile's data rows this warp takes (chunks of 8 rows: [0, 8) and [8, 15))
template <int EPI>
__device__ __forceinline__ void epilogue_tile_f4(uint32_t taddr, int64_t row, int nt, const RowState* rs, const EpiArgs& ea,
                                                 int half) {
  if (EPI == EPI_GAIN2) {
    const int pop = ea.cand_pop[row];
    long long sum_p = 0, sum_n = 0;
    const int c_begin = half ? 8 : 0, c_end = half ? HALFN / 8 : 8;
    // B200's vector FP64 pipe is narrow: evaluating the fp64 row test for all 8.5e9 elements of a step bounds the kernel
    // (math-pipe throttle = 66 % of the stall samples).  So each element is first decided in fixed point:
    //   d = round(w_fn 2^20) P - round(w_fp 2^20) N  differs from 2^20 (w_fn P - w_fp N) by at most (P + N) / 2, and the fp64
    //   evaluation of s_new vs s_old is off by < 2^-51 |w| n, i.e. < 0.5 units of d under the host gate |w| n < 2^30 (see
    //   bmf_cover_score_f4_general), hence |d| > P + N + 2 fixes the outcome of the fp64 comparison;
    // only the undecided elements (exact or near ties such as 0.8 P = 0.2 N) go through the literal fp64 expression, one
    // per lane and pass, so the number of fp64 passes per chunk is the LARGEST per-lane count, not the number of
    // elements that are undecided in some lane.  The result is identical to evaluating fp64 everywhere.
    const long long w_fn_fix = ea.w_fn_fix, w_fp_fix = ea.w_fp_fix;
    const bool fix_ok = ea.fix_ok != 0;
#pragma unroll 1
    for (int c = c_begin; c < c_end; ++c) {
      uint32_t vp[8], vq[8];
      tmem_ld_32x32_x8(taddr + (uint32_t)(c * 8), vp);
      tmem_ld_32x32_x8(taddr + (uint32_t)(HALFN + c * 8), vq);
      tmem_ld_wait();
      int part_p = 0, part_n = 0;
      int P[8], N[8];
      uint32_t undecided = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        P[q] = f32_bits_to_int(vp[q]);
        N[q] = pop - f32_bits_to_int(vq[q]) - P[q];
        const long long d = w_fn_fix * P[q] - w_fp_fix * N[q];
        const int margin = P[q] + N[q] + 2;
        const bool use = d > margin;
        if (!fix_ok || (d <= margin && d >= -margin)) undecided |= 1u << q;
        else { part_p += use ? P[q] : 0; part_n += use ? N[q] : 0; }
      }
      while (__any_sync(0xffffffffu, undecided != 0)) {     // fp64 passes: one undecided element per lane and pass
        if (undecided) {
          const int q = __ffs((int)undecided) - 1;
          undecided &= undecided - 1;
          int Pq = 0, Nq = 0;
#pragma unroll
          for (int e = 0; e < 8; ++e) if (e == q) { Pq = P[e]; Nq = N[e]; }
          const RowState r = rs[c * 8 + q];
          if (cover_score_f64(ea.neg_w_fp, ea.w_fn, r.fpo + Nq, r.tpo + Pq) > r.s_old) { part_p += Pq; part_n += Nq; }
        }
      }
      sum_p += part_p;
      sum_n += part_n;
    }
    if (sum_p | sum_n) {
      atomicAdd(ea.gain + row, (unsigned long long)(ea.gain_sign < 0 ? -sum_p : sum_p));
      atomicAdd(ea.gain_n + row, (unsigned long long)(ea.gain_sign < 0 ? -sum_n : sum_n));
    }
    return;
  }
  const int bias = (EPI == EPI_GAIN && ea.cand_pop != nullptr) ? ea.bias_scale * ea.cand_pop[row] : 0;
  long long relu_sum = 0;
#pragma unroll 1
  for (int c = 0; c < BN4 / 16; ++c) {
    uint32_t lo[8], hi[8];
    tmem_ld_32x32_x8(taddr + (uint32_t)(c * 16), lo);
    tmem_ld_32x32_x8(taddr + (uint32_t)(c * 16 + 8), hi);
    tmem_ld_wait();
    if (EPI == EPI_GAIN) {
      int part = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) part += max(f32_bits_to_int(lo[q]) - bias, 0) + max(f32_bits_to_int(hi[q]) - bias, 0);
      relu_sum += part;
    } else {
      int4* dst = reinterpret_cast<int4*>(ea.C + row * ea.ldc + (int64_t)nt * BN4 + c * 16);
      dst[0] = make_int4(f32_bits_to_int(lo[0]), f32_bits_to_int(lo[1]), f32_bits_to_int(lo[2]), f32_bits_to_int(lo[3]));
      dst[1] = make_int4(f32_bits_to_int(lo[4]), f32_bits_to_int(lo[5]), f32_bits_to_int(lo[6]), f32_bits_to_int(lo[7]));
      dst[2] = make_int4(f32_bits_to_int(hi[0]), f32_bits_to_int(hi[1]), f32_bits_to_int(hi[2]), f32_bits_to_int(hi[3]));
      dst[3] = make_int4(f32_bits_to_int(hi[4]), f32_bits_to_int(hi[5]), f32_bits_to_int(hi[6]), f32_bits_to_int(hi[7]));
    }
  }
  if (EPI == EPI_GAIN && relu_sum != 0)
    atomicAdd(ea.gain + row, (unsigned long long)(ea.gain_sign < 0 ? -relu_sum : relu_sum));
}

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(F4Threads<EPI>::value, 1)
gemm_f4_2sm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   int mt_total, int nt_total_in, int kb_total, int group_m, const EpiArgs ea) {
  extern __shared__ uint8_t smem_raw[];
  const int nt_total = dyn_row_tiles(ea, nt_total_in, EPI == EPI_GAIN2 ? HALFN : BN4);   // GAIN2: a tile = 120 P + 120 Q rows
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES4 * STAGE_BYTES4);
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES4 + 4);
  RowState* row_state = reinterpret_cast<RowState*>(smem + STAGES4 * STAGE_BYTES4 + 256);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES4 + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES4 + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES4 + 2 + a); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int64_t pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int64_t total_tiles = (int64_t)mt_total * nt_total;

  if (threadIdx.x == 0) {
    constexpr int EPI_WARPS = F4Threads<EPI>::value / 32 - 2;               // 4, or 8 for EPI_GAIN2
    for (int s = 0; s < STAGES4; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 2 * EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_base_slot);
  if (warp >= 2 && warp < 6) {                            // unit scale factors: all 128 lanes x columns [480, 512)
    const uint32_t sf_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)SF_COL;
#pragma unroll
    for (int c = 0; c < 4; ++c) tmem_st_32x32_x8(sf_addr + (uint32_t)(c * 8), SF_ONE);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();                                     // scale factors of BOTH CTAs are in place before any MMA
  tcgen05_fence_after();

  if (warp == 0) {
    {                                                     // whole warp, converged; one elected lane issues the TMA
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t sb = warp_uniform(smem_base);
      for (int64_t t = pair; t < total_tiles; t += num_pairs) {
        int mt, nt;
        tile_coords(t, mt_total, nt_total, group_m, mt, nt);
#ifdef BMF_F4_TIMING_PROBE   /* timing experiment only: every tile re-reads tile (0, 0) -> operands always hit L2 */
        mt = 0; nt = 0;
#endif
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t leader_full = full_bar(stage) & PEER_MASK;
#if defined(BMF_F4_TIMING_PROBE) && BMF_F4_TIMING_PROBE == 2   /* no operand traffic at all: MMA issue + pipe only */
          if (leader && elect_one()) mbar_arrive(full_bar(stage));
          __syncwarp();
          if (++stage == STAGES4) { stage = 0; phase ^= 1u; }
          continue;
#endif
#if defined(BMF_F4_TIMING_PROBE) && BMF_F4_TIMING_PROBE >= 3   /* MMA warp free-runs: no producer, no stage barriers */
          break;
#endif
          const uint32_t a_dst = sb + stage * STAGE_BYTES4;
          if (elect_one()) {
            if (leader) mbar_expect_tx(full_bar(stage), 2 * STAGE_BYTES4);
            tma_load_2d_2sm(a_dst, &tmap_a, leader_full, kb * BK, mt * BM4 + (int)rank * HALFM, ea.policy_a);
            tma_load_2d_2sm(a_dst + A_OP, &tmap_b, leader_full, kb * BK, nt * BN4 + (int)rank * HALFN, ea.policy_b);
          }
          __syncwarp();
          if (++stage == STAGES4) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (leader) {                                         // whole warp, converged (see elect_one)
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint32_t tb = warp_uniform(tmem_base), sb = warp_uniform(smem_base);
      const uint32_t sfa = tb + (uint32_t)SF_COL, sfb = tb + (uint32_t)SF_COL + 8u;
      for (int64_t t = pair; t < total_tiles; t += num_pairs) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tb + (uint32_t)(acc * BN4);
        for (int kb = 0; kb < kb_total; ++kb) {
#if !defined(BMF_F4_TIMING_PROBE) || BMF_F4_TIMING_PROBE < 3
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
#endif
          const uint32_t a_addr = sb + stage * STAGE_BYTES4;
          const uint64_t da = make_smem_desc(a_addr), db = make_smem_desc(a_addr + A_OP);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k)                   // K = 64 elements = 32 bytes per MMA
              tcgen05_mma_f4_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), IDESC_F4,
                                 (uint32_t)((kb | k) != 0), sfa, sfb);
#if !defined(BMF_F4_TIMING_PROBE) || BMF_F4_TIMING_PROBE < 3 || BMF_F4_TIMING_PROBE == 5
            tcgen05_commit_2sm(empty_bar(stage));
#endif
          }
          __syncwarp();
          if (++stage == STAGES4) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) tcgen05_commit_2sm(tfull_bar(acc));
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    const int quad = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int64_t t = pair; t < total_tiles; t += num_pairs) {
      int mt, nt;
      tile_coords(t, mt_total, nt_total, group_m, mt, nt);
      if (EPI == EPI_GAIN2) stage_row_state_f4<F4Threads<EPI>::value - 64>(row_state, acc, (int)threadIdx.x - 64, nt, ea);
      mbar_wait(tfull_bar(acc), acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN4);
      const int64_t row = (int64_t)mt * BM4 + (int64_t)rank * HALFM + quad * 32 + lane;
      epilogue_tile_f4<EPI>(taddr, row, nt, row_state + acc * 128, ea, (warp - 2) >> 2);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

template <int EPI>
static int launch_gemm_f4(const uint8_t* a, int64_t a_rows, const uint8_t* b, int64_t b_rows, int64_t ld_bytes,
                          const EpiArgs& ea_in, cudaStream_t stream) {
  CUtensorMap ma, mb;
  int rc = make_plane_map(&ma, reinterpret_cast<const int8_t*>(a), a_rows, ld_bytes, HALFM);
  if (rc) return rc;
  rc = make_plane_map(&mb, reinterpret_cast<const int8_t*>(b), b_rows, ld_bytes, HALFN);
  if (rc) return rc;
  static bool attr_set[3] = {false, false, false};
  if (!attr_set[EPI]) {
    rc = check_cuda(cudaFuncSetAttribute(gemm_f4_2sm_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES4),
                    "cudaFuncSetAttribute(gemm_f4_2sm_kernel)");
    if (rc) return rc;
    attr_set[EPI] = true;
  }
  EpiArgs ea = ea_in;
  ea.policy_a = L2_EVICT_NORMAL;
  ea.policy_b = L2_EVICT_NORMAL;
  const int mt = (int)(a_rows / BM4), nt = (int)(b_rows / BN4), kb = (int)(ld_bytes / BK);
  const int64_t tiles = (int64_t)mt * nt;
  const int pairs_max = num_sms() / 2;
  const int pairs = (int)(tiles < pairs_max ? tiles : pairs_max);
  int group_m = 16;
  if (const char* e = getenv("BMF_GROUP_M2")) { int v = atoi(e); if (v >= 1 && v <= 64) group_m = v; }
  gemm_f4_2sm_kernel<EPI><<<2 * pairs, F4Threads<EPI>::value, SMEM_BYTES4, stream>>>(ma, mb, mt, nt, kb, group_m, ea);
  return check_cuda(cudaGetLastError(), "gemm_f4_2sm_kernel launch");
}

// -------------------------------------------------------------------------------------------------
// Super-tile variant (EPI_GAIN / EPI_STORE): a kind::mxf4 instruction costs ~150 cycles whatever N is, so wider is
// better, but two 256-column accumulators leave no TMEM for the scale factors.  Here a CTA pair walks SUPER tiles of
// 256 candidates x 496 data rows as two back-to-back sub-tiles: N = 256 into accumulator 0 (columns [0, 256)) and
// N = 240 into accumulator 1 (columns [256, 496)); scale factors sit in columns [496, 512).  Average N = 248
// instead of 240 (+3 %), the A tile is re-used by both sub-tiles out of L2, and the accumulator index equals the
// sub-tile index, so the double-buffering protocol is unchanged.
// -------------------------------------------------------------------------------------------------
constexpr int SUPER_ROWS = BMF_F4_SUPER_ROWS;   // 496
static inline bool super_tiles_disabled() {
  const char* e = getenv("BMF_F4_NO_SUPER");
  return e != nullptr && e[0] == '1';
}
constexpr int SUB0 = 256, SUB1 = SUPER_ROWS - SUB0;          // sub-tile widths
constexpr int STAGES_S = 6;
constexpr int STAGE_BYTES_S = A_OP + (SUB0 / 2) * BK;        // 32 KB (sub-tile 1 uses 31 KB of it)
constexpr int SMEM_BYTES_S = STAGES_S * STAGE_BYTES_S + 1024 + 256;
constexpr int SF_COL_S = SUPER_ROWS;                          // scale-factor columns [496, 512)
constexpr uint32_t idesc_f4(int n) {
  return (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | (1u << 23) | ((uint32_t)(BM4 >> 4) << 24);
}

template <int EPI, int NCOLS>
__device__ __forceinline__ void epilogue_cols_f4(uint32_t taddr, int64_t row, int64_t col0, const EpiArgs& ea) {
  const int bias = (EPI == EPI_GAIN && ea.cand_pop != nullptr) ? ea.bias_scale * ea.cand_pop[row] : 0;
  long long relu_sum = 0;
#pragma unroll 1
  for (int c = 0; c < NCOLS / 16; ++c) {
    uint32_t lo[8], hi[8];
    tmem_ld_32x32_x8(taddr + (uint32_t)(c * 16), lo);
    tmem_ld_32x32_x8(taddr + (uint32_t)(c * 16 + 8), hi);
    tmem_ld_wait();
    if (EPI == EPI_GAIN) {
      int part = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) part += max(f32_bits_to_int(lo[q]) - bias, 0) + max(f32_bits_to_int(hi[q]) - bias, 0);
      relu_sum += part;
    } else {
      int4* dst = reinterpret_cast<int4*>(ea.C + row * ea.ldc + col0 + c * 16);
      int4 o[4];
      o[0] = make_int4(f32_bits_to_int(lo[0]), f32_bits_to_int(lo[1]), f32_bits_to_int(lo[2]), f32_bits_to_int(lo[3]));
      o[1] = make_int4(f32_bits_to_int(lo[4]), f32_bits_to_int(lo[5]), f32_bits_to_int(lo[6]), f32_bits_to_int(lo[7]));
      o[2] = make_int4(f32_bits_to_int(hi[0]), f32_bits_to_int(hi[1]), f32_bits_to_int(hi[2]), f32_bits_to_int(hi[3]));
      o[3] = make_int4(f32_bits_to_int(hi[4]), f32_bits_to_int(hi[5]), f32_bits_to_int(hi[6]), f32_bits_to_int(hi[7]));
      if (ea.accumulate) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int4 p = dst[q];
          o[q].x += p.x; o[q].y += p.y; o[q].z += p.z; o[q].w += p.w;
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) dst[q] = o[q];
    }
  }
  if (EPI == EPI_GAIN && relu_sum != 0)
    atomicAdd(ea.gain + row, (unsigned long long)(ea.gain_sign < 0 ? -relu_sum : relu_sum));
}

// X^T X is symmetric: a super tile whose last data row lies before its first candidate row is entirely below the
// diagonal; bmf_basis_threshold(symmetric) reads cnt[min(i,j)][max(i,j)] instead.  All three warp roles evaluate the
// same predicate, so the pipeline protocol is untouched.
__device__ __forceinline__ bool skip_lower(const EpiArgs& ea, int mt, int st) {
  return ea.symmetric && ((int64_t)st * SUPER_ROWS + (SUPER_ROWS - 1) < (int64_t)mt * BM4);
}

// The super tiles of one CTA pair, in launch order.  Plain: t = pair, pair + P, ... through the grouped raster.  Symmetric
// (X^T X): the KEPT tiles are dealt round-robin.  Striding over all tiles and skipping the lower ones left the pairs with
// uneven shares (14..21 kept tiles around a mean of 17.6 at 17770 columns: the association ran at 0.77 of the pipe).
// The three warp roles build the same iterator, so they agree on the sequence without talking to each other; the walk is
// incremental (no division per visited tile).
struct SuperTileIter {
  bool sym;
  int64_t t, total, stride;
  int mt_total, nt_total, group_m, first, gsize, mi, nt, kept_mod, pair, num_pairs;
  __device__ __forceinline__ SuperTileIter(bool sym_, int64_t pair_, int64_t num_pairs_, int64_t total_, int mt_total_,
                                           int nt_total_, int group_m_)
      : sym(sym_), t(pair_), total(total_), stride(num_pairs_), mt_total(mt_total_), nt_total(nt_total_), group_m(group_m_),
        first(total_ > 0 ? 0 : mt_total_), gsize(min(group_m_, mt_total_)), mi(0), nt(0), kept_mod(0), pair((int)pair_),
        num_pairs((int)num_pairs_) {}
  __device__ __forceinline__ bool next(const EpiArgs& ea, int& mt, int& st) {
    if (!sym) {
      if (t >= total) return false;
      tile_coords(t, mt_total, nt_total, group_m, mt, st);
      t += stride;
      return true;
    }
    while (first < mt_total) {
      mt = first + mi;
      st = nt;
      if (++mi == gsize) {
        mi = 0;
        if (++nt == nt_total) { nt = 0; first += group_m; gsize = min(group_m, mt_total - first); }
      }
      if (skip_lower(ea, mt, st)) continue;
      const bool mine = kept_mod == pair;
      if (++kept_mod == num_pairs) kept_mod = 0;
      if (mine) return true;
    }
    return false;
  }
};

// Block-sparse walk (EPI_GAIN with a K-block table): the units are (super tile st, candidate tile mt) in st-major order, and
// unit (st, mt) costs cnt[mt] = cum[mt + 1] - cum[mt] K blocks (per sub-tile).  With the candidates and columns reordered
// most tiles hold few nonzero K blocks (2 to 36 of 70 at c4), so dealing tiles round-robin would leave pairs with several
// times the work of others: pair p instead takes the units whose cost prefix st * C + cum[mt] lies in
// [ceil(p T / P), ceil((p + 1) T / P)), T = st_total * C.  Super tiles outer keeps the nonzero candidate blocks (C x 32 KB)
// resident in L2 while every pair streams its own data rows from DRAM about once.  Units of cost 0 (all-zero candidate
// tiles: relu(0 - bias) = 0) are skipped.  All three warp roles build the same walk.
struct SparseWalk {
  const int32_t* cum;
  int mt_total, st_total, mt, st;
  int64_t C, end;
  __device__ __forceinline__ SparseWalk(const int32_t* cum_, int mt_total_, int st_total_, int64_t pair, int64_t num_pairs)
      : cum(cum_), mt_total(mt_total_), st_total(st_total_), mt(0), st(st_total_), C(cum_ != nullptr ? cum_[mt_total_] : 0),
        end(0) {
    const int64_t T = (int64_t)st_total * C;
    if (T == 0) return;
    const int64_t begin = (pair * T + num_pairs - 1) / num_pairs;
    end = ((pair + 1) * T + num_pairs - 1) / num_pairs;
    st = (int)(begin / C);
    const int64_t r = begin - (int64_t)st * C;
    int lo = 0, hi = mt_total;                            // first mt with cum[mt] >= r (mt_total: none in this super tile)
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (cum[mid] < r) lo = mid + 1; else hi = mid;
    }
    mt = lo;
    if (mt == mt_total) { mt = 0; ++st; }
  }
  __device__ __forceinline__ bool next(int& mt_out, int& st_out, int& nkb) {
    while (st < st_total) {
      const int c0 = cum[mt], c1 = cum[mt + 1];
      if ((int64_t)st * C + c0 >= end) return false;
      mt_out = mt;
      st_out = st;
      if (++mt == mt_total) { mt = 0; ++st; }
      if (c1 > c0) { nkb = c1 - c0; return true; }
    }
    return false;
  }
};

// The units of one CTA pair for all three warp roles: the dense raster (SuperTileIter, every K block) or, with a K-block
// table, the block-sparse walk.  nkb = K blocks of the unit; the producer reads their indices from the list (kb_list).
struct UnitWalk {
  SuperTileIter dense;
  SparseWalk sparse;
  bool is_sparse;
  int kb_total;
  __device__ __forceinline__ UnitWalk(const EpiArgs& ea, bool sym, int64_t pair, int64_t num_pairs, int mt_total,
                                      int st_total, int kb_total_, int group_m)
      : dense(sym, pair, num_pairs, (int64_t)mt_total * st_total, mt_total, st_total, group_m),
        sparse(ea.kb_table, mt_total, st_total, pair, num_pairs),
        is_sparse(ea.kb_table != nullptr), kb_total(kb_total_) {}
  __device__ __forceinline__ bool next(const EpiArgs& ea, int& mt, int& st, int& nkb) {
    if (is_sparse) return sparse.next(mt, st, nkb);
    nkb = kb_total;
    return dense.next(ea, mt, st);
  }
};

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_f4s_2sm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b0,
                    const __grid_constant__ CUtensorMap tmap_b1, int mt_total, int st_total_in, int kb_total, int group_m,
                    const EpiArgs ea) {
  extern __shared__ uint8_t smem_raw[];
  const int st_total = dyn_row_tiles(ea, st_total_in, SUPER_ROWS);
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES_S * STAGE_BYTES_S);
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES_S + 4);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES_S + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES_S + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES_S + 2 + a); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int64_t pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES_S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b0)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b1)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_base_slot);
  if (warp >= 2) {                                        // unit scale factors: all 128 lanes x columns [496, 512)
    const uint32_t sf_addr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)SF_COL_S;
    tmem_st_32x32_x8(sf_addr, SF_ONE);
    tmem_st_32x32_x8(sf_addr + 8u, SF_ONE);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();

  if (warp == 0) {
    {                                                     // whole warp, converged; one elected lane issues the TMA
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t sb = warp_uniform(smem_base);
      UnitWalk units(ea, EPI == EPI_STORE && ea.symmetric, pair, num_pairs, mt_total, st_total, kb_total, group_m);
      const int32_t* kb_lists = ea.kb_table != nullptr ? ea.kb_table + mt_total + 1 : nullptr;
      int mt, st, nkb;
      while (units.next(ea, mt, st, nkb)) {
#pragma unroll 1
        for (int sub = 0; sub < 2; ++sub) {
          const int half = sub ? SUB1 / 2 : SUB0 / 2;                       // data rows this CTA stages
          const int row0 = st * SUPER_ROWS + (sub ? SUB0 : 0) + (int)rank * half;
          const CUtensorMap* mb = sub ? &tmap_b1 : &tmap_b0;
          const uint32_t tx = 2u * (uint32_t)(A_OP + half * BK);
          for (int i0 = 0; i0 < nkb; i0 += 32) {                          // the list, 32 entries per coalesced load
            const int kv = (kb_lists != nullptr && i0 + lane < nkb) ? kb_lists[(int64_t)mt * kb_total + i0 + lane] : 0;
            const int nb = min(32, nkb - i0);
            for (int j = 0; j < nb; ++j) {
              const int kb = kb_lists != nullptr ? __shfl_sync(0xffffffffu, kv, j) : i0 + j;
              mbar_wait(empty_bar(stage), phase ^ 1u);
              const uint32_t leader_full = full_bar(stage) & PEER_MASK;
              const uint32_t a_dst = sb + stage * STAGE_BYTES_S;
              if (elect_one()) {
                if (leader) mbar_expect_tx(full_bar(stage), tx);
                tma_load_2d_2sm(a_dst, &tmap_a, leader_full, kb * BK, mt * BM4 + (int)rank * HALFM, ea.policy_a);
                tma_load_2d_2sm(a_dst + A_OP, mb, leader_full, kb * BK, row0, ea.policy_b);
              }
              __syncwarp();
              if (++stage == STAGES_S) { stage = 0; phase ^= 1u; }
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (leader) {                                         // whole warp, converged (see elect_one)
      int stage = 0;
      uint32_t phase = 0, acc_phase = 0;
      const uint32_t tb = warp_uniform(tmem_base), sb = warp_uniform(smem_base);
      const uint32_t sfa = tb + (uint32_t)SF_COL_S, sfb = tb + (uint32_t)SF_COL_S + 8u;
      UnitWalk units(ea, EPI == EPI_STORE && ea.symmetric, pair, num_pairs, mt_total, st_total, kb_total, group_m);
      int mt, st, nkb;
      while (units.next(ea, mt, st, nkb)) {
#pragma unroll 1
        for (int sub = 0; sub < 2; ++sub) {
          mbar_wait(tempty_bar(sub), acc_phase ^ 1u);
          tcgen05_fence_after();
          const uint32_t d_tmem = tb + (uint32_t)(sub ? SUB0 : 0);
          const uint32_t idesc = sub ? idesc_f4(SUB1) : idesc_f4(SUB0);
          for (int kb = 0; kb < nkb; ++kb) {                              // kb counts the unit's blocks (0 = first)
            mbar_wait(full_bar(stage), phase);
            tcgen05_fence_after();
            const uint32_t a_addr = sb + stage * STAGE_BYTES_S;
            const uint64_t da = make_smem_desc(a_addr), db = make_smem_desc(a_addr + A_OP);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                tcgen05_mma_f4_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                   (uint32_t)((kb | k) != 0), sfa, sfb);
              tcgen05_commit_2sm(empty_bar(stage));
            }
            __syncwarp();
            if (++stage == STAGES_S) { stage = 0; phase ^= 1u; }
          }
          if (elect_one()) tcgen05_commit_2sm(tfull_bar(sub));
          __syncwarp();
        }
        acc_phase ^= 1u;
      }
    }
    __syncwarp();
  } else {
    const int quad = warp & 3;
    uint32_t acc_phase = 0;
    UnitWalk units(ea, EPI == EPI_STORE && ea.symmetric, pair, num_pairs, mt_total, st_total, kb_total, group_m);
    int mt, st, nkb;
    while (units.next(ea, mt, st, nkb)) {
      const int64_t plane_row = (int64_t)mt * BM4 + (int64_t)rank * HALFM + quad * 32 + lane;
      const int64_t row = (EPI == EPI_GAIN && ea.cand_id != nullptr) ? (int64_t)ea.cand_id[plane_row] : plane_row;
      const uint32_t lane_base = tmem_base + ((uint32_t)(quad * 32) << 16);
      mbar_wait(tfull_bar(0), acc_phase);
      tcgen05_fence_after();
      epilogue_cols_f4<EPI, SUB0>(lane_base, row, (int64_t)st * SUPER_ROWS, ea);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tempty_bar(0));
      mbar_wait(tfull_bar(1), acc_phase);
      tcgen05_fence_after();
      epilogue_cols_f4<EPI, SUB1>(lane_base + (uint32_t)SUB0, row, (int64_t)st * SUPER_ROWS + SUB0, ea);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tempty_bar(1));
      acc_phase ^= 1u;
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

template <int EPI>
static int launch_gemm_f4s(const uint8_t* a, int64_t a_rows, const uint8_t* b, int64_t b_rows, int64_t ld_bytes,
                           const EpiArgs& ea_in, cudaStream_t stream) {
  CUtensorMap ma, mb0, mb1;
  int rc = make_plane_map(&ma, reinterpret_cast<const int8_t*>(a), a_rows, ld_bytes, HALFM);
  if (rc) return rc;
  rc = make_plane_map(&mb0, reinterpret_cast<const int8_t*>(b), b_rows, ld_bytes, SUB0 / 2);
  if (rc) return rc;
  rc = make_plane_map(&mb1, reinterpret_cast<const int8_t*>(b), b_rows, ld_bytes, SUB1 / 2);
  if (rc) return rc;
  static bool attr_set[2] = {false, false};
  if (!attr_set[EPI]) {
    rc = check_cuda(cudaFuncSetAttribute(gemm_f4s_2sm_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES_S),
                    "cudaFuncSetAttribute(gemm_f4s_2sm_kernel)");
    if (rc) return rc;
    attr_set[EPI] = true;
  }
  EpiArgs ea = ea_in;
  ea.policy_a = L2_EVICT_NORMAL;
  ea.policy_b = L2_EVICT_NORMAL;
  const int mt = (int)(a_rows / BM4), st = (int)(b_rows / SUPER_ROWS), kb = (int)(ld_bytes / BK);
  const int64_t tiles = (int64_t)mt * st;
  const int pairs_max = num_sms() / 2;
  const int pairs = (int)(tiles < pairs_max ? tiles : pairs_max);
  // Raster: candidate tiles cycle fastest inside a group of group_m, data-row tiles advance per group pass.  Measured at c4
  // (profiles/r02_group_sweep.log, profiles/r02g_shard_kernel_probe.log): groups of 8 / 16 / 24 candidate tiles (18-55 MB
  // candidate panels) all run at the pipe's issue rate (34.6 ms; 28 GB of DRAM reads per launch at 16); a group of 35 (an
  // 80 MB panel) falls off the L2 cliff -- 134 GB, hit rate 66 %, sw_power_cap -- because the 126 MB L2 is two 63 MB halves;
  // one group over ALL 70 candidate tiles (160 MB panel) is 30 % slower (43 ms).  Keep 16.
  int group_m = 16;
  if (const char* e = getenv("BMF_GROUP_M2")) { int v = atoi(e); if (v >= 1 && v <= 1024) group_m = v; }
  gemm_f4s_2sm_kernel<EPI><<<2 * pairs, NUM_THREADS, SMEM_BYTES_S, stream>>>(ma, mb0, mb1, mt, st, kb, group_m, ea);
  return check_cuda(cudaGetLastError(), "gemm_f4s_2sm_kernel launch");
}
}  // namespace f4

// =================================================================================================
// Tensor-pipe ceiling probe (bench.py's roofline denominator, measured live on the box): a CTA pair per TPC issues
// `iters` x 4 back-to-back tcgen05.mma instructions of the production shape -- kind::mxf4 M = 256, N = 256, K = 64
// with unit scales, or kind::i8 M = 256, N = 256, K = 32 -- on operands that already sit in shared memory (sparse
// small integers like the workload's; no TMA, no epilogue, one commit at the end).  What it measures is the issue rate
// of the pipe itself at the clocks this kind of data sustains; the scoring kernels cannot be faster than this.
// =================================================================================================
namespace probe {
using sm2::cluster_ctarank;
using sm2::cluster_sync_all;
using sm2::tcgen05_commit_2sm;
using sm2::tcgen05_mma_i8_2sm;
using f4::tcgen05_mma_f4_2sm;
using f4::tmem_st_32x32_x8;
constexpr int PROBE_THREADS = 128;
constexpr int PROBE_SMEM = 2 * 16384 + 1024 + 64;

template <int KIND>   // 0 = kind::i8, 1 = kind::mxf4
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PROBE_THREADS, 1)
mma_rate_probe_kernel(int iters, uint32_t seed) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * 16384);
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const int warp = threadIdx.x >> 5;
  const bool leader = cluster_ctarank() == 0;
  // operands: A = 128 rows x 128 B, B = 128 rows x 128 B per CTA; ~1/32 of the elements are a small integer
  for (int i = threadIdx.x; i < 2 * 16384 / 4; i += PROBE_THREADS) {
    uint32_t h = (uint32_t)i * 2654435761u + seed + blockIdx.x * 40503u;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
    uint32_t w = 0;
    if ((h & 7u) == 0u) w = (KIND == 1 ? 0x2u : 0x1u) << (((h >> 3) & 7u) * 4u) % 32u;
    reinterpret_cast<uint32_t*>(smem)[i] = w;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(bars), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_base_slot);
  if (KIND == 1) {                                        // unit UE8M0 scale factors in columns [496, 512)
    const uint32_t sf_addr = tmem_base + ((uint32_t)(warp * 32) << 16) + 496u;
    tmem_st_32x32_x8(sf_addr, f4::SF_ONE);
    tmem_st_32x32_x8(sf_addr + 8u, f4::SF_ONE);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  if (warp == 0 && leader) {
    const uint32_t tb = warp_uniform(tmem_base), sb = warp_uniform(smem_u32(smem));
    const uint64_t da = make_smem_desc(sb), db = make_smem_desc(sb + 16384u);
    const uint32_t sfa = tb + 496u, sfb = tb + 504u;
    constexpr uint32_t idesc_f4 = f4::idesc_f4(256);
    for (int it = 0; it < iters; ++it) {
      const uint32_t d_tmem = tb + (uint32_t)((it & 1) ? 240 : 0);     // two accumulators, like the production kernels
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (KIND == 1)
            tcgen05_mma_f4_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc_f4, (uint32_t)(it > 1 || k),
                               sfa, sfb);
          else
            tcgen05_mma_i8_2sm(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), sm2::IDESC_I8_2SM,
                               (uint32_t)(it > 1 || k));
        }
      }
      __syncwarp();
    }
    if (elect_one()) tcgen05_commit_2sm(smem_u32(bars));
    __syncwarp();
  }
  mbar_wait(smem_u32(bars), 0);                          // the multicast commit arrives in both CTAs
  tcgen05_fence_after();
  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 0) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}
}  // namespace probe

// variant: 0 = auto (2-SM when the candidate rows are a multiple of 256), 1 = 1-SM, 2 = 2-SM
template <int EPI>
static int dispatch_gemm(int variant, const int8_t* a, int64_t a_rows, const int8_t* b, int64_t b_rows, int64_t ld,
                         const EpiArgs& ea_in, cudaStream_t stream) {
  if (const char* e = getenv("BMF_GEMM_VARIANT")) { int v = atoi(e); if (v == 1 || v == 2) variant = v; }
  EpiArgs ea = ea_in;
  // measured at c4 (profiles/r01b_l2_hint_sweep.md): the data-row tiles ARE re-read inside a wave (16 pairs share one), so
  // evict_first on them raises DRAM traffic 295 -> 450 GB per launch; evict_last on the candidate panel changes nothing
  // measurable.  Default: no hint.  0 none, 1 A evict_last + B evict_first, 2 B only, 3 A only
  int hint = 0;
  if (const char* e = getenv("BMF_L2_HINT")) { int v = atoi(e); if (v >= 0 && v <= 3) hint = v; }
  ea.policy_a = (hint == 1 || hint == 3) ? L2_EVICT_LAST : L2_EVICT_NORMAL;
  ea.policy_b = (hint == 1 || hint == 2) ? L2_EVICT_FIRST : L2_EVICT_NORMAL;
  const bool ok2 = (a_rows % sm2::BM2) == 0;
  if (variant == 2 && !ok2) {
    set_error("2-SM int8 kernel needs the candidate rows padded to a multiple of 256 (got %lld)", (long long)a_rows);
    return BMF_E_ARG;
  }
  if (variant == 2 || (variant == 0 && ok2))
    return sm2::launch_gemm_2sm<EPI>(a, a_rows, b, b_rows, ld, ea, stream);
  return launch_gemm<EPI>(a, a_rows, b, b_rows, ld, ea, stream);
}

}  // namespace tc
}  // namespace bmf

using namespace bmf;

extern "C" int bmf_gemm_i8_nt(const int8_t* a_plane, int64_t a_rows_pad, const int8_t* b_plane, int64_t b_rows_pad,
                              int64_t ld, int32_t* c, int64_t ldc, bmf_stream_t stream) {
  BMF_REQUIRE(a_plane && b_plane && c, "bmf_gemm_i8_nt: null pointer");
  BMF_REQUIRE(a_rows_pad > 0 && a_rows_pad % tc::BM == 0, "bmf_gemm_i8_nt: a rows must be a positive multiple of 128");
  BMF_REQUIRE(b_rows_pad > 0 && b_rows_pad % tc::BN == 0, "bmf_gemm_i8_nt: b rows must be a positive multiple of 256");
  BMF_REQUIRE(ld > 0 && ld % tc::BK == 0, "bmf_gemm_i8_nt: ld must be a positive multiple of 128");
  BMF_REQUIRE(ldc >= b_rows_pad && ldc % 4 == 0, "bmf_gemm_i8_nt: ldc must cover b rows and be a multiple of 4");
  tc::EpiArgs ea = {};
  ea.C = c;
  ea.ldc = ldc;
  return tc::dispatch_gemm<tc::EPI_STORE>(0, a_plane, a_rows_pad, b_plane, b_rows_pad, ld, ea, as_stream(stream));
}

extern "C" int bmf_assoc_counts_i8(const int8_t* xt_plane, int64_t n, int64_t n_pad, int64_t ld, int32_t* cnt,
                                   int64_t ldc, bmf_stream_t stream) {
  BMF_REQUIRE(xt_plane && cnt && n > 0, "bmf_assoc_counts_i8: null pointer or empty matrix");
  BMF_REQUIRE(n_pad >= n && n_pad % tc::BN == 0, "bmf_assoc_counts_i8: n_pad must be a multiple of 256 covering n");
  BMF_REQUIRE(ld > 0 && ld % tc::BK == 0, "bmf_assoc_counts_i8: ld must be a positive multiple of 128");
  BMF_REQUIRE(ldc >= n_pad && ldc % 4 == 0, "bmf_assoc_counts_i8: ldc must be >= n_pad and a multiple of 4");
  tc::EpiArgs ea = {};
  ea.C = cnt;
  ea.ldc = ldc;
  return tc::dispatch_gemm<tc::EPI_STORE>(0, xt_plane, n_pad, xt_plane, n_pad, ld, ea, as_stream(stream));
}

extern "C" int bmf_cover_score_i8(const int8_t* cand_plane, int64_t cand_pad, const int8_t* rows_plane,
                                  int64_t rows_pad, int64_t ld, int32_t sign, const int32_t* cand_pop, int32_t bias_scale,
                                  int64_t* gain, bmf_stream_t stream) {
  BMF_REQUIRE(sign == 1 || sign == -1, "bmf_cover_score_i8: sign must be +1 or -1");
  BMF_REQUIRE(cand_plane && rows_plane && gain, "bmf_cover_score_i8: null pointer");
  BMF_REQUIRE(cand_pad > 0 && cand_pad % tc::BM == 0, "bmf_cover_score_i8: cand_pad must be a positive multiple of 128");
  BMF_REQUIRE(rows_pad > 0 && rows_pad % tc::BN == 0, "bmf_cover_score_i8: rows_pad must be a positive multiple of 256");
  BMF_REQUIRE(ld > 0 && ld % tc::BK == 0, "bmf_cover_score_i8: ld must be a positive multiple of 128");
  BMF_REQUIRE(ld <= 524288, "bmf_cover_score_i8: more than 524288 columns would overflow the epilogue's int32 partial sums "
                            "(32 elements x 127 x ld)");
  int rc = check_cuda(cudaMemsetAsync(gain, 0, sizeof(int64_t) * cand_pad, as_stream(stream)), "bmf_cover_score_i8");
  if (rc) return rc;
  tc::EpiArgs ea = {};
  ea.sign = sign;
  ea.cand_pop = cand_pop;
  ea.bias_scale = bias_scale;
  ea.gain_sign = 1;
  ea.gain = reinterpret_cast<unsigned long long*>(gain);
  return tc::dispatch_gemm<tc::EPI_GAIN>(0, cand_plane, cand_pad, rows_plane, rows_pad, ld, ea, as_stream(stream));
}

extern "C" int bmf_cover_rescore_i8(const int8_t* cand_plane, int64_t cand_pad, const int8_t* compact_plane,
                                    int64_t rows_cap, int64_t ld, int32_t sign, const int32_t* cand_pop,
                                    int32_t bias_scale, const int32_t* dyn_rows, int32_t gain_sign, int64_t* gain,
                                    bmf_stream_t stream) {
  BMF_REQUIRE(sign == 1 || sign == -1, "bmf_cover_rescore_i8: sign must be +1 or -1");
  BMF_REQUIRE(gain_sign == 1 || gain_sign == -1, "bmf_cover_rescore_i8: gain_sign must be +1 or -1");
  BMF_REQUIRE(cand_plane && compact_plane && gain && dyn_rows, "bmf_cover_rescore_i8: null pointer");
  BMF_REQUIRE(cand_pad > 0 && cand_pad % tc::BM == 0, "bmf_cover_rescore_i8: cand_pad must be a positive multiple of 128");
  BMF_REQUIRE(rows_cap > 0 && rows_cap % tc::BN == 0, "bmf_cover_rescore_i8: rows_cap must be a positive multiple of 256");
  BMF_REQUIRE(ld > 0 && ld % tc::BK == 0 && ld <= 524288, "bmf_cover_rescore_i8: ld must be a multiple of 128, at most 524288");
  tc::EpiArgs ea = {};
  ea.sign = sign;
  ea.cand_pop = cand_pop;
  ea.bias_scale = bias_scale;
  ea.gain_sign = gain_sign;
  ea.dyn_rows = dyn_rows;
  ea.gain = reinterpret_cast<unsigned long long*>(gain);
  return tc::dispatch_gemm<tc::EPI_GAIN>(0, cand_plane, cand_pad, compact_plane, rows_cap, ld, ea, as_stream(stream));
}

static int cover_score_i8_general_impl(const int8_t* cand_plane, int64_t cand_pad, const int8_t* pq_plane, int64_t m,
                                       int64_t ld, const int32_t* cand_pop, const int32_t* tp_old, const int32_t* fp_old,
                                       double w_fp, double w_fn, int64_t* gain_p, int64_t* gain_n, const int32_t* dyn_rows,
                                       int gain_sign, bmf_stream_t stream) {
  BMF_REQUIRE(cand_plane && pq_plane && cand_pop && tp_old && fp_old && gain_p && gain_n,
              "bmf_cover_score_i8_general: null pointer");
  BMF_REQUIRE(cand_pad > 0 && cand_pad % tc::BM == 0, "bmf_cover_score_i8_general: cand_pad must be a positive multiple of 128");
  BMF_REQUIRE(m > 0, "bmf_cover_score_i8_general: no data rows");
  BMF_REQUIRE(ld > 0 && ld % tc::BK == 0, "bmf_cover_score_i8_general: ld must be a positive multiple of 128");
  const int64_t plane_rows = 2 * ceil_div(m, 128) * 128;   // [ceil(m/128)][P|Q][128] rows of ld bytes
  if (dyn_rows == nullptr) {                               // a full pass overwrites; a re-score accumulates
    int rc = check_cuda(cudaMemsetAsync(gain_p, 0, sizeof(int64_t) * cand_pad, as_stream(stream)), "bmf_cover_score_i8_general");
    if (rc) return rc;
    rc = check_cuda(cudaMemsetAsync(gain_n, 0, sizeof(int64_t) * cand_pad, as_stream(stream)), "bmf_cover_score_i8_general");
    if (rc) return rc;
  }
  tc::EpiArgs ea = {};
  ea.cand_pop = cand_pop;
  ea.gain = reinterpret_cast<unsigned long long*>(gain_p);
  ea.gain_n = reinterpret_cast<unsigned long long*>(gain_n);
  ea.tp_old = tp_old;
  ea.fp_old = fp_old;
  ea.m_rows = m;
  ea.neg_w_fp = -w_fp;
  ea.w_fn = w_fn;
  ea.dyn_rows = dyn_rows;
  ea.gain_sign = gain_sign;
  return tc::dispatch_gemm<tc::EPI_GAIN2>(0, cand_plane, cand_pad, pq_plane, plane_rows, ld, ea, as_stream(stream));
}

extern "C" int bmf_cover_score_i8_general(const int8_t* cand_plane, int64_t cand_pad, const int8_t* pq_plane,
                                          int64_t m, int64_t ld, const int32_t* cand_pop, const int32_t* tp_old,
                                          const int32_t* fp_old, double w_fp, double w_fn, int64_t* gain_p,
                                          int64_t* gain_n, bmf_stream_t stream) {
  return cover_score_i8_general_impl(cand_plane, cand_pad, pq_plane, m, ld, cand_pop, tp_old, fp_old, w_fp, w_fn, gain_p,
                                     gain_n, nullptr, 1, stream);
}

extern "C" int bmf_cover_rescore_i8_general(const int8_t* cand_plane, int64_t cand_pad, const int8_t* compact_pq_plane,
                                            int64_t rows_cap, int64_t ld, const int32_t* cand_pop, const int32_t* comp_tp,
                                            const int32_t* comp_fp, double w_fp, double w_fn, const int32_t* dyn_rows,
                                            int32_t gain_sign, int64_t* gain_p, int64_t* gain_n, bmf_stream_t stream) {
  BMF_REQUIRE(dyn_rows != nullptr && (gain_sign == 1 || gain_sign == -1), "bmf_cover_rescore_i8_general: dyn_rows / gain_sign");
  return cover_score_i8_general_impl(cand_plane, cand_pad, compact_pq_plane, rows_cap, ld, cand_pop, comp_tp, comp_fp, w_fp,
                                     w_fn, gain_p, gain_n, dyn_rows, gain_sign, stream);
}

// ---- FP4 (kind::mxf4) entry points -------------------------------------------------------------------
extern "C" int bmf_gemm_f4_nt(const uint8_t* a_plane, int64_t a_rows_pad, const uint8_t* b_plane, int64_t b_rows_pad,
                              int64_t ld_bytes, int32_t* c, int64_t ldc, int32_t accumulate, bmf_stream_t stream) {
  BMF_REQUIRE(a_plane && b_plane && c, "bmf_gemm_f4_nt: null pointer");
  BMF_REQUIRE(a_rows_pad > 0 && a_rows_pad % tc::f4::BM4 == 0, "bmf_gemm_f4_nt: a rows must be a positive multiple of 256");
  BMF_REQUIRE(b_rows_pad > 0 && (b_rows_pad % tc::f4::BN4 == 0 || b_rows_pad % tc::f4::SUPER_ROWS == 0),
              "bmf_gemm_f4_nt: b rows must be a positive multiple of 240 or of 496");
  BMF_REQUIRE(ld_bytes > 0 && ld_bytes % tc::BK == 0, "bmf_gemm_f4_nt: ld_bytes must be a positive multiple of 128");
  BMF_REQUIRE(ldc >= b_rows_pad && ldc % 4 == 0, "bmf_gemm_f4_nt: ldc must cover b rows and be a multiple of 4");
  tc::EpiArgs ea = {};
  ea.C = c;
  ea.ldc = ldc;
  ea.accumulate = (accumulate & 1) ? 1 : 0;
  ea.symmetric = (accumulate & 2) ? 1 : 0;      // bit 1: a_plane == b_plane (X^T X), tiles below the diagonal are skipped
  BMF_REQUIRE(!accumulate || (b_rows_pad % tc::f4::SUPER_ROWS == 0 && !tc::f4::super_tiles_disabled()),
              "bmf_gemm_f4_nt: accumulate / symmetric need b rows padded to 496 (super-tile kernel)");
  BMF_REQUIRE(!ea.symmetric || a_plane == b_plane, "bmf_gemm_f4_nt: symmetric needs a_plane == b_plane");
  if (b_rows_pad % tc::f4::SUPER_ROWS == 0 && !tc::f4::super_tiles_disabled())
    return tc::f4::launch_gemm_f4s<tc::EPI_STORE>(a_plane, a_rows_pad, b_plane, b_rows_pad, ld_bytes, ea, as_stream(stream));
  BMF_REQUIRE(b_rows_pad % tc::f4::BN4 == 0, "bmf_gemm_f4_nt: b rows must be a multiple of 240 for the plain-tile kernel");
  return tc::f4::launch_gemm_f4<tc::EPI_STORE>(a_plane, a_rows_pad, b_plane, b_rows_pad, ld_bytes, ea, as_stream(stream));
}

extern "C" int bmf_cover_score_f4_blocks(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* rows_plane,
                                         int64_t rows_pad, int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale,
                                         const int32_t* kb_table, const int32_t* cand_id, int64_t* gain, bmf_stream_t stream) {
  BMF_REQUIRE(cand_plane && rows_plane && gain, "bmf_cover_score_f4: null pointer");
  BMF_REQUIRE(cand_pad > 0 && cand_pad % tc::f4::BM4 == 0, "bmf_cover_score_f4: cand_pad must be a positive multiple of 256");
  BMF_REQUIRE(rows_pad > 0 && (rows_pad % tc::f4::BN4 == 0 || rows_pad % tc::f4::SUPER_ROWS == 0),
              "bmf_cover_score_f4: rows_pad must be a positive multiple of 240 or of 496");
  BMF_REQUIRE(ld_bytes > 0 && ld_bytes % tc::BK == 0, "bmf_cover_score_f4: ld_bytes must be a positive multiple of 128");
  BMF_REQUIRE(cand_pop != nullptr || bias_scale == 0, "bmf_cover_score_f4: a bias needs cand_pop");
  const bool super = rows_pad % tc::f4::SUPER_ROWS == 0 && !tc::f4::super_tiles_disabled();
  BMF_REQUIRE(super || (kb_table == nullptr && cand_id == nullptr),
              "bmf_cover_score_f4_blocks: a K-block table / candidate map needs rows_pad padded to 496 (super-tile kernel)");
  int rc = check_cuda(cudaMemsetAsync(gain, 0, sizeof(int64_t) * cand_pad, as_stream(stream)), "bmf_cover_score_f4");
  if (rc) return rc;
  tc::EpiArgs ea = {};
  ea.sign = 1;
  ea.cand_pop = cand_pop;
  ea.bias_scale = bias_scale;
  ea.gain_sign = 1;
  ea.gain = reinterpret_cast<unsigned long long*>(gain);
  ea.kb_table = kb_table;
  ea.cand_id = cand_id;
  if (super)
    return tc::f4::launch_gemm_f4s<tc::EPI_GAIN>(cand_plane, cand_pad, rows_plane, rows_pad, ld_bytes, ea, as_stream(stream));
  BMF_REQUIRE(rows_pad % tc::f4::BN4 == 0, "bmf_cover_score_f4: rows_pad must be a multiple of 240 for the plain-tile kernel");
  return tc::f4::launch_gemm_f4<tc::EPI_GAIN>(cand_plane, cand_pad, rows_plane, rows_pad, ld_bytes, ea, as_stream(stream));
}

extern "C" int bmf_cover_score_f4(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* rows_plane,
                                  int64_t rows_pad, int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale,
                                  int64_t* gain, bmf_stream_t stream) {
  return bmf_cover_score_f4_blocks(cand_plane, cand_pad, rows_plane, rows_pad, ld_bytes, cand_pop, bias_scale, nullptr,
                                   nullptr, gain, stream);
}

extern "C" int bmf_cover_rescore_f4_blocks(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* compact_plane,
                                           int64_t rows_cap, int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale,
                                           const int32_t* kb_table, const int32_t* cand_id, const int32_t* dyn_rows,
                                           int32_t gain_sign, int64_t* gain, bmf_stream_t stream) {
  BMF_REQUIRE(cand_plane && compact_plane && gain && dyn_rows, "bmf_cover_rescore_f4: null pointer");
  BMF_REQUIRE(gain_sign == 1 || gain_sign == -1, "bmf_cover_rescore_f4: gain_sign must be +1 or -1");
  BMF_REQUIRE(cand_pad > 0 && cand_pad % tc::f4::BM4 == 0, "bmf_cover_rescore_f4: cand_pad must be a positive multiple of 256");
  BMF_REQUIRE(rows_cap > 0 && rows_cap % tc::f4::SUPER_ROWS == 0, "bmf_cover_rescore_f4: rows_cap must be a positive multiple of 496");
  BMF_REQUIRE(ld_bytes > 0 && ld_bytes % tc::BK == 0, "bmf_cover_rescore_f4: ld_bytes must be a positive multiple of 128");
  BMF_REQUIRE(cand_pop != nullptr || bias_scale == 0, "bmf_cover_rescore_f4: a bias needs cand_pop");
  tc::EpiArgs ea = {};
  ea.sign = 1;
  ea.cand_pop = cand_pop;
  ea.bias_scale = bias_scale;
  ea.gain_sign = gain_sign;
  ea.dyn_rows = dyn_rows;
  ea.gain = reinterpret_cast<unsigned long long*>(gain);
  ea.kb_table = kb_table;
  ea.cand_id = cand_id;
  return tc::f4::launch_gemm_f4s<tc::EPI_GAIN>(cand_plane, cand_pad, compact_plane, rows_cap, ld_bytes, ea, as_stream(stream));
}

extern "C" int bmf_cover_rescore_f4(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* compact_plane,
                                    int64_t rows_cap, int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale,
                                    const int32_t* dyn_rows, int32_t gain_sign, int64_t* gain, bmf_stream_t stream) {
  return bmf_cover_rescore_f4_blocks(cand_plane, cand_pad, compact_plane, rows_cap, ld_bytes, cand_pop, bias_scale, nullptr,
                                     nullptr, dyn_rows, gain_sign, gain, stream);
}

static int cover_score_f4_general_impl(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* pq_plane, int64_t m,
                                       int64_t ld_bytes, const int32_t* cand_pop, const int32_t* tp_old,
                                       const int32_t* fp_old, double w_fp, double w_fn, int64_t* gain_p, int64_t* gain_n,
                                       const int32_t* dyn_rows, int gain_sign, bmf_stream_t stream) {
  BMF_REQUIRE(cand_plane && pq_plane && cand_pop && tp_old && fp_old && gain_p && gain_n,
              "bmf_cover_score_f4_general: null pointer");
  BMF_REQUIRE(cand_pad > 0 && cand_pad % tc::f4::BM4 == 0, "bmf_cover_score_f4_general: cand_pad must be a positive multiple of 256");
  BMF_REQUIRE(m > 0, "bmf_cover_score_f4_general: no data rows");
  BMF_REQUIRE(ld_bytes > 0 && ld_bytes % tc::BK == 0, "bmf_cover_score_f4_general: ld_bytes must be a positive multiple of 128");
  const int64_t plane_rows = 2 * ceil_div(m, tc::f4::HALFN) * tc::f4::HALFN;   // [ceil(m/120)][P|Q][120] rows
  if (dyn_rows == nullptr) {                               // a full pass overwrites; a re-score accumulates
    int rc = check_cuda(cudaMemsetAsync(gain_p, 0, sizeof(int64_t) * cand_pad, as_stream(stream)), "bmf_cover_score_f4_general");
    if (rc) return rc;
    rc = check_cuda(cudaMemsetAsync(gain_n, 0, sizeof(int64_t) * cand_pad, as_stream(stream)), "bmf_cover_score_f4_general");
    if (rc) return rc;
  }
  tc::EpiArgs ea = {};
  ea.cand_pop = cand_pop;
  ea.gain = reinterpret_cast<unsigned long long*>(gain_p);
  ea.gain_n = reinterpret_cast<unsigned long long*>(gain_n);
  ea.tp_old = tp_old;
  ea.fp_old = fp_old;
  ea.m_rows = m;
  ea.neg_w_fp = -w_fp;
  ea.w_fn = w_fn;
  ea.dyn_rows = dyn_rows;
  ea.gain_sign = gain_sign;
  // The fixed-point pre-decision may only settle an element when the literal fp64 comparison cannot disagree with it.  The
  // fp64 evaluation of s_new and s_old carries ~4 roundings of terms up to |w| * count (count <= number of columns), i.e.
  // an error below 2^-51 |w| n, which is 2^-31 |w| n in units of d = 2^20 (w_fn P - w_fp N).  The margin P + N + 2 leaves a
  // slack of (P + N) / 2 + 2 >= 2 such units beyond the weight rounding, so the gate is |w| n < 2^30 (error < 0.5 units).
  const double wmax = fmax(fabs(w_fp), fabs(w_fn));
  const bool fix_ok = (w_fp == w_fp) && (w_fn == w_fn) && wmax < 1024.0 && wmax * (double)(ld_bytes * 2) < 1073741824.0;
  const char* no_fix = getenv("BMF_NO_FIXED_PREDECISION");
  ea.fix_ok = (fix_ok && !(no_fix && no_fix[0] == '1')) ? 1 : 0;
  ea.w_fp_fix = fix_ok ? llrint(w_fp * 1048576.0) : 0;
  ea.w_fn_fix = fix_ok ? llrint(w_fn * 1048576.0) : 0;
  return tc::f4::launch_gemm_f4<tc::EPI_GAIN2>(cand_plane, cand_pad, pq_plane, plane_rows, ld_bytes, ea, as_stream(stream));
}

extern "C" int bmf_cover_score_f4_general(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* pq_plane, int64_t m,
                                          int64_t ld_bytes, const int32_t* cand_pop, const int32_t* tp_old,
                                          const int32_t* fp_old, double w_fp, double w_fn, int64_t* gain_p,
                                          int64_t* gain_n, bmf_stream_t stream) {
  return cover_score_f4_general_impl(cand_plane, cand_pad, pq_plane, m, ld_bytes, cand_pop, tp_old, fp_old, w_fp, w_fn,
                                     gain_p, gain_n, nullptr, 1, stream);
}

extern "C" int bmf_cover_rescore_f4_general(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* compact_pq_plane,
                                            int64_t rows_cap, int64_t ld_bytes, const int32_t* cand_pop,
                                            const int32_t* comp_tp, const int32_t* comp_fp, double w_fp, double w_fn,
                                            const int32_t* dyn_rows, int32_t gain_sign, int64_t* gain_p, int64_t* gain_n,
                                            bmf_stream_t stream) {
  BMF_REQUIRE(dyn_rows != nullptr && (gain_sign == 1 || gain_sign == -1), "bmf_cover_rescore_f4_general: dyn_rows / gain_sign");
  return cover_score_f4_general_impl(cand_plane, cand_pad, compact_pq_plane, rows_cap, ld_bytes, cand_pop, comp_tp, comp_fp,
                                     w_fp, w_fn, gain_p, gain_n, dyn_rows, gain_sign, stream);
}


// Tensor-pipe ceiling probe: see tc::probe.  kind 0 = kind::i8 (256 x 256 x 32 per instruction), 1 = kind::mxf4
// (256 x 256 x 64).  Enqueues ONE launch of `iters` x 4 instructions per CTA pair on every TPC; the caller times it with
// CUDA events.  *ops_out (host pointer) receives the operations the launch performs (2 * M * N * K per instruction).
extern "C" int bmf_probe_mma_rate(int32_t kind, int32_t iters, double* ops_out_host, bmf_stream_t stream) {
  BMF_REQUIRE((kind == 0 || kind == 1) && iters > 0 && iters <= (1 << 24), "bmf_probe_mma_rate: kind 0/1, 0 < iters <= 2^24");
  const int pairs = num_sms() / 2;
  int rc;
  if (kind == 1) {
    rc = check_cuda(cudaFuncSetAttribute(tc::probe::mma_rate_probe_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         tc::probe::PROBE_SMEM), "bmf_probe_mma_rate");
    if (rc) return rc;
    tc::probe::mma_rate_probe_kernel<1><<<2 * pairs, tc::probe::PROBE_THREADS, tc::probe::PROBE_SMEM, as_stream(stream)>>>(iters, 12345u);
  } else {
    rc = check_cuda(cudaFuncSetAttribute(tc::probe::mma_rate_probe_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         tc::probe::PROBE_SMEM), "bmf_probe_mma_rate");
    if (rc) return rc;
    tc::probe::mma_rate_probe_kernel<0><<<2 * pairs, tc::probe::PROBE_THREADS, tc::probe::PROBE_SMEM, as_stream(stream)>>>(iters, 12345u);
  }
  if (ops_out_host) *ops_out_host = 2.0 * 256.0 * 256.0 * (kind == 1 ? 64.0 : 32.0) * 4.0 * (double)iters * (double)pairs;
  return check_cuda(cudaGetLastError(), "bmf_probe_mma_rate launch");
}
