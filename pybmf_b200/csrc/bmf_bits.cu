// Bit-packed kernels of the Asso hot path (sm_100a): packing, popcount contractions,
// covered-mask update, Boolean product, confusion counts, AssoIter column refinement.
// All of these are streaming integer kernels bound by HBM bandwidth or by the integer
// pipe (POPC); rows are 16-byte aligned so every row stream uses 128-bit loads.
#include <stdlib.h>

#include <algorithm>
#include <climits>
#include <map>
#include <mutex>
#include <utility>

#include "bmf_common.cuh"

namespace bmf {

// =========================================================================================
// packing
// =========================================================================================
__global__ void pack_csr_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                int64_t m, int transposed, unsigned long long* __restrict__ bits,
                                int64_t words) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp0; r < m; r += nwarps) {
    const int64_t beg = indptr[r], end = indptr[r + 1];
    for (int64_t e = beg + lane; e < end; e += 32) {
      const int64_t c = indices[e];
      if (!transposed)
        atomicOr(bits + r * words + (c >> 6), 1ull << (c & 63));
      else
        atomicOr(bits + c * words + (r >> 6), 1ull << (r & 63));
    }
  }
}

// 16 bits -> 16 int8 per thread, one 128-bit store
__global__ void expand_bits_i8_kernel(const uint64_t* __restrict__ bits, const uint64_t* __restrict__ mask,
                                      int64_t rows, int64_t ncols, int64_t words, int one, int zero, int masked,
                                      int8_t* __restrict__ plane, int64_t rows_pad, int64_t ld) {
  const int64_t chunks = ld >> 4;
  const int64_t total = rows_pad * chunks;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / chunks, ch = t - r * chunks;
    const int64_t c0 = ch << 4;
    uint32_t out[4] = {0, 0, 0, 0};
    if (r < rows && c0 < ncols) {
      const int64_t w = c0 >> 6;
      const uint32_t b16 = (w < words) ? (uint32_t)((bits[r * words + w] >> (c0 & 63)) & 0xffffu) : 0u;
      const uint32_t k16 = (mask != nullptr && w < words) ? (uint32_t)((mask[r * words + w] >> (c0 & 63)) & 0xffffu) : 0u;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        int v = 0;
        if (c0 + i < ncols) v = ((k16 >> i) & 1u) ? masked : (((b16 >> i) & 1u) ? one : zero);
        out[i >> 2] |= (uint32_t)(uint8_t)(int8_t)v << ((i & 3) * 8);
      }
    }
    *reinterpret_cast<uint4*>(plane + r * ld + c0) = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// 8 bits -> 8 nibbles (bit i lands on the least significant bit of nibble i); multiplying the result by a 4-bit
// code then writes that code into every selected nibble (codes <= 7: no carries between nibbles)
__device__ __forceinline__ uint32_t spread8(uint32_t x) {
  x = (x | (x << 12)) & 0x000F000Fu;
  x = (x | (x << 6)) & 0x03030303u;
  x = (x | (x << 3)) & 0x11111111u;
  return x;
}

// 16 bits -> 16 nibbles holding `code` where the bit is set (element k in byte k / 2, low nibble for even k).  The bits
// are first spread into 2-bit groups, one per nibble; each nibble then SELECTS, through PRMT, the byte that encodes its
// two elements: {0, code, code << 4, code | code << 4}.  Nine instructions per 16 elements; the shift-and-mask spread to
// single nibbles followed by a multiply took 3.5x as many, which made the plane expansions instruction bound
// (4.3 GB written at 2.3 TB/s).
__device__ __forceinline__ uint32_t f4_pair_lut(uint32_t code) { return (code | (code << 4)) << 24 | (code << 4) << 16 | code << 8; }
__device__ __forceinline__ void f4_spread16(uint32_t x16, uint32_t lut, uint32_t& lo, uint32_t& hi) {
  uint32_t t = x16;
  t = (t | (t << 8)) & 0x00FF00FFu;
  t = (t | (t << 4)) & 0x0F0F0F0Fu;
  t = (t | (t << 2)) & 0x33333333u;                        // bits 2j, 2j+1 -> nibble j
  lo |= __byte_perm(lut, 0u, t);
  hi |= __byte_perm(lut, 0u, t >> 16);
}
// 32 data bits + 32 mask bits -> 32 E2M1 codes (16 bytes): `masked` where the mask bit is set, else `one` / `zero`;
// a set whose code is 0 costs nothing (the codes are launch constants, so the branches are uniform)
__device__ __forceinline__ uint4 f4_codes32(uint32_t b32, uint32_t k32, uint32_t valid, uint32_t one, uint32_t zero,
                                            uint32_t masked) {
  uint32_t out[4] = {0u, 0u, 0u, 0u};
  if (one) {
    const uint32_t s = b32 & ~k32 & valid, lut = f4_pair_lut(one);
    f4_spread16(s & 0xFFFFu, lut, out[0], out[1]);
    f4_spread16(s >> 16, lut, out[2], out[3]);
  }
  if (zero) {
    const uint32_t s = ~b32 & ~k32 & valid, lut = f4_pair_lut(zero);
    f4_spread16(s & 0xFFFFu, lut, out[0], out[1]);
    f4_spread16(s >> 16, lut, out[2], out[3]);
  }
  if (masked) {
    const uint32_t s = k32 & valid, lut = f4_pair_lut(masked);
    f4_spread16(s & 0xFFFFu, lut, out[0], out[1]);
    f4_spread16(s >> 16, lut, out[2], out[3]);
  }
  return make_uint4(out[0], out[1], out[2], out[3]);
}
// 16 data bits + 16 mask bits -> 16 int8 values
__device__ __forceinline__ uint4 i8_bytes16(uint32_t b16, uint32_t k16, uint32_t valid16, int one, int zero, int masked) {
  uint32_t out[4] = {0, 0, 0, 0};
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    int v = 0;
    if ((valid16 >> i) & 1u) v = ((k16 >> i) & 1u) ? masked : (((b16 >> i) & 1u) ? one : zero);
    out[i >> 2] |= (uint32_t)(uint8_t)(int8_t)v << ((i & 3) * 8);
  }
  return make_uint4(out[0], out[1], out[2], out[3]);
}

// One warp per plane row, 32 elements (16 bytes of E2M1 codes, one 128-bit store) per lane and pass: a pass reads 16 bit
// words (two lanes share one, a broadcast) and writes 512 contiguous bytes -- fully coalesced sectors; there is no index
// arithmetic beyond a pointer bump.  Element k of a row lives in byte k/2, low nibble for even k; rows >= `rows` and
// columns >= ncols are zero.
__global__ void __launch_bounds__(256)
expand_bits_f4_kernel(const uint64_t* __restrict__ bits, const uint64_t* __restrict__ mask,
                      int64_t rows, int64_t ncols, int64_t words, uint32_t one, uint32_t zero,
                      uint32_t masked, uint8_t* __restrict__ plane, int64_t rows_pad, int64_t ld_bytes) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t pieces = ld_bytes >> 4;                            // 32-element groups per plane row
  for (int64_t r = warp0; r < rows_pad; r += nwarps) {
    uint4* dst = reinterpret_cast<uint4*>(plane + r * ld_bytes);
    const bool live = r < rows;
    for (int64_t q0 = lane; q0 < pieces; q0 += 128) {              // four pieces per lane: eight loads in flight, then the math
      uint64_t bw[4], kw[4];
      uint32_t valid[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t q = q0 + 32 * u, w = q >> 1, left = ncols - (q << 5);
        const bool ok = live && q < pieces && w < words && left > 0;
        bw[u] = ok ? bits[r * words + w] : 0ull;
        kw[u] = (ok && mask != nullptr) ? mask[r * words + w] : 0ull;
        valid[u] = ok ? (left >= 32 ? 0xFFFFFFFFu : ((1u << left) - 1u)) : 0u;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t q = q0 + 32 * u;
        if (q >= pieces) break;
        const int sh = (int)(q & 1) * 32;
        dst[q] = f4_codes32((uint32_t)(bw[u] >> sh), (uint32_t)(kw[u] >> sh), valid[u], one, zero, masked);
      }
    }
  }
}

// Codes of one 64-column bit word at mapped plane positions: `masked` where c is set, else `one` where x is set (the zero
// code is 0, so only set bits cost work).  Element e of a row is nibble e % 8 of 32-bit word e / 8; lanes may share a
// word, hence the atomics.  col_pos == nullptr is the identity map.
__device__ __forceinline__ void f4_scatter64(uint32_t* row, uint64_t x, uint64_t c, uint64_t valid, int64_t col0,
                                             const int32_t* __restrict__ col_pos, uint32_t one, uint32_t masked) {
  uint64_t s = (x | c) & valid;
  while (s) {
    const int t = __ffsll((long long)s) - 1;
    s &= s - 1;
    const uint32_t code = ((c >> t) & 1ull) ? masked : one;
    if (code) {
      const int64_t e = col_pos != nullptr ? (int64_t)col_pos[col0 + t] : col0 + t;
      atomicOr(row + (e >> 3), code << ((e & 7) * 4));
    }
  }
}

// bmf_expand_bits_f4 with maps (the block-sparse scorer's operand order): plane row r < rows holds bit row row_src[r], and
// column k of it lands on element col_pos[k].  One warp per plane row: the row is built in a zeroed shared-memory copy by
// f4_scatter64 and written with coalesced 128-bit stores.
__global__ void __launch_bounds__(256)
expand_bits_f4_mapped_kernel(const uint64_t* __restrict__ bits, const uint64_t* __restrict__ mask, int64_t rows,
                             int64_t ncols, int64_t words, uint32_t one, uint32_t masked, const int32_t* __restrict__ row_src,
                             const int32_t* __restrict__ col_pos, uint8_t* __restrict__ plane, int64_t rows_pad,
                             int64_t ld_bytes) {
  extern __shared__ uint4 expand_smem[];
  const int lane = threadIdx.x & 31;
  const int64_t n16 = ld_bytes >> 4;
  uint4* buf = expand_smem + (threadIdx.x >> 5) * n16;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp0; r < rows_pad; r += nwarps) {
    for (int64_t q = lane; q < n16; q += 32) buf[q] = make_uint4(0u, 0u, 0u, 0u);
    __syncwarp();
    if (r < rows) {
      const int64_t src = row_src != nullptr ? (int64_t)row_src[r] : r;
      for (int64_t w = lane; w < words && w * 64 < ncols; w += 32) {
        const int64_t left = ncols - w * 64;
        const uint64_t valid = left >= 64 ? ~0ull : ((1ull << left) - 1ull);
        f4_scatter64(reinterpret_cast<uint32_t*>(buf), bits[src * words + w], mask != nullptr ? mask[src * words + w] : 0ull,
                     valid, w * 64, col_pos, one, masked);
      }
    }
    __syncwarp();
    uint4* dst = reinterpret_cast<uint4*>(plane + r * ld_bytes);
    for (int64_t q = lane; q < n16; q += 32) dst[q] = buf[q];
    __syncwarp();
  }
}

// Per bit row j: row_first[j] = its lowest set column (ncols when the row is empty); col_first[k] = min of row_rank[j] over
// the rows j that hold column k (the caller fills col_first with INT_MAX first).  Either output is nullable.  One warp per row.
__global__ void __launch_bounds__(256)
bits_first_set_kernel(const uint64_t* __restrict__ bits, int64_t rows, int64_t ncols, int64_t words,
                      const int32_t* __restrict__ row_rank, int32_t* __restrict__ row_first, int32_t* __restrict__ col_first) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t j = warp0; j < rows; j += nwarps) {
    const int rank = col_first != nullptr ? row_rank[j] : 0;
    int first = INT_MAX;
    for (int64_t w = lane; w < words && w * 64 < ncols; w += 32) {
      const int64_t left = ncols - w * 64;
      uint64_t b = bits[j * words + w] & (left >= 64 ? ~0ull : ((1ull << left) - 1ull));
      if (b != 0ull && first == INT_MAX) first = (int)(w * 64) + __ffsll((long long)b) - 1;
      if (col_first != nullptr)
        while (b) {
          const int t = __ffsll((long long)b) - 1;
          b &= b - 1;
          atomicMin(col_first + w * 64 + t, rank);
        }
    }
    first = (int)__reduce_min_sync(0xffffffffu, (unsigned)first);
    if (row_first != nullptr && lane == 0) row_first[j] = first == INT_MAX ? (int)ncols : first;
  }
}

// x bits + covered mask -> the interleaved P/Q operand of the general-weights tensor-core scorer:
// per block of 128 data rows, 128 rows of P_i = x_i & ~c_i followed by 128 rows of Q_i = c_i (0/1 bytes);
// plane row of data row i: (i / 128) * 256 + (i % 128) for P, + 128 for Q.  Padding rows / columns are 0.
__global__ void expand_bits_pq_kernel(const uint64_t* __restrict__ xb, const uint64_t* __restrict__ cb,
                                      int64_t rows, int64_t ncols, int64_t words, int8_t* __restrict__ plane,
                                      int64_t plane_rows, int64_t ld) {
  const int64_t chunks = ld >> 4;
  const int64_t total = plane_rows * chunks;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pr = t / chunks, ch = t - pr * chunks;
    const int64_t c0 = ch << 4;
    const int64_t r = (pr >> 8) * 128 + (pr & 127);
    const bool is_q = (pr & 128) != 0;
    uint32_t out[4] = {0, 0, 0, 0};
    const int64_t w = c0 >> 6;
    if (r < rows && c0 < ncols && w < words) {
      const uint32_t x16 = (uint32_t)((xb[r * words + w] >> (c0 & 63)) & 0xffffu);
      const uint32_t c16 = (uint32_t)((cb[r * words + w] >> (c0 & 63)) & 0xffffu);
      const uint32_t b16 = is_q ? c16 : (x16 & ~c16);
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (c0 + i < ncols) out[i >> 2] |= ((b16 >> i) & 1u) << ((i & 3) * 8);
    }
    *reinterpret_cast<uint4*>(plane + pr * ld + c0) = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// the same P/Q operand as packed E2M1 0/1 for the FP4 kernel: blocks of 120 data rows (its tile holds 120 P + 120 Q)
__global__ void expand_bits_pq_f4_kernel(const uint64_t* __restrict__ xb, const uint64_t* __restrict__ cb,
                                         int64_t rows, int64_t ncols, int64_t words, uint8_t* __restrict__ plane,
                                         int64_t plane_rows, int64_t ld_bytes) {
  const int64_t chunks = ld_bytes >> 4;
  const int64_t total = plane_rows * chunks;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pr = t / chunks, ch = t - pr * chunks;
    const int64_t c0 = ch << 5;
    const int64_t blk = pr / 240, within = pr - blk * 240;
    const bool is_q = within >= 120;
    const int64_t r = blk * 120 + (is_q ? within - 120 : within);
    uint32_t out[4] = {0, 0, 0, 0};
    const int64_t w = c0 >> 6;
    if (r < rows && c0 < ncols && w < words) {
      const uint32_t x32 = (uint32_t)(xb[r * words + w] >> (c0 & 63));
      const uint32_t c32 = (uint32_t)(cb[r * words + w] >> (c0 & 63));
      const int64_t left = ncols - c0;
      const uint32_t valid = left >= 32 ? 0xFFFFFFFFu : ((1u << left) - 1u);
      const uint32_t b32 = (is_q ? c32 : (x32 & ~c32)) & valid;
#pragma unroll
      for (int q = 0; q < 4; ++q) out[q] = spread8((b32 >> (8 * q)) & 0xFFu) * 2u;        // E2M1 code 2 = 1.0
    }
    *reinterpret_cast<uint4*>(plane + pr * ld_bytes + (ch << 4)) = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// =========================================================================================
// popcount contraction tiles.  Block = 256 threads computes a 64 x 64 tile of
// (row i of A) x (row j of B); thread (ty, tx) owns rows ty*4+r and columns c*16+tx so that
// shared-memory reads of B are conflict free and reads of A are broadcasts.
// =========================================================================================
constexpr int PT = 64;    // tile edge
constexpr int PW = 16;    // words per shared-memory chunk
constexpr int PWP = PW + 1;

__device__ __forceinline__ void stage_words(uint64_t (*dst)[PWP], const uint64_t* __restrict__ src,
                                            int64_t row0, int64_t nrows, int64_t words, int64_t w0) {
  // 64 rows x 16 words, 256 threads: each thread moves 4 words
  for (int e = threadIdx.x; e < PT * PW; e += blockDim.x) {
    const int r = e / PW, w = e % PW;
    const int64_t gr = row0 + r, gw = w0 + w;
    dst[r][w] = (gr < nrows && gw < words) ? __ldg(src + gr * words + gw) : 0ull;
  }
}

__global__ void __launch_bounds__(256) assoc_counts_popc_kernel(const uint64_t* __restrict__ xt, int64_t n,
                                                               int64_t words, int32_t* __restrict__ cnt,
                                                               int64_t ldc) {
  __shared__ uint64_t As[PT][PWP];
  __shared__ uint64_t Bs[PT][PWP];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t i0 = (int64_t)blockIdx.y * PT, j0 = (int64_t)blockIdx.x * PT;
  int acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0;
  for (int64_t w0 = 0; w0 < words; w0 += PW) {
    stage_words(As, xt, i0, n, words, w0);
    stage_words(Bs, xt, j0, n, words, w0);
    __syncthreads();
#pragma unroll 4
    for (int w = 0; w < PW; ++w) {
      uint64_t a[4], b[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = As[ty * 4 + r][w];
#pragma unroll
      for (int c = 0; c < 4; ++c) b[c] = Bs[c * 16 + tx][w];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] += __popcll(a[r] & b[c]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int64_t i = i0 + ty * 4 + r, j = j0 + c * 16 + tx;
      if (i < n && j < n) cnt[i * ldc + j] = acc[r][c];
    }
}

// basis bit (i, j) = cnt[i][j] / cnt[i][i] > tau, one warp per row, one 64-bit word per lane pass
// Rows [row0, row0 + nrows) of the n x n matrix; cnt / basis_bits / cand_plane / alive / row_pop point at row row0
// (multi-GPU: every rank thresholds the row block it received from the reduce-scatter).  symmetric != 0 (row0 = 0
// only): the counts below the diagonal were never computed, cnt[i][j] is read as cnt[min][max].
// The reference's test is `(double)c / (double)s > tau` (IEEE division, strict; Asso.py:207-212 + binarize).  Correctly
// rounded division is monotone in c, so for a row with support s the test holds exactly for c >= c_min(s, tau): c_min is
// found once per row with the LITERAL division around floor(tau * s), and the n^2 elements are compared as integers
// (B200's fp64 divide is a long instruction sequence: 316 M of them were most of this kernel).  No c in [0, s] passes
// (tau >= 1, NaN) -> s + 1; counts never exceed s.
__device__ __forceinline__ int32_t assoc_min_count(int32_t si, double tau) {
  if (si <= 0) return 0.0 > tau ? 0 : 1;                  // empty column: the reference sets its association row to 0 (Asso.py:211)
  const double s = (double)si;
  auto passes = [&](int32_t c) { return ((double)c / s) > tau; };
  const double guess = tau * s;
  int32_t c = guess >= s ? si : (guess > 0.0 ? (int32_t)guess : 0);       // NaN -> 0, walks up to s + 1 only if nothing passes
  if (!(tau == tau)) return si + 1;
  while (c > 0 && passes(c - 1)) --c;
  while (c <= si && !passes(c)) ++c;
  return c;
}

__global__ void basis_threshold_kernel(const int32_t* __restrict__ cnt, int64_t ldc, int64_t n, int64_t row0,
                                       int64_t nrows, int symmetric, double tau,
                                       uint64_t* __restrict__ basis_bits, int64_t words,
                                       int8_t* __restrict__ cand_plane, int64_t ld,
                                       uint8_t* __restrict__ alive, int32_t* __restrict__ row_pop) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp0; i < nrows; i += nwarps) {
    const int64_t gi = row0 + i;                 // global row = diagonal column
    const int32_t si = cnt[i * ldc + gi];
    const int32_t cmin = assoc_min_count(si, tau);
    int any = 0, pop = 0;
    for (int64_t w = 0; w < words; ++w) {       // each pass: 2 x 32 columns -> one word
      uint64_t word = 0;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int64_t j = w * 64 + h * 32 + lane;
        bool bit = false;
        if (j < n) {
          const int32_t cij = (symmetric && j < gi) ? cnt[j * ldc + gi] : cnt[i * ldc + j];
          bit = cij >= cmin;                                                 // <=> (double)cij / (double)si > tau
        }
        if (cand_plane != nullptr && j < ld) cand_plane[i * ld + j] = bit ? 1 : 0;
        const uint32_t bal = __ballot_sync(0xffffffffu, bit);
        word |= (uint64_t)bal << (h * 32);
      }
      if (lane == 0) basis_bits[i * words + w] = word;
      any |= (word != 0);
      pop += __popcll(word);
    }
    if (cand_plane != nullptr)                     // tail of the padded row beyond words*64
      for (int64_t j = words * 64 + lane; j < ld; j += 32) cand_plane[i * ld + j] = 0;
    if (lane == 0) {
      alive[i] = any ? 1 : 0;
      if (row_pop != nullptr) row_pop[i] = pop;
    }
  }
}

// Tile form of the threshold for the UPPER-stored symmetric count matrix of one GPU (the row-per-warp kernel above reads
// cnt[j][i] for j < i down a column: one 32-byte sector per 4 useful bytes, 1.15 ms at n = 17770).  A block takes a 64 x 64
// tile (bi <= bj) of the stored triangle with coalesced row reads and emits BOTH words it decides: basis[i][bj] for the
// tile's rows against their own minimal counts, and -- reading the tile transposed out of shared memory -- basis[j][bi] for
// the tile's columns against theirs.  basis_rows_finish_kernel then counts each row (alive, |b_i|) and clears the pad words.
constexpr int BT = 64;
__global__ void __launch_bounds__(256)
basis_threshold_tile_kernel(const int32_t* __restrict__ cnt, int64_t ldc, int64_t n, double tau,
                            const int32_t* __restrict__ min_count, uint64_t* __restrict__ basis_bits, int64_t words) {
  const int bi = blockIdx.y, bj = blockIdx.x;
  if (bi > bj) return;
  __shared__ int32_t tile[BT][BT + 1];
  __shared__ int32_t cmin_i[BT], cmin_j[BT];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t i0 = (int64_t)bi * BT, j0 = (int64_t)bj * BT;
  if (threadIdx.x < 2 * BT) {                                   // minimal counts of the tile's rows and of its columns
    const int t = threadIdx.x & (BT - 1);
    const int64_t g = (threadIdx.x < BT ? i0 : j0) + t;
    const int32_t c = g >= n ? 0x7fffffff : (min_count != nullptr ? min_count[g] : assoc_min_count(cnt[g * ldc + g], tau));
    if (threadIdx.x < BT) cmin_i[t] = c; else cmin_j[t] = c;
  }
  for (int a = warp; a < BT; a += 8) {                          // 64 rows x 256 bytes, coalesced
    const int64_t gi = i0 + a;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t gj = j0 + h * 32 + lane;
      tile[a][h * 32 + lane] = (gi < n && gj < n) ? cnt[gi * ldc + gj] : 0;
    }
  }
  __syncthreads();
  const bool diag = bi == bj;                                   // only a <= b is stored there: read tile[min][max]
  for (int a = warp * 8; a < warp * 8 + 8; ++a) {
    const int32_t need = cmin_i[a];
    uint64_t word = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int b = h * 32 + lane;
      const int32_t c = (diag && b < a) ? tile[b][a] : tile[a][b];
      const bool bit = (j0 + b < n) && c >= need;
      word |= (uint64_t)__ballot_sync(0xffffffffu, bit) << (h * 32);
    }
    if (lane == 0 && i0 + a < n) basis_bits[(i0 + a) * words + bj] = word;
  }
  if (diag) return;
  for (int b = warp * 8; b < warp * 8 + 8; ++b) {               // the mirrored word: rows j of block bj, columns of block bi
    const int32_t need = cmin_j[b];
    uint64_t word = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int a = h * 32 + lane;
      const bool bit = (i0 + a < n) && tile[a][b] >= need;
      word |= (uint64_t)__ballot_sync(0xffffffffu, bit) << (h * 32);
    }
    if (lane == 0 && j0 + b < n) basis_bits[(j0 + b) * words + bi] = word;
  }
}
// c_min of every column, once (the fp64 divisions it takes are long sequences: 2 x 64 of them per tile were half the tile kernel)
__global__ void assoc_min_counts_kernel(const int32_t* __restrict__ cnt, int64_t ldc, int64_t n, double tau,
                                        int32_t* __restrict__ min_count) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n) min_count[g] = assoc_min_count(cnt[g * ldc + g], tau);
}
__global__ void __launch_bounds__(256)
basis_rows_finish_kernel(uint64_t* __restrict__ basis_bits, int64_t n, int64_t words, int64_t used_words,
                         uint8_t* __restrict__ alive, int32_t* __restrict__ row_pop) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= n) return;
  int pop = 0;
  for (int64_t w = lane; w < words; w += 32) {
    if (w < used_words) pop += __popcll(basis_bits[i * words + w]);
    else basis_bits[i * words + w] = 0ull;
  }
  pop = warp_sum(pop);
  if (lane == 0) {
    alive[i] = pop ? 1 : 0;
    if (row_pop != nullptr) row_pop[i] = pop;
  }
}

// =========================================================================================
// cover-gain scoring, popcount variant.
// grid.x = candidate tiles (64), grid.y = row splits; every block walks its share of row
// tiles and keeps per-candidate partial gains in registers; one atomic per candidate at the end.
// =========================================================================================
__global__ void __launch_bounds__(256)
cover_score_popc_kernel(const uint64_t* __restrict__ xb, const uint64_t* __restrict__ cb, int64_t m,
                        int64_t n, int64_t words, const uint64_t* __restrict__ basis,
                        const uint8_t* __restrict__ alive, const int32_t* __restrict__ tp_old,
                        const int32_t* __restrict__ fp_old, int wa, int wb, double neg_w_fp, double w_fn,
                        unsigned long long* __restrict__ gain_p, unsigned long long* __restrict__ gain_n) {
  __shared__ uint64_t Ps[PT][PWP];   // x & ~c        (uncovered ones)
  __shared__ uint64_t Ns[PT][PWP];   // ~x & ~c & valid (uncovered zeros)
  __shared__ uint64_t Bs[PT][PWP];
  __shared__ long long red_p[PT];
  __shared__ long long red_n[PT];
  __shared__ int any_alive;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t j0 = (int64_t)blockIdx.x * PT;
  if (threadIdx.x == 0) any_alive = 0;
  if (threadIdx.x < PT) { red_p[threadIdx.x] = 0; red_n[threadIdx.x] = 0; }
  __syncthreads();
  if (threadIdx.x < PT && j0 + threadIdx.x < n && alive[j0 + threadIdx.x]) any_alive = 1;
  __syncthreads();
  if (!any_alive) return;

  long long gp[4] = {0, 0, 0, 0}, gn[4] = {0, 0, 0, 0};
  // A row whose cover is still empty has N = |b_j| - P: its second contraction is redundant, |b_j| is counted once per
  // candidate instead (4 popcounts per word instead of 16).  cov_rows[r] says whether row r of the tile has any cover.
  __shared__ int cov_rows[PT];
  const int64_t row_tiles = (m + PT - 1) / PT;
  for (int64_t rt = blockIdx.y; rt < row_tiles; rt += gridDim.y) {
    const int64_t i0 = rt * PT;
    int accp[4][4], accn[4][4], accb[4] = {0, 0, 0, 0};
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) { accp[r][c] = 0; accn[r][c] = 0; }
    if (threadIdx.x < PT) cov_rows[threadIdx.x] = 0;
    __syncthreads();
    for (int64_t w0 = 0; w0 < words; w0 += PW)                      // pass 1 over the tile's cover words: which rows are covered?
      for (int e = threadIdx.x; e < PT * PW; e += blockDim.x) {
        const int r = e / PW, w = e % PW;
        const int64_t gr = i0 + r, gw = w0 + w;
        if (gr < m && gw < words && __ldg(cb + gr * words + gw) != 0ull) cov_rows[r] = 1;
      }
    __syncthreads();
    bool need_n[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) need_n[r] = cov_rows[ty * 4 + r] != 0;
    const bool any_need = need_n[0] | need_n[1] | need_n[2] | need_n[3];
    for (int64_t w0 = 0; w0 < words; w0 += PW) {
      for (int e = threadIdx.x; e < PT * PW; e += blockDim.x) {
        const int r = e / PW, w = e % PW;
        const int64_t gr = i0 + r, gw = w0 + w;
        uint64_t p = 0, q = 0;
        if (gr < m && gw < words) {
          const uint64_t x = __ldg(xb + gr * words + gw), c = __ldg(cb + gr * words + gw);
          const int64_t rem = n - gw * 64;                      // valid columns in this word
          const uint64_t valid = rem >= 64 ? ~0ull : (rem <= 0 ? 0ull : ((1ull << rem) - 1ull));
          p = x & ~c;
          q = ~x & ~c & valid;
        }
        Ps[r][w] = p;
        Ns[r][w] = q;
      }
      stage_words(Bs, basis, j0, n, words, w0);
      __syncthreads();
#pragma unroll 2
      for (int w = 0; w < PW; ++w) {
        uint64_t p[4], q[4], b[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) { p[r] = Ps[ty * 4 + r][w]; q[r] = Ns[ty * 4 + r][w]; }
#pragma unroll
        for (int c = 0; c < 4; ++c) { b[c] = Bs[c * 16 + tx][w]; accb[c] += __popcll(b[c]); }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) accp[r][c] += __popcll(p[r] & b[c]);
        if (any_need) {
#pragma unroll
          for (int r = 0; r < 4; ++r)
            if (need_n[r]) {
#pragma unroll
              for (int c = 0; c < 4; ++c) accn[r][c] += __popcll(q[r] & b[c]);
            }
        }
      }
      __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int64_t i = i0 + ty * 4 + r;
      if (i >= m) continue;
      int tpo = 0, fpo = 0;
      if (!(wa | wb)) { tpo = tp_old[i]; fpo = fp_old[i]; }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int P = accp[r][c], N = need_n[r] ? accn[r][c] : accb[c] - accp[r][c];
        if (wa | wb) {
          const int d = wb * P - wa * N;
          gp[c] += d > 0 ? d : 0;
        } else if (row_uses(0, 0, neg_w_fp, w_fn, tpo, fpo, P, N)) {
          gp[c] += P;
          gn[c] += N;
        }
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    atomicAdd((unsigned long long*)&red_p[c * 16 + tx], (unsigned long long)gp[c]);
    if (!(wa | wb)) atomicAdd((unsigned long long*)&red_n[c * 16 + tx], (unsigned long long)gn[c]);
  }
  __syncthreads();
  if (threadIdx.x < PT && j0 + threadIdx.x < n) {
    atomicAdd(gain_p + j0 + threadIdx.x, (unsigned long long)red_p[threadIdx.x]);
    if (!(wa | wb)) atomicAdd(gain_n + j0 + threadIdx.x, (unsigned long long)red_n[threadIdx.x]);
  }
}

// =========================================================================================
// argmax with the reference's tie-breaking (first strict maximum above the inherited best)
// =========================================================================================
__global__ void __launch_bounds__(1024)
select_first_max_kernel(const int64_t* __restrict__ gain_p, const int64_t* __restrict__ gain_n,
                        const uint8_t* __restrict__ alive, int64_t n, int wa, int wb, int64_t base_int,
                        double scale, double neg_w_fp, double w_fn, int64_t tp_tot, int64_t fp_tot,
                        double best_score, int64_t* __restrict__ record) {
  __shared__ double s_val[32];
  __shared__ long long s_idx[32];
  double best = 0.0;
  long long idx = -1;
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
    if (!alive[j]) continue;
    double sc;
    if (wa | wb)
      sc = __dmul_rn((double)(base_int + gain_p[j]), scale);
    else
      sc = __dadd_rn(__dmul_rn(neg_w_fp, (double)(fp_tot + gain_n[j])),
                     __dmul_rn(w_fn, (double)(tp_tot + gain_p[j])));
    if (idx < 0 || sc > best) { best = sc; idx = j; }   // ascending j per thread: first max kept
  }
  // warp then block reduction; on equal scores the lower index wins
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (oi >= 0 && (idx < 0 || ov > best || (ov == best && oi < idx))) { best = ov; idx = oi; }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_val[warp] = best; s_idx[warp] = idx; }
  __syncthreads();
  if (warp == 0) {
    best = s_val[lane];
    idx = s_idx[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, best, o);
      const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
      if (oi >= 0 && (idx < 0 || ov > best || (ov == best && oi < idx))) { best = ov; idx = oi; }
    }
    if (lane == 0) {
      if (idx >= 0 && !(best > best_score)) idx = -1;       // Asso.py:94 `score > best_score`
      record[0] = idx;
      record[1] = __double_as_longlong(idx >= 0 ? best : best_score);
    }
  }
}

// =========================================================================================
// The argmax of a DEVICE-RESIDENT greedy loop: the inherited threshold, the running TP / FP totals and the per-step
// result table live in device memory, so k greedy steps are enqueued back to back without a host round trip.
//   state[0] = bits of the inherited best score, [1] = TP total, [2] = FP total, [3] = stopped, [4] = steps selected
//   table row (8 x int64): winner, score bits, #used rows, sum P, sum N, TP total after, FP total after, status
//   status: 0 = no winner, 1 = winner chosen (counters pending), 2 = complete
// `tail` holds (#used, sum P, sum N) of the PREVIOUS step's apply, already summed over the ranks (it travels at the end
// of the all-reduced gain vector, so a step needs ONE collective); they are folded into the state and the previous
// table row first.  tail_zero (the local copy) and *nused are cleared for the coming apply.
// =========================================================================================
__global__ void __launch_bounds__(1024)
greedy_select_kernel(const int64_t* __restrict__ gain_p, const int64_t* __restrict__ gain_n,
                     const long long* __restrict__ tail, long long* __restrict__ tail_zero,
                     uint8_t* __restrict__ alive, int64_t n, int wa, int wb, double scale, double neg_w_fp,
                     double w_fn, int first, long long* __restrict__ state, long long* __restrict__ row,
                     long long* __restrict__ prev_row, long long* __restrict__ record, int* __restrict__ nused) {
  __shared__ double s_val[32];
  __shared__ long long s_idx[32];
  __shared__ long long s_tp, s_fp;
  __shared__ int s_go;
  if (threadIdx.x == 0) {
    long long tp = state[1], fp = state[2];
    if (prev_row != nullptr && prev_row[7] == 1) {
      const long long used = tail[0], sp = tail[1], sn = tail[2];
      tp += sp;
      fp += sn;
      state[1] = tp;
      state[2] = fp;
      prev_row[2] = used; prev_row[3] = sp; prev_row[4] = sn; prev_row[5] = tp; prev_row[6] = fp; prev_row[7] = 2;
    }
    if (tail_zero != nullptr) { tail_zero[0] = 0; tail_zero[1] = 0; tail_zero[2] = 0; }
    if (nused != nullptr) *nused = 0;
    s_tp = tp;
    s_fp = fp;
    s_go = (row != nullptr) && state[3] == 0;
    if (!s_go) {
      record[0] = -1;
      if (row != nullptr) { row[0] = -1; row[7] = 0; }
    }
  }
  __syncthreads();
  if (!s_go) return;
  const long long tp_tot = s_tp, fp_tot = s_fp;
  const long long base_int = (long long)wb * tp_tot - (long long)wa * fp_tot;
  double best = 0.0;
  long long idx = -1;
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
    if (!alive[j]) continue;
    double sc;
    if (wa | wb)
      sc = __dmul_rn((double)(base_int + gain_p[j]), scale);
    else
      sc = __dadd_rn(__dmul_rn(neg_w_fp, (double)(fp_tot + gain_n[j])),
                     __dmul_rn(w_fn, (double)(tp_tot + gain_p[j])));
    if (idx < 0 || sc > best) { best = sc; idx = j; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (oi >= 0 && (idx < 0 || ov > best || (ov == best && oi < idx))) { best = ov; idx = oi; }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_val[warp] = best; s_idx[warp] = idx; }
  __syncthreads();
  if (warp == 0) {
    best = s_val[lane];
    idx = s_idx[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, best, o);
      const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
      if (oi >= 0 && (idx < 0 || ov > best || (ov == best && oi < idx))) { best = ov; idx = oi; }
    }
    if (lane == 0) {
      const double best_score = first ? 0.0 : __longlong_as_double(state[0]);       // Asso.py:71
      if (idx >= 0 && !(best > best_score)) idx = -1;                                // Asso.py:94 `score > best_score`
      const long long bits = __double_as_longlong(idx >= 0 ? best : best_score);
      record[0] = idx;
      record[1] = bits;
      row[0] = idx;
      row[1] = bits;
      row[2] = 0; row[3] = 0; row[4] = 0; row[5] = tp_tot; row[6] = fp_tot;
      row[7] = idx >= 0 ? 1 : 0;
      if (idx >= 0) {
        state[0] = bits;
        alive[idx] = 0;                                                              // Asso.py:106-107
      } else {
        state[3] = 1;                                                                // nothing improves: the loop is over
      }
      state[4] += 1;
    }
  }
}

// rows [*nused, round_up(*nused, tile)) of both compact planes := 0, so that the last (partial) row tile of the
// incremental GEMMs sees padding rows (which score relu(-bias) = 0)
__global__ void compact_tail_zero_kernel(uint8_t* __restrict__ a, uint8_t* __restrict__ b, int64_t ld, int64_t cap,
                                         const int* __restrict__ nused, int tile) {
  const int64_t used = *nused < cap ? *nused : cap;
  int64_t end = (used + tile - 1) / tile * tile;
  if (end > cap) end = cap;
  const int64_t chunks = ld >> 4;
  const int64_t total = (end - used) * chunks;
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = used + t / chunks, ch = t % chunks;
    reinterpret_cast<uint4*>(a + r * ld)[ch] = z;
    reinterpret_cast<uint4*>(b + r * ld)[ch] = z;
  }
}

// the same for the interleaved P/Q layouts (blocks of `blk` data rows: blk P rows then blk Q rows): slots
// [*nused, round_up(*nused, blk)) of the last block.  The FP4 general-weights epilogue settles most elements in fixed point
// WITHOUT looking at the row state, so padding rows must really be zero (P = N = 0 leaves them undecided -> fp64 -> +inf).
__global__ void compact_tail_zero_pq_kernel(uint8_t* __restrict__ a, uint8_t* __restrict__ b, int64_t ld, int64_t cap,
                                            const int* __restrict__ nused, int blk) {
  const int64_t used = *nused < cap ? *nused : cap;
  int64_t end = (used + blk - 1) / blk * blk;
  if (end > cap) end = (cap + blk - 1) / blk * blk;
  const int64_t chunks = ld >> 4;
  const int64_t total = (end - used) * chunks;
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t slot = used + t / chunks, ch = t % chunks;
    const int64_t prow = (slot / blk) * (2 * blk) + slot % blk;
    reinterpret_cast<uint4*>(a + prow * ld)[ch] = z;
    reinterpret_cast<uint4*>(b + prow * ld)[ch] = z;
    reinterpret_cast<uint4*>(a + (prow + blk) * ld)[ch] = z;
    reinterpret_cast<uint4*>(b + (prow + blk) * ld)[ch] = z;
  }
}

// =========================================================================================
// apply the chosen candidate: one warp per data row, 128-bit row streams
// =========================================================================================
// Extras of the device-resident greedy loop (all optional, zero-initialised = the plain kernel):
//  * compaction for incremental rescoring: every USED row's operand-plane row is written twice, as it was before the
//    update (comp_old) and as it is after (comp_new), at a slot drawn from the device counter *nused; the scoring GEMM
//    then runs over those few rows only: gain += sum relu(new) - sum relu(old).  The rows are generated from the bit
//    rows (x, c) with the same codes bmf_expand_bits_* uses, so the big plane need not be kept current.
//  * u_words: bit `factor_bit` of the row-major usage words (the form bmf_confusion_factors / bmf_bool_product read);
//  * vt_row: a copy of the winner's basis row (row `factor_bit` of the selected-V^T matrix).
struct ApplyExtra {
  uint8_t* comp_old;
  uint8_t* comp_new;
  int64_t comp_ld;          // bytes per compact row
  int64_t comp_cap;         // rows the buffers hold
  int* nused;               // device counter, zeroed by bmf_greedy_select
  int comp_kind;            // 0 none, 1 packed E2M1, 2 int8
  int v_one, v_zero, v_cov; // operand values (E2M1 codes for kind 1, int8 values for kind 2)
  uint64_t* u_words;
  int64_t kw;
  int factor_bit;
  uint64_t* vt_row;
  // general weights (kinds 3 = packed E2M1 P/Q blocks of 120 rows, 4 = int8 P/Q blocks of 128 rows): the used rows' per-row
  // TP / FP before and after the update travel with the compacted planes (the fp64 row test needs them)
  int32_t* comp_tp_old;
  int32_t* comp_fp_old;
  int32_t* comp_tp_new;
  int32_t* comp_fp_new;
  // packed E2M1 planes in a column order (the block-sparse scorer's): column k of X is element col_pos[k] of the rows plane
  // patch (pq_layout 2) and of the compacted rows (kind 1); nullptr = natural order
  const int32_t* col_pos;
};

// The E2M1 rows-plane patch of newly covered columns s (64 columns from col0) at mapped positions: the nibble becomes `code`
__device__ __forceinline__ void f4_patch64(uint32_t* row, uint64_t s, int64_t col0, const int32_t* __restrict__ col_pos,
                                           uint32_t code) {
  while (s) {
    const int t = __ffsll((long long)s) - 1;
    s &= s - 1;
    const int64_t e = col_pos[col0 + t];
    const int sh = (int)(e & 7) * 4;
    atomicAnd(row + (e >> 3), ~(0xFu << sh));
    atomicOr(row + (e >> 3), code << sh);
  }
}

// The update of ONE data row that uses the winner (warp-collective; P / N = the row's new true / false positives, tpo / fpo
// its counters before): usage bit, cover OR, counters, the operand-plane patch and the compacted before / after rows.
__device__ __forceinline__ void apply_used_row(const uint64_t* __restrict__ xb, uint64_t* __restrict__ cb, int64_t n, int64_t words,
                                               const uint64_t* __restrict__ b, int32_t* __restrict__ tp_old,
                                               int32_t* __restrict__ fp_old, int8_t* __restrict__ rows_plane, int64_t ld,
                                               int covered_value, int pq_layout, unsigned long long* __restrict__ u_bits,
                                               const ApplyExtra& ex, int64_t i, int lane, int P, int N, int tpo, int fpo,
                                               long long& t_used, long long& t_p, long long& t_n) {
  const int64_t pairs = words >> 1;
  int64_t slot = -1;
  if (ex.comp_kind) {
    int s0 = 0;
    if (lane == 0) s0 = atomicAdd(ex.nused, 1);
    s0 = __shfl_sync(0xffffffffu, s0, 0);
    slot = s0 < ex.comp_cap ? s0 : -1;                                // capacity = all rows: never exceeded
  }
  const bool mapped = ex.col_pos != nullptr;
  if (slot >= 0 && ex.comp_kind == 1 && mapped) {                     // mapped compact rows are scattered into zeroed rows
    for (int64_t q = lane; q < (ex.comp_ld >> 4); q += 32) {
      reinterpret_cast<uint4*>(ex.comp_old + slot * ex.comp_ld)[q] = make_uint4(0u, 0u, 0u, 0u);
      reinterpret_cast<uint4*>(ex.comp_new + slot * ex.comp_ld)[q] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncwarp();
  }
  for (int64_t p = lane; p < pairs; p += 32) {
    ulonglong2* cp = reinterpret_cast<ulonglong2*>(cb + i * words + 2 * p);
    ulonglong2 c = *cp;
    const ulonglong2 v = ld_words2(b + 2 * p);
    if (slot >= 0) {                                                  // this row before / after the update
      const ulonglong2 x = ld_words2(xb + i * words + 2 * p);
      const uint64_t xw[2] = {x.x, x.y}, cw[2] = {c.x, c.y}, nw[2] = {c.x | v.x, c.y | v.y};
      const int kind = ex.comp_kind;
      // plane row of this slot (P row for the P/Q layouts; the Q row sits q_off rows further)
      const int64_t prow = kind == 3 ? (slot / 120) * 240 + slot % 120 : (kind == 4 ? (slot >> 7) * 256 + (slot & 127) : slot);
      const int64_t q_off = (kind == 3 ? 120 : 128) * ex.comp_ld;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int64_t col0 = (2 * p + h) * 64;
        const int64_t left = n - col0;
        const uint64_t valid = left >= 64 ? ~0ull : (left <= 0 ? 0ull : ((1ull << left) - 1ull));
        if (kind == 1 && mapped) {
          f4_scatter64(reinterpret_cast<uint32_t*>(ex.comp_old + prow * ex.comp_ld), xw[h], cw[h], valid, col0, ex.col_pos,
                       ex.v_one, ex.v_cov);
          f4_scatter64(reinterpret_cast<uint32_t*>(ex.comp_new + prow * ex.comp_ld), xw[h], nw[h], valid, col0, ex.col_pos,
                       ex.v_one, ex.v_cov);
        } else if (kind == 1 || kind == 3) {                          // 64 bits -> 32 bytes of packed E2M1
          uint4* o = reinterpret_cast<uint4*>(ex.comp_old + prow * ex.comp_ld + (2 * p + h) * 32);
          uint4* q = reinterpret_cast<uint4*>(ex.comp_new + prow * ex.comp_ld + (2 * p + h) * 32);
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            const uint32_t x32 = (uint32_t)(xw[h] >> (32 * g)), vd = (uint32_t)(valid >> (32 * g));
            const uint32_t c32 = (uint32_t)(cw[h] >> (32 * g)), n32 = (uint32_t)(nw[h] >> (32 * g));
            if (kind == 1) {
              o[g] = f4_codes32(x32, c32, vd, ex.v_one, ex.v_zero, ex.v_cov);
              q[g] = f4_codes32(x32, n32, vd, ex.v_one, ex.v_zero, ex.v_cov);
            } else {                                                  // P = x & ~c and Q = c as E2M1 1.0 (code 2)
              o[g] = f4_codes32(x32 & ~c32, 0u, vd, 2u, 0u, 0u);
              q[g] = f4_codes32(x32 & ~n32, 0u, vd, 2u, 0u, 0u);
              reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(o) + q_off)[g] = f4_codes32(c32, 0u, vd, 2u, 0u, 0u);
              reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(q) + q_off)[g] = f4_codes32(n32, 0u, vd, 2u, 0u, 0u);
            }
          }
        } else {                                                      // 64 bits -> 64 int8
          uint4* o = reinterpret_cast<uint4*>(ex.comp_old + prow * ex.comp_ld + (2 * p + h) * 64);
          uint4* q = reinterpret_cast<uint4*>(ex.comp_new + prow * ex.comp_ld + (2 * p + h) * 64);
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const uint32_t x16 = (uint32_t)(xw[h] >> (16 * g)) & 0xffffu, vd = (uint32_t)(valid >> (16 * g)) & 0xffffu;
            const uint32_t c16 = (uint32_t)(cw[h] >> (16 * g)) & 0xffffu, n16 = (uint32_t)(nw[h] >> (16 * g)) & 0xffffu;
            if (kind == 2) {
              o[g] = i8_bytes16(x16, c16, vd, ex.v_one, ex.v_zero, ex.v_cov);
              q[g] = i8_bytes16(x16, n16, vd, ex.v_one, ex.v_zero, ex.v_cov);
            } else {
              o[g] = i8_bytes16(x16 & ~c16, 0u, vd, 1, 0, 0);
              q[g] = i8_bytes16(x16 & ~n16, 0u, vd, 1, 0, 0);
              reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(o) + q_off)[g] = i8_bytes16(c16, 0u, vd, 1, 0, 0);
              reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(q) + q_off)[g] = i8_bytes16(n16, 0u, vd, 1, 0, 0);
            }
          }
        }
      }
    }
    if (rows_plane != nullptr) {
      uint64_t s0 = v.x & ~c.x, s1 = v.y & ~c.y;                      // newly covered columns
      if (!pq_layout) {
        int8_t* rowp = rows_plane + i * ld + p * 128;
        while (s0) { const int k = __ffsll((long long)s0) - 1; s0 &= s0 - 1; rowp[k] = (int8_t)covered_value; }
        while (s1) { const int k = __ffsll((long long)s1) - 1; s1 &= s1 - 1; rowp[64 + k] = (int8_t)covered_value; }
      } else if (pq_layout == 2 && mapped) {
        uint32_t* roww = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(rows_plane) + i * ld);
        f4_patch64(roww, s0, p * 128, ex.col_pos, (uint32_t)covered_value & 0xFu);
        f4_patch64(roww, s1, p * 128 + 64, ex.col_pos, (uint32_t)covered_value & 0xFu);
      } else if (pq_layout == 2) {                                     // packed E2M1 plane: rewrite the nibble
        uint8_t* rowp = reinterpret_cast<uint8_t*>(rows_plane) + i * ld + p * 64;
        const uint32_t code = (uint32_t)covered_value & 0xFu;
        while (s0) {
          const int k = __ffsll((long long)s0) - 1; s0 &= s0 - 1;
          uint8_t* bp = rowp + (k >> 1);
          *bp = (k & 1) ? (uint8_t)((*bp & 0x0Fu) | (code << 4)) : (uint8_t)((*bp & 0xF0u) | code);
        }
        while (s1) {
          const int k = __ffsll((long long)s1) - 1; s1 &= s1 - 1;
          uint8_t* bp = rowp + 32 + (k >> 1);
          *bp = (k & 1) ? (uint8_t)((*bp & 0x0Fu) | (code << 4)) : (uint8_t)((*bp & 0xF0u) | code);
        }
      } else if (pq_layout == 3) {                                     // packed E2M1 P/Q planes, blocks of 120 rows
        uint8_t* rowp = reinterpret_cast<uint8_t*>(rows_plane) + ((i / 120) * 240 + (i % 120)) * ld + p * 64;
        uint8_t* rowq = rowp + 120 * ld;
        while (s0) {
          const int k = __ffsll((long long)s0) - 1; s0 &= s0 - 1;
          const int b = k >> 1;
          if (k & 1) { rowp[b] &= 0x0Fu; rowq[b] = (uint8_t)((rowq[b] & 0x0Fu) | 0x20u); }
          else       { rowp[b] &= 0xF0u; rowq[b] = (uint8_t)((rowq[b] & 0xF0u) | 0x02u); }
        }
        while (s1) {
          const int k = __ffsll((long long)s1) - 1; s1 &= s1 - 1;
          const int b = 32 + (k >> 1);
          if (k & 1) { rowp[b] &= 0x0Fu; rowq[b] = (uint8_t)((rowq[b] & 0x0Fu) | 0x20u); }
          else       { rowp[b] &= 0xF0u; rowq[b] = (uint8_t)((rowq[b] & 0xF0u) | 0x02u); }
        }
      } else {                                                         // P plane: no longer uncovered; Q plane: covered
        int8_t* rowp = rows_plane + ((i >> 7) * 256 + (i & 127)) * ld + p * 128;
        int8_t* rowq = rowp + 128 * ld;
        while (s0) { const int k = __ffsll((long long)s0) - 1; s0 &= s0 - 1; rowp[k] = 0; rowq[k] = 1; }
        while (s1) { const int k = __ffsll((long long)s1) - 1; s1 &= s1 - 1; rowp[64 + k] = 0; rowq[64 + k] = 1; }
      }
    }
    c.x |= v.x;
    c.y |= v.y;
    *cp = c;
  }
  if (slot >= 0) {                                                    // K padding of the compact rows (never written above)
    const int kind = ex.comp_kind;
    const int64_t used_bytes = words * ((kind == 1 || kind == 3) ? 32 : 64);
    const int64_t prow = kind == 3 ? (slot / 120) * 240 + slot % 120 : (kind == 4 ? (slot >> 7) * 256 + (slot & 127) : slot);
    const int64_t q_off = (kind == 3 ? 120 : 128) * ex.comp_ld;
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    for (int64_t q = lane; q < ((ex.comp_ld - used_bytes) >> 4); q += 32) {
      uint4* o = reinterpret_cast<uint4*>(ex.comp_old + prow * ex.comp_ld + used_bytes) + q;
      uint4* w = reinterpret_cast<uint4*>(ex.comp_new + prow * ex.comp_ld + used_bytes) + q;
      *o = z;
      *w = z;
      if (kind >= 3) {
        *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(o) + q_off) = z;
        *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(w) + q_off) = z;
      }
    }
    if (lane == 0 && kind >= 3) {
      ex.comp_tp_old[slot] = tpo; ex.comp_fp_old[slot] = fpo;
      ex.comp_tp_new[slot] = tpo + P; ex.comp_fp_new[slot] = fpo + N;
    }
  }
  if (lane == 0) {
    tp_old[i] = tpo + P;
    fp_old[i] = fpo + N;
    atomicOr(u_bits + (i >> 6), 1ull << (i & 63));
    if (ex.u_words != nullptr) ex.u_words[i * ex.kw + (ex.factor_bit >> 6)] |= 1ull << (ex.factor_bit & 63);
    t_used += 1; t_p += P; t_n += N;
  }
}

__global__ void __launch_bounds__(256)
cover_apply_kernel(const uint64_t* __restrict__ xb, uint64_t* __restrict__ cb, int64_t m, int64_t n,
                   int64_t words, const uint64_t* __restrict__ basis, uint8_t* __restrict__ alive,
                   const int64_t* __restrict__ winner, int32_t* __restrict__ tp_old,
                   int32_t* __restrict__ fp_old, int wa, int wb, double neg_w_fp, double w_fn,
                   int8_t* __restrict__ rows_plane, int64_t ld, int covered_value, int pq_layout,
                   unsigned long long* __restrict__ u_bits, unsigned long long* __restrict__ totals,
                   const ApplyExtra ex) {
  const int64_t j = *winner;
  if (j < 0) return;
  const uint64_t* __restrict__ b = basis + j * words;
  const int lane = threadIdx.x & 31;
  if (ex.vt_row != nullptr && blockIdx.x == 0)
    for (int64_t q = threadIdx.x; q < words; q += blockDim.x) ex.vt_row[q] = b[q];
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t pairs = words >> 1;
  long long t_used = 0, t_p = 0, t_n = 0;
  for (int64_t i = warp0; i < m; i += nwarps) {
    int P = 0, N = 0;
    for (int64_t p = lane; p < pairs; p += 32) {
      const ulonglong2 x = ld_words2(xb + i * words + 2 * p);
      const ulonglong2 c = *reinterpret_cast<const ulonglong2*>(cb + i * words + 2 * p);
      const ulonglong2 v = ld_words2(b + 2 * p);
      P += __popcll(x.x & ~c.x & v.x) + __popcll(x.y & ~c.y & v.y);
      N += __popcll(~c.x & v.x) + __popcll(~c.y & v.y);                 // |v & ~c| (v has zero pad bits), minus P below
    }
    P = warp_sum(P);
    N = warp_sum(N) - P;
    const int tpo = tp_old[i], fpo = fp_old[i];
    if (!row_uses(wa, wb, neg_w_fp, w_fn, tpo, fpo, P, N)) continue;    // warp-uniform
    apply_used_row(xb, cb, n, words, b, tp_old, fp_old, rows_plane, ld, covered_value, pq_layout, u_bits, ex, i, lane, P, N,
                   tpo, fpo, t_used, t_p, t_n);
  }
  if (lane == 0 && t_used) {
    atomicAdd(totals + 0, (unsigned long long)t_used);
    atomicAdd(totals + 1, (unsigned long long)t_p);
    atomicAdd(totals + 2, (unsigned long long)t_n);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) alive[j] = 0;               // Asso.py:106-107
}

// Ring-fed form of cover_apply_kernel.  ncu on the register-fed kernel above at 480189 x 17770: 59 % of DRAM peak,
// 12 of 24 resident warps per scheduler waiting on global loads (80 registers cap the occupancy, a warp has two or three
// 128-bit loads in flight per row).  Here every warp streams ITS rows -- the x row and the cover row, 2 x words x 8 bytes --
// through a private ring of shared-memory slots filled by 1-D bulk copies (TMA engine, mbarrier complete_tx), the same
// protocol as confusion_panel_list_kernel: depth x 16 row pairs in flight per SM at no register cost.  The winner's basis row
// sits in shared memory.  Rows that use the winner (1-2 %) take apply_used_row, which works on global memory as before;
// the slot is re-armed first, so the copy engine never waits for an update.
constexpr int APPLY_RING_THREADS = 512;
constexpr int APPLY_RING_WARPS = APPLY_RING_THREADS / 32;
constexpr int APPLY_RING_DEPTH_MAX = 4;
__global__ void __launch_bounds__(APPLY_RING_THREADS, 1)
cover_apply_ring_kernel(const uint64_t* __restrict__ xb, uint64_t* __restrict__ cb, int64_t m, int64_t n,
                        int64_t words, const uint64_t* __restrict__ basis, uint8_t* __restrict__ alive,
                        const int64_t* __restrict__ winner, int32_t* __restrict__ tp_old,
                        int32_t* __restrict__ fp_old, int wa, int wb, double neg_w_fp, double w_fn,
                        int8_t* __restrict__ rows_plane, int64_t ld, int covered_value, int pq_layout,
                        unsigned long long* __restrict__ u_bits, unsigned long long* __restrict__ totals,
                        const ApplyExtra ex, int depth) {
  extern __shared__ __align__(128) uint8_t apply_smem[];
  const int64_t j = *winner;
  if (j < 0) return;
  const uint64_t* __restrict__ b = basis + j * words;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t pairs = words >> 1;
  const uint32_t row_bytes = (uint32_t)(words * 8);
  ulonglong2* bs = reinterpret_cast<ulonglong2*>(apply_smem);
  uint8_t* ring = apply_smem + row_bytes + (size_t)warp * depth * 2 * row_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(apply_smem + row_bytes + (size_t)APPLY_RING_WARPS * depth * 2 * row_bytes);
  const uint32_t bar0 = smem_u32(bars + warp * depth);
  const uint32_t ring0 = smem_u32(ring);
  if (lane == 0) {
    for (int s = 0; s < depth; ++s) mbar_init(bar0 + 8u * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int64_t q = threadIdx.x; q < pairs; q += blockDim.x) bs[q] = ld_words2(b + 2 * q);
  if (ex.vt_row != nullptr && blockIdx.x == 0)
    for (int64_t q = threadIdx.x; q < words; q += blockDim.x) ex.vt_row[q] = b[q];
  __syncthreads();

  const int64_t gw = (int64_t)blockIdx.x * APPLY_RING_WARPS + warp;
  const int64_t nwarps = (int64_t)gridDim.x * APPLY_RING_WARPS;
  const int64_t my_rows = gw < m ? (m - 1 - gw) / nwarps + 1 : 0;
  int64_t issued = 0;
  int iss_slot = 0;
  auto issue = [&]() {                                                 // lane 0: x row and cover row of this warp's next row
    const int64_t i = gw + issued * nwarps;
    const uint32_t bar = bar0 + 8u * iss_slot, dst = ring0 + (uint32_t)iss_slot * 2u * row_bytes;
    mbar_expect_tx(bar, 2u * row_bytes);
    bulk_load(dst, xb + i * words, row_bytes, bar);
    bulk_load(dst + row_bytes, cb + i * words, row_bytes, bar);
    iss_slot = iss_slot == depth - 1 ? 0 : iss_slot + 1;
    ++issued;
  };
  if (lane == 0)
    for (int d = 0; d < depth && issued < my_rows; ++d) issue();

  const bool general = (wa | wb) == 0;
  long long t_used = 0, t_p = 0, t_n = 0;
  int slot = 0;
  uint32_t phase = 0;
  for (int64_t t = 0; t < my_rows; ++t) {
    const int64_t i = gw + t * nwarps;
    int tpo = 0, fpo = 0;
    if (general) { tpo = tp_old[i]; fpo = fp_old[i]; }                  // the fp64 row test needs them; in flight during the wait
    const ulonglong2* xs = reinterpret_cast<const ulonglong2*>(ring + (size_t)slot * 2 * row_bytes);
    const ulonglong2* cs = reinterpret_cast<const ulonglong2*>(ring + (size_t)slot * 2 * row_bytes + row_bytes);
    mbar_wait(bar0 + 8u * slot, phase);
    int P = 0, N = 0;
    for (int64_t p = lane; p < pairs; p += 32) {
      const ulonglong2 x = xs[p], c = cs[p], v = bs[p];
      P += __popcll(x.x & ~c.x & v.x) + __popcll(x.y & ~c.y & v.y);
      N += __popcll(~c.x & v.x) + __popcll(~c.y & v.y);                 // |v & ~c| (v has zero pad bits), minus P below
    }
    __syncwarp();                                                       // every lane has read the slot
    if (lane == 0 && issued < my_rows) issue();
    if (++slot == depth) { slot = 0; phase ^= 1u; }
    P = warp_sum(P);
    N = warp_sum(N) - P;
    if (!row_uses(wa, wb, neg_w_fp, w_fn, tpo, fpo, P, N)) continue;    // warp-uniform
    if (!general) { tpo = tp_old[i]; fpo = fp_old[i]; }
    apply_used_row(xb, cb, n, words, b, tp_old, fp_old, rows_plane, ld, covered_value, pq_layout, u_bits, ex, i, lane, P, N,
                   tpo, fpo, t_used, t_p, t_n);
  }
  if (lane == 0 && t_used) {
    atomicAdd(totals + 0, (unsigned long long)t_used);
    atomicAdd(totals + 1, (unsigned long long)t_p);
    atomicAdd(totals + 2, (unsigned long long)t_n);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) alive[j] = 0;               // Asso.py:106-107
}
// ring slots per warp that fit next to the basis row; < 2 = use the register-fed kernel (very wide matrices)
static inline int apply_ring_depth(int64_t words) {
  const char* e = getenv("BMF_APPLY_RING");
  if (e != nullptr && e[0] == '0') return 0;
  const int64_t row_bytes = words * 8;
  int64_t depth = (224 * 1024 - row_bytes - APPLY_RING_WARPS * APPLY_RING_DEPTH_MAX * 8) / (APPLY_RING_WARPS * 2 * row_bytes);
  if (depth > APPLY_RING_DEPTH_MAX) depth = APPLY_RING_DEPTH_MAX;
  return (int)depth;
}

// =========================================================================================
// Boolean product and confusion counts.  One warp per row; a row's prediction is the OR of
// the V^T rows selected by the set bits of its k-bit usage word(s).
// =========================================================================================
// Four pair positions (p, p+32, p+64, p+96) of one row at once: the factor-selection bits are decoded
// once per group and the 4 x 128-bit loads per selected V^T row are independent, so every lane keeps
// several memory requests in flight (the single-pair form is latency bound: ~35-45 % of HBM).
constexpr int PU = 4;
__device__ __forceinline__ void product_quad(const uint64_t* __restrict__ uw, int64_t kw,
                                             const uint64_t* __restrict__ vt, int64_t words, int64_t p0,
                                             int64_t pairs, int64_t skip, ulonglong2 (&acc)[PU]) {
#pragma unroll
  for (int u = 0; u < PU; ++u) acc[u] = make_ulonglong2(0ull, 0ull);
  for (int64_t q = 0; q < kw; ++q) {
    uint64_t sel = uw[q];
    if (skip >= 0 && (skip >> 6) == q) sel &= ~(1ull << (skip & 63));
    while (sel) {
      const int l = __ffsll((long long)sel) - 1;
      sel &= sel - 1;
      const uint64_t* __restrict__ vrow = vt + (q * 64 + l) * words;
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int64_t p = p0 + 32 * u;
        if (p < pairs) {
          const ulonglong2 v = ld_words2(vrow + 2 * p);
          acc[u].x |= v.x;
          acc[u].y |= v.y;
        }
      }
    }
  }
}

// RESIDUAL (get_residual): x holds X with the layout of pd, and pd receives x AND NOT (the product).  The x pairs are
// loaded before the OR chain, so their latency overlaps the V^T reads; a row that uses no factor stores x unchanged.
template <bool RESIDUAL = false>
__global__ void __launch_bounds__(256)
bool_product_kernel(const uint64_t* __restrict__ u_words, int64_t m, int64_t kw,
                    const uint64_t* __restrict__ vt, int64_t words, const uint64_t* __restrict__ x,
                    uint64_t* __restrict__ pd) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t pairs = words >> 1;
  for (int64_t i = warp0; i < m; i += nwarps) {
    const uint64_t* uw = u_words + i * kw;
    for (int64_t p0 = lane; p0 < pairs; p0 += 32 * PU) {
      ulonglong2 xv[PU], acc[PU];
      if (RESIDUAL) {
#pragma unroll
        for (int u = 0; u < PU; ++u) {
          const int64_t p = p0 + 32 * u;
          xv[u] = p < pairs ? ld_words2(x + i * words + 2 * p) : make_ulonglong2(0ull, 0ull);
        }
      }
      product_quad(uw, kw, vt, words, p0, pairs, -1, acc);
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int64_t p = p0 + 32 * u;
        if (RESIDUAL) acc[u] = make_ulonglong2(xv[u].x & ~acc[u].x, xv[u].y & ~acc[u].y);
        if (p < pairs) __stcs(reinterpret_cast<ulonglong2*>(pd + i * words + 2 * p), acc[u]);   // 128-bit streaming store
      }
    }
  }
}

// Confusion counts.  Per word only TWO (three when |gt| is not known) popcounts are taken:
// TP = |gt & pd| and |pd| (FP = |pd| - TP); FN = |gt| - TP with |gt| either supplied by the caller
// (the number of stored ones, free on the host) or counted (COUNT_GT).  The integer (POPC/ALU) pipe is
// the busiest unit of this kernel, so the main loop runs without bounds checks on whole groups of
// 4 x 32 pairs with pointer increments, and a checked tail handles the last < 128 pairs of a row.
// ENTRIES (stored-entry counts, task='prediction'): gt holds the stored ones and zt (nullable) the explicitly stored
// zeros; counts[0..3] += (|gt & pd|, |zt & pd|, |gt|, |zt|) in the same single pass (COUNT_GT must be set).
template <bool FROM_FACTORS, bool COUNT_GT, bool ENTRIES = false>
__global__ void __launch_bounds__(256)
confusion_kernel(const uint64_t* __restrict__ gt, const uint64_t* __restrict__ zt, const uint64_t* __restrict__ pd_bits,
                 int64_t m, int64_t words, const uint64_t* __restrict__ u_words, int64_t kw,
                 const uint64_t* __restrict__ vt, unsigned long long* __restrict__ counts,
                 int32_t* __restrict__ row_tp, int32_t* __restrict__ row_fp) {
  static_assert(!ENTRIES || COUNT_GT, "stored-entry counts count |gt|");
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t pairs = words >> 1;
  const int64_t full = pairs / (32 * PU);                    // unchecked groups per row
  const bool has_z = ENTRIES && zt != nullptr;
  long long t_tp = 0, t_pd = 0, t_gt = 0, t_z = 0;
  for (int64_t i = warp0; i < m; i += nwarps) {
    int tp = 0, np = 0, ng = 0, nz = 0;
    const ulonglong2* gp = reinterpret_cast<const ulonglong2*>(gt + i * words) + lane;
    const ulonglong2* zp = has_z ? reinterpret_cast<const ulonglong2*>(zt + i * words) + lane : nullptr;
    const ulonglong2* dp = FROM_FACTORS ? nullptr : reinterpret_cast<const ulonglong2*>(pd_bits + i * words) + lane;
    const uint64_t* uw = FROM_FACTORS ? u_words + i * kw : nullptr;
    for (int64_t it = 0; it < full; ++it) {
      ulonglong2 g[PU], d[PU], z[PU];
#pragma unroll
      for (int u = 0; u < PU; ++u) g[u] = __ldcs(gp + 32 * u);
      if (has_z) {
#pragma unroll
        for (int u = 0; u < PU; ++u) z[u] = __ldcs(zp + 32 * u);
        zp += 32 * PU;
      }
      if (!FROM_FACTORS) {
#pragma unroll
        for (int u = 0; u < PU; ++u) d[u] = __ldcs(dp + 32 * u);
        dp += 32 * PU;
      } else {
#pragma unroll
        for (int u = 0; u < PU; ++u) d[u] = make_ulonglong2(0ull, 0ull);
        for (int64_t q = 0; q < kw; ++q) {
          uint64_t sel = uw[q];
          while (sel) {
            const int l = __ffsll((long long)sel) - 1;
            sel &= sel - 1;
            const ulonglong2* vp = reinterpret_cast<const ulonglong2*>(vt + (q * 64 + l) * words) + it * (32 * PU) + lane;
#pragma unroll
            for (int u = 0; u < PU; ++u) {
              const ulonglong2 v = __ldg(vp + 32 * u);
              d[u].x |= v.x;
              d[u].y |= v.y;
            }
          }
        }
      }
      gp += 32 * PU;
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        tp += __popcll(g[u].x & d[u].x) + __popcll(g[u].y & d[u].y);
        if (!ENTRIES) np += __popcll(d[u].x) + __popcll(d[u].y);
        if (COUNT_GT) ng += __popcll(g[u].x) + __popcll(g[u].y);
        if (has_z) {
          np += __popcll(z[u].x & d[u].x) + __popcll(z[u].y & d[u].y);
          nz += __popcll(z[u].x) + __popcll(z[u].y);
        }
      }
    }
    {                                                         // checked tail
      const int64_t p0 = full * (32 * PU) + lane;
      if (full * (32 * PU) < pairs) {
        ulonglong2 g[PU], d[PU], z[PU];
#pragma unroll
        for (int u = 0; u < PU; ++u) {
          const int64_t p = p0 + 32 * u;
          g[u] = make_ulonglong2(0ull, 0ull);
          d[u] = make_ulonglong2(0ull, 0ull);
          z[u] = make_ulonglong2(0ull, 0ull);
          if (p < pairs) {
            g[u] = __ldcs(reinterpret_cast<const ulonglong2*>(gt + i * words + 2 * p));
            if (has_z) z[u] = __ldcs(reinterpret_cast<const ulonglong2*>(zt + i * words + 2 * p));
            if (!FROM_FACTORS) d[u] = __ldcs(reinterpret_cast<const ulonglong2*>(pd_bits + i * words + 2 * p));
          }
        }
        if (FROM_FACTORS) product_quad(uw, kw, vt, words, p0, pairs, -1, d);
#pragma unroll
        for (int u = 0; u < PU; ++u) {
          tp += __popcll(g[u].x & d[u].x) + __popcll(g[u].y & d[u].y);
          if (!ENTRIES) np += __popcll(d[u].x) + __popcll(d[u].y);
          if (COUNT_GT) ng += __popcll(g[u].x) + __popcll(g[u].y);
          if (has_z) {
            np += __popcll(z[u].x & d[u].x) + __popcll(z[u].y & d[u].y);
            nz += __popcll(z[u].x) + __popcll(z[u].y);
          }
        }
      }
    }
    tp = warp_sum(tp);
    np = warp_sum(np);
    if (COUNT_GT) ng = warp_sum(ng);
    if (has_z) nz = warp_sum(nz);
    if (lane == 0) {
      if (row_tp != nullptr) row_tp[i] = tp;
      if (row_fp != nullptr) row_fp[i] = np - tp;
      t_tp += tp; t_pd += np; t_gt += ng; t_z += nz;
    }
  }
  if (lane == 0 && (t_pd | t_gt)) {
    atomicAdd(counts + 0, (unsigned long long)t_tp);
    atomicAdd(counts + 1, (unsigned long long)t_pd);
    if (COUNT_GT) atomicAdd(counts + 2, (unsigned long long)t_gt);
  }
  if (ENTRIES && lane == 0 && t_z) atomicAdd(counts + 3, (unsigned long long)t_z);
}

// =========================================================================================
// Column-panel variants of the Boolean product and of the confusion counts from factors.
//
// ncu on the row-stream kernels above at m = 1M, n = 100k, k = 64 (profiles/r01_c5_*): the V^T rows a
// data row selects are re-fetched from L2 (2.5x the HBM bytes through L1) and the XU pipe (POPC) is
// 68 % busy at 52 % of HBM peak, i.e. four POPCs per 64-bit word cap the kernel near 5 TB/s.
// Here a CTA owns a panel of one or two chunks of 256 bit-words (2 KB per row and chunk) of ALL k <= 64
// rows of V^T in shared memory; its warps stream their data rows through the panel, so
//  * V^T is read from L2 once per CTA, the selected rows are ORed from shared memory (conflict free:
//    a warp reads 512 contiguous bytes), and HBM only carries the ground truth / the product;
//  * set bits are counted with a Harley-Seal carry-save adder tree (LOP3 on the ALU pipe): 16 words
//    cost 15 CSAs and ONE popcount instead of 16, which takes the XU pipe out of the picture
//    (HarleySeal8 below folds the 8 words a lane holds per row and pairs two rows per popcount).
// =========================================================================================
constexpr int CH_PAIRS = 128;            // 16-byte pairs per chunk and row: 32 lanes x 4
constexpr int PANEL_THREADS = 512;

__device__ __forceinline__ void csa64(uint64_t& h, uint64_t& l, uint64_t a, uint64_t b, uint64_t c) {
  const uint64_t u = a ^ b;
  h = (a & b) | (u & c);                 // majority -> one LOP3 per 32-bit half
  l = u ^ c;                             // parity   -> one LOP3 per 32-bit half
}
// V^T panel -> shared memory: Vs[l][p] (pairs), zero beyond the matrix
__device__ __forceinline__ void load_vt_panel(ulonglong2* Vs, const uint64_t* __restrict__ vt, int64_t k,
                                              int64_t words, int64_t pair0, int panel_pairs, int valid_pairs) {
  const int total = (int)k * panel_pairs;
  for (int e = threadIdx.x; e < total; e += blockDim.x) {
    const int l = e / panel_pairs, p = e - l * panel_pairs;
    Vs[e] = p < valid_pairs ? ld_words2(vt + (int64_t)l * words + 2 * (pair0 + p)) : make_ulonglong2(0ull, 0ull);
  }
  __syncthreads();
}

// OR of the V^T rows selected by ONE usage word (k <= 64) at the lane's four pair slots
__device__ __forceinline__ void panel_or1(const ulonglong2* Vs, int panel_pairs, uint64_t sel, int slot0,
                                          ulonglong2 (&d)[4]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) d[u] = make_ulonglong2(0ull, 0ull);
  while (sel) {
    const int l = __ffsll((long long)sel) - 1;
    sel &= sel - 1;
    const ulonglong2* vr = Vs + l * panel_pairs + slot0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const ulonglong2 v = vr[32 * u];
      d[u].x |= v.x;
      d[u].y |= v.y;
    }
  }
}

// Confusion counts from factors, k <= 64.  CTA (panel, split), 16 warps.  Every warp streams ITS rows (blocks of
// 32 consecutive rows, usage words fetched with one coalesced load per block and broadcast by shuffle) through a
// PRIVATE ring of RING_DEPTH (3 at k = 64, up to 8) shared-memory slots filled by 1-D bulk copies (TMA engine, mbarrier complete_tx):
// lane 0 re-issues the copy for row idx + RING_DEPTH as soon as row idx has been consumed, so 16 x RING_DEPTH row
// segments (2 KB each) are in flight per SM at no register cost -- what it takes to cover HBM latency at 6-7 TB/s.
// Producer and consumer of a slot are the same warp, so one "full" barrier per slot is the whole protocol.
constexpr int RING_DEPTH_MAX = 8;       // slots per warp: as many as shared memory allows next to the V^T panel
constexpr int PANEL_WARPS = PANEL_THREADS / 32;

// half a Harley-Seal block: 8 words -> one "eights" carry; two of them make a "sixteens" word
struct HarleySeal8 {
  uint64_t ones = 0, twos = 0, fours = 0, eights = 0, pend = 0;
  long long sixteens = 0;
  __device__ __forceinline__ uint64_t fold8(const uint64_t (&w)[8]) {
    uint64_t t2a, t2b, t4a, t4b, t8;
    csa64(t2a, ones, ones, w[0], w[1]);
    csa64(t2b, ones, ones, w[2], w[3]);
    csa64(t4a, twos, twos, t2a, t2b);
    csa64(t2a, ones, ones, w[4], w[5]);
    csa64(t2b, ones, ones, w[6], w[7]);
    csa64(t4b, twos, twos, t2a, t2b);
    csa64(t8, fours, fours, t4a, t4b);
    return t8;
  }
  __device__ __forceinline__ void add8_first(const uint64_t (&w)[8]) { pend = fold8(w); }
  __device__ __forceinline__ void add8_second(const uint64_t (&w)[8]) {
    uint64_t t16;
    const uint64_t t8 = fold8(w);
    csa64(t16, eights, eights, pend, t8);
    pend = 0;
    sixteens += __popcll(t16);
  }
  __device__ __forceinline__ long long total() const {
    return 16 * sixteens + 8 * (long long)(__popcll(eights) + __popcll(pend)) + 4 * (long long)__popcll(fours) +
           2 * (long long)__popcll(twos) + (long long)__popcll(ones);
  }
};

__device__ __forceinline__ ulonglong2 or2(const ulonglong2 a, const ulonglong2 b) {
  return make_ulonglong2(a.x | b.x, a.y | b.y);
}
__device__ __forceinline__ ulonglong2 or3(const ulonglong2 a, const ulonglong2 b, const ulonglong2 c) {
  return make_ulonglong2(a.x | b.x | c.x, a.y | b.y | c.y);
}

// d = OR of the V^T rows selected by `sel` (warp-uniform) at the lane's four pair slots; the common cases of one and
// two selected rows are straight-line code (sel comes from a shuffle, so the branch never diverges).
// SEED: d enters with a value and the rows are ORed into it.
template <bool SEED = false>
__device__ __forceinline__ void panel_or_fast(const ulonglong2* Vs, int panel_pairs, uint64_t sel, int slot0,
                                              ulonglong2 (&d)[4]) {
  if (sel == 0) {
    if (!SEED) {
#pragma unroll
      for (int u = 0; u < 4; ++u) d[u] = make_ulonglong2(0ull, 0ull);
    }
    return;
  }
  const int l0 = __ffsll((long long)sel) - 1;
  sel &= sel - 1;
  const ulonglong2* v0 = Vs + l0 * panel_pairs + slot0;
#pragma unroll
  for (int u = 0; u < 4; ++u) d[u] = SEED ? or2(d[u], v0[32 * u]) : v0[32 * u];
  while (sel) {
    const int l = __ffsll((long long)sel) - 1;
    sel &= sel - 1;
    const ulonglong2* vr = Vs + l * panel_pairs + slot0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const ulonglong2 v = vr[32 * u];
      d[u].x |= v.x;
      d[u].y |= v.y;
    }
  }
}

// ---- selection lists ---------------------------------------------------------------------------------
// Scanning a usage word bit by bit (ffs, clear lowest bit, address) costs ~15 integer instructions per selected V^T row
// on the ALU pipe, which is what bounds the panel kernels (ncu: ALU 74 %, DRAM 62 %).  The scan is therefore done ONCE
// per row by the lane that loaded the word -- 32 rows in parallel -- into a packed list: the indices of the set bits in
// bytes 0..6, their number in byte 7 (0xff = more than seven: the row takes the bit-scan path).  The row loop then
// broadcasts the list and runs straight-line code: all selected rows are loaded before the first OR (independent
// shared-memory loads instead of a load -> OR -> load chain) and three rows are combined per LOP3.
__device__ __forceinline__ uint64_t pack_selection(uint64_t u) {
  const int c = __popcll(u);
  if (c > 7) return ~0ull;
  uint64_t p = (uint64_t)c << 56;
  for (int s = 0; u != 0; s += 8) {
    p |= (uint64_t)(__ffsll((long long)u) - 1) << s;
    u &= u - 1;
  }
  return p;
}
// d = OR of the cnt (1..7) V^T rows named by the list bytes (lo = bytes 0..3, hi = bytes 4..6), at the lane's four pair
// slots; SEED: d enters with a value and the rows are ORed into it
template <bool SEED = false>
__device__ __forceinline__ void panel_or_list(const ulonglong2* Vs, int panel_pairs, uint32_t lo, uint32_t hi, int cnt,
                                              int slot0, ulonglong2 (&d)[4]) {
  const ulonglong2* base = Vs + slot0;
  const ulonglong2* r0 = base + __byte_perm(lo, 0u, 0x4440u) * panel_pairs;
  if (cnt == 1) {
#pragma unroll
    for (int u = 0; u < 4; ++u) d[u] = SEED ? or2(d[u], r0[32 * u]) : r0[32 * u];
    return;
  }
  const ulonglong2* r1 = base + __byte_perm(lo, 0u, 0x4441u) * panel_pairs;
  if (cnt == 2) {
#pragma unroll
    for (int u = 0; u < 4; ++u) d[u] = SEED ? or3(d[u], r0[32 * u], r1[32 * u]) : or2(r0[32 * u], r1[32 * u]);
    return;
  }
  const ulonglong2* r2 = base + __byte_perm(lo, 0u, 0x4442u) * panel_pairs;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    d[u] = SEED ? or2(d[u], or3(r0[32 * u], r1[32 * u], r2[32 * u])) : or3(r0[32 * u], r1[32 * u], r2[32 * u]);
  if (cnt == 3) return;
  const ulonglong2* r3 = base + (lo >> 24) * panel_pairs;
  if (cnt == 4) {
#pragma unroll
    for (int u = 0; u < 4; ++u) d[u] = or2(d[u], r3[32 * u]);
    return;
  }
  const ulonglong2* r4 = base + __byte_perm(hi, 0u, 0x4440u) * panel_pairs;
#pragma unroll
  for (int u = 0; u < 4; ++u) d[u] = or3(d[u], r3[32 * u], r4[32 * u]);
  if (cnt == 5) return;
  const ulonglong2* r5 = base + __byte_perm(hi, 0u, 0x4441u) * panel_pairs;
  if (cnt == 6) {
#pragma unroll
    for (int u = 0; u < 4; ++u) d[u] = or2(d[u], r5[32 * u]);
    return;
  }
  const ulonglong2* r6 = base + __byte_perm(hi, 0u, 0x4442u) * panel_pairs;
#pragma unroll
  for (int u = 0; u < 4; ++u) d[u] = or3(d[u], r5[32 * u], r6[32 * u]);
}
// |V^T row l| inside this CTA's column panel, l < k: the prediction of a data row that uses ONE factor has exactly that
// many ones, so such rows (27 % at two factors per row on average) need no popcount of the prediction at all
__device__ __forceinline__ void panel_row_counts(const ulonglong2* Vs, int panel_pairs, int k, int* pop_v) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int l = warp; l < k; l += nw) {
    int c = 0;
    for (int p = lane; p < panel_pairs; p += 32) c += __popcll(Vs[l * panel_pairs + p].x) + __popcll(Vs[l * panel_pairs + p].y);
    c = warp_sum(c);
    if (lane == 0) pop_v[l] = c;
  }
  __syncthreads();
}

// four words -> one "fours" carry; two of them make an "eights" word (the half-width tree of count mode 3)
struct HarleySeal4 {
  uint64_t ones = 0, twos = 0, fours = 0, pend = 0;
  int eights = 0;
  __device__ __forceinline__ uint64_t fold4(uint64_t a, uint64_t b, uint64_t c, uint64_t d) {
    uint64_t t2a, t2b, t4;
    csa64(t2a, ones, ones, a, b);
    csa64(t2b, ones, ones, c, d);
    csa64(t4, twos, twos, t2a, t2b);
    return t4;
  }
  __device__ __forceinline__ void add4(bool second, uint64_t a, uint64_t b, uint64_t c, uint64_t d) {
    const uint64_t t4 = fold4(a, b, c, d);
    if (!second) { pend = t4; return; }
    uint64_t t8;
    csa64(t8, fours, fours, pend, t4);
    pend = 0;
    eights += __popcll(t8);
  }
  __device__ __forceinline__ long long total() const {
    return 8 * (long long)eights + 4 * (long long)(__popcll(fours) + __popcll(pend)) + 2 * (long long)__popcll(twos) +
           (long long)__popcll(ones);
  }
};

// CTA -> (column panel, row split) for the panel kernels.  A row is ceil(pairs / panel_pairs) panels wide; cutting it into
// panels of the FULL width leaves a narrow last one (n = 100 000 bits: six 2 KB panels and one of 224 bytes) whose CTAs
// spend the same per-row instruction overhead on a ninth of the bytes -- 21 of 147 SMs moved 1.8 % of the data.  The row
// is therefore cut into panels of EQUAL width (782 pairs -> 7 x 112): every CTA carries the same useful bytes per row.
struct PanelGrid {
  int panels;           // column panels per row
  int splits;           // row splits (CTAs) per panel
  int width_pairs;      // pairs per panel (<= the shared-memory panel width)
};
__device__ __forceinline__ void panel_coords(const PanelGrid& g, int& panel, int& split, int& nsplit) {
  const int b = (int)blockIdx.x;
  split = b / g.panels;                                    // panel fastest: neighbouring CTAs write neighbouring columns
  panel = b - split * g.panels;
  nsplit = g.splits;
}

// Row order (ROWMAP): 0 = every warp owns blocks of 32 CONSECUTIVE rows (one coalesced load of the usage words);
// 1 = interleaved: a CTA owns super-blocks of 32 x (#warps) rows and at any moment its warps work on CONSECUTIVE rows
// (warp w takes rows base + r * #warps + w), so the 2 KB segments the CTAs of one row range write (or read) at the same
// time tile a contiguous stretch of memory the way a memset does, instead of 32 x #CTAs scattered rows.
__device__ __forceinline__ int64_t panel_row(int rowmap, int64_t block, int r, int warp, int nw) {
  return rowmap ? (block * nw * 32 + (int64_t)r * nw + warp) : (block * 32 + r);
}

// MODE: how the two counts |gt & pd| and |pd| are taken -- 0: both through the carry-save tree (ALU pipe, LOP3),
// 1: |gt & pd| through the tree and |pd| through POPC (XU pipe), 2: both through POPC.
template <bool COUNT_GT, int MODE>
__global__ void __launch_bounds__(PANEL_THREADS, 1)
confusion_panel_kernel(const uint64_t* __restrict__ gt, int64_t m, int64_t words,
                       const uint64_t* __restrict__ u_words, const uint64_t* __restrict__ vt, int64_t k,
                       int panel_chunks, int RING_DEPTH, const PanelGrid pg, unsigned long long* __restrict__ counts) {
  extern __shared__ __align__(128) uint8_t panel_smem[];
  const int panel_pairs = panel_chunks * CH_PAIRS;
  const int row_bytes = panel_pairs * 16;
  int pg_panel, pg_split, pg_nsplit;
  panel_coords(pg, pg_panel, pg_split, pg_nsplit);
  ulonglong2* Vs = reinterpret_cast<ulonglong2*>(panel_smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* ring = panel_smem + (size_t)k * row_bytes + (size_t)warp * RING_DEPTH * row_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(panel_smem + (size_t)(k + PANEL_WARPS * RING_DEPTH) * row_bytes);
  const uint32_t bar0 = smem_u32(bars + warp * RING_DEPTH);
  const uint32_t ring0 = smem_u32(ring);

  const int64_t pairs = words >> 1;
  const int64_t pair0 = (int64_t)pg_panel * pg.width_pairs;
  const int valid_pairs = (int)((pairs - pair0) < pg.width_pairs ? (pairs - pair0) : pg.width_pairs);
  const uint32_t seg_bytes = (uint32_t)valid_pairs * 16u;
  const int nch = (valid_pairs + CH_PAIRS - 1) / CH_PAIRS;  // chunks this panel really has
  if (lane == 0) {
    for (int s = 0; s < RING_DEPTH; ++s) mbar_init(bar0 + 8u * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // the bulk copies only ever write seg_bytes per slot: zero the slots once and their tails stay zero, so the
  // consumer needs no column predicates
  for (int e = lane; e < RING_DEPTH * panel_pairs; e += 32)
    reinterpret_cast<ulonglong2*>(ring)[e] = make_ulonglong2(0ull, 0ull);
  fence_proxy_async();
  load_vt_panel(Vs, vt, k, words, pair0, panel_pairs, valid_pairs);     // ends with __syncthreads()

  // this warp's rows: 32-row blocks gw, gw + nwarps, ...
  const int64_t gw = (int64_t)pg_split * PANEL_WARPS + warp;
  const int64_t nwarps = (int64_t)pg_nsplit * PANEL_WARPS;
  const int64_t blocks_total = (m + 31) >> 5;
  int my_blocks = 0, last_rows = 0;
  if (gw < blocks_total) {
    my_blocks = (int)((blocks_total - 1 - gw) / nwarps) + 1;
    const int64_t last_block = gw + (int64_t)(my_blocks - 1) * nwarps;
    last_rows = (int)((m - last_block * 32) < 32 ? (m - last_block * 32) : 32);
  }
  int to_issue = my_blocks > 0 ? (my_blocks - 1) * 32 + last_rows : 0;    // rows not yet requested
  // issue side (meaningful in lane 0): next row segment to request, as an incrementally updated pointer
  const uint64_t* iss_ptr = gt + 2 * pair0 + gw * 32 * words;
  const int64_t step_block = (nwarps * 32 - 31) * words;
  int iss_r = 0, iss_slot = 0;
  auto issue = [&]() {
    mbar_expect_tx(bar0 + 8u * iss_slot, seg_bytes);
    bulk_load(ring0 + (uint32_t)(iss_slot * row_bytes), iss_ptr, seg_bytes, bar0 + 8u * iss_slot);
    iss_slot = iss_slot == RING_DEPTH - 1 ? 0 : iss_slot + 1;
    if (++iss_r == 32) { iss_r = 0; iss_ptr += step_block; } else { iss_ptr += words; }
    --to_issue;
  };
  if (lane == 0)
    for (int d = 0; d < RING_DEPTH && to_issue > 0; ++d) issue();

  HarleySeal8 hs_tp, hs_pd, hs_gt;
  long long n_pd = 0, n_tp = 0;
  int slot = 0;
  uint32_t phase = 0;
  bool second = false;
  const uint64_t* u_ptr = u_words + gw * 32 + lane;
  uint64_t u_next = (my_blocks > 0 && gw * 32 + lane < m) ? __ldg(u_ptr) : 0ull;
  for (int blk = 0; blk < my_blocks; ++blk) {
    const uint64_t u_cur = u_next;
    u_ptr += nwarps * 32;
    u_next = (blk + 1 < my_blocks && (gw + (int64_t)(blk + 1) * nwarps) * 32 + lane < m) ? __ldg(u_ptr) : 0ull;
    const int nrows = blk + 1 < my_blocks ? 32 : last_rows;
    for (int r = 0; r < nrows; ++r) {
      const uint64_t sel = __shfl_sync(0xffffffffu, u_cur, r);
      const ulonglong2* seg = reinterpret_cast<const ulonglong2*>(ring + (size_t)slot * row_bytes);
      mbar_wait(bar0 + 8u * slot, phase);
      for (int c = 0; c < nch; ++c) {
        const int slot0 = c * CH_PAIRS + lane;
        ulonglong2 g[4], d[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) g[u] = seg[slot0 + 32 * u];
        panel_or_fast(Vs, panel_pairs, sel, slot0, d);
        uint64_t w[8];
#pragma unroll
        for (int u = 0; u < 4; ++u) { w[2 * u] = g[u].x & d[u].x; w[2 * u + 1] = g[u].y & d[u].y; }
        if (MODE == 2) {
#pragma unroll
          for (int u = 0; u < 8; ++u) n_tp += __popcll(w[u]);
        } else {
          if (!second) hs_tp.add8_first(w); else hs_tp.add8_second(w);
        }
        if (MODE == 0) {
#pragma unroll
          for (int u = 0; u < 4; ++u) { w[2 * u] = d[u].x; w[2 * u + 1] = d[u].y; }
          if (!second) hs_pd.add8_first(w); else hs_pd.add8_second(w);
        } else {
#pragma unroll
          for (int u = 0; u < 4; ++u) n_pd += __popcll(d[u].x) + __popcll(d[u].y);
        }
        if (COUNT_GT) {
#pragma unroll
          for (int u = 0; u < 4; ++u) { w[2 * u] = g[u].x; w[2 * u + 1] = g[u].y; }
          if (!second) hs_gt.add8_first(w); else hs_gt.add8_second(w);
        }
        second = !second;
      }
      __syncwarp();                                         // every lane has consumed the slot
      if (lane == 0 && to_issue > 0) issue();               // refill it with the row RING_DEPTH ahead (a converged-warp
                                                            // elect_one issue was measured: no change, 2.352 vs 2.334 ms)
      if (++slot == RING_DEPTH) { slot = 0; phase ^= 1u; }
    }
  }
  const long long t_tp = warp_sum_ll(MODE == 2 ? n_tp : hs_tp.total());
  const long long t_pd = warp_sum_ll(MODE == 0 ? hs_pd.total() : n_pd);
  const long long t_gt = COUNT_GT ? warp_sum_ll(hs_gt.total()) : 0;
  if (lane == 0 && (t_pd | t_gt)) {
    atomicAdd(counts + 0, (unsigned long long)t_tp);
    atomicAdd(counts + 1, (unsigned long long)t_pd);
    if (COUNT_GT) atomicAdd(counts + 2, (unsigned long long)t_gt);
  }
}

// Boolean product, k <= 64: a warp owns 32 consecutive rows per pass, fetches their usage words with ONE
// coalesced load (the next block's is prefetched) and broadcasts them by shuffle, so no global load sits on the
// critical path of a row; 1024 threads keep enough 128-bit streaming stores in flight.
constexpr int PRODUCT_THREADS = 1024;
__global__ void __launch_bounds__(PRODUCT_THREADS, 1)
bool_product_panel_kernel(const uint64_t* __restrict__ u_words, int64_t m, const uint64_t* __restrict__ vt,
                          int64_t k, int64_t words, int panel_chunks, int rowmap, int store_mode, const PanelGrid pg,
                          uint64_t* __restrict__ pd) {
  extern __shared__ __align__(128) uint8_t panel_smem[];
  ulonglong2* Vs = reinterpret_cast<ulonglong2*>(panel_smem);
  const int panel_pairs = panel_chunks * CH_PAIRS;
  const int64_t pairs = words >> 1;
  int pg_panel, pg_split, pg_nsplit;
  panel_coords(pg, pg_panel, pg_split, pg_nsplit);
  const int64_t pair0 = (int64_t)pg_panel * pg.width_pairs;
  const int valid_pairs = (int)((pairs - pair0) < pg.width_pairs ? (pairs - pair0) : pg.width_pairs);
  load_vt_panel(Vs, vt, k, words, pair0, panel_pairs, valid_pairs);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // block index space: rowmap 0 -> 32-row blocks, one per warp and pass; rowmap 1 -> super-blocks, one per CTA and pass
  const int64_t blk0 = rowmap ? (int64_t)pg_split : (int64_t)pg_split * nw + warp;
  const int64_t blk_step = rowmap ? (int64_t)pg_nsplit : (int64_t)pg_nsplit * nw;
  const int64_t blk_rows = rowmap ? (int64_t)nw * 32 : 32;
  auto my_row = [&](int64_t blk) { return panel_row(rowmap, blk, lane, warp, nw); };
  int64_t ri = my_row(blk0);
  uint64_t mine = (blk0 * blk_rows < m && ri < m) ? __ldg(u_words + ri) : 0ull;
  for (int64_t blk = blk0; blk * blk_rows < m; blk += blk_step) {
    const uint64_t cur = mine;
    const int64_t nxt = blk + blk_step;
    ri = my_row(nxt);
    mine = (nxt * blk_rows < m && ri < m) ? __ldg(u_words + ri) : 0ull;
    for (int r = 0; r < 32; ++r) {
      const int64_t row = panel_row(rowmap, blk, r, warp, nw);
      if (row >= m) break;
      const uint64_t sel = __shfl_sync(0xffffffffu, cur, r);
      uint64_t* out = pd + row * words;
      for (int c = 0; c < panel_chunks; ++c) {
        const int slot0 = c * CH_PAIRS + lane;
        if (c * CH_PAIRS >= valid_pairs) break;
        ulonglong2 d[4];
        panel_or1(Vs, panel_pairs, sel, slot0, d);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int64_t gp = pair0 + slot0 + 32 * u;
          if (slot0 + 32 * u < valid_pairs) {
            ulonglong2* dst = reinterpret_cast<ulonglong2*>(out) + gp;
            if (store_mode == 0) __stcs(dst, d[u]);
            else if (store_mode == 1) *dst = d[u];
            else __stwt(dst, d[u]);
          }
        }
      }
    }
  }
}

// The selection-list forms of the two panel kernels (see pack_selection above): same grid, same ring, same results.
// ENTRIES (stored-entry counts, task='prediction'): gt holds the stored ones and zt (nullable) the explicitly stored
// zeros, counts[0..3] += (|gt & pd|, |zt & pd|, |gt|, |zt|), the product computed once for both.  A row's zeros segment
// takes the ring slot after its ones segment (RING_DEPTH >= 2), so the bytes in flight per warp are those of the plain
// form.  COUNT_GT must be set; MODE applies to |gt & pd|, and |zt & pd| goes through POPC.
template <bool COUNT_GT, int MODE, bool ENTRIES = false>
__global__ void __launch_bounds__(PANEL_THREADS, 1)
confusion_panel_list_kernel(const uint64_t* __restrict__ gt, const uint64_t* __restrict__ zt, int64_t m, int64_t words,
                            const uint64_t* __restrict__ u_words, const uint64_t* __restrict__ vt, int64_t k,
                            int panel_chunks, int RING_DEPTH, const PanelGrid pg, unsigned long long* __restrict__ counts) {
  static_assert(!ENTRIES || COUNT_GT, "stored-entry counts count |gt|");
  const bool has_z = ENTRIES && zt != nullptr;
  const int segs = has_z ? 2 : 1;                                 // ring slots per row
  extern __shared__ __align__(128) uint8_t panel_smem[];
  const int panel_pairs = panel_chunks * CH_PAIRS;
  const int row_bytes = panel_pairs * 16;
  int pg_panel, pg_split, pg_nsplit;
  panel_coords(pg, pg_panel, pg_split, pg_nsplit);
  ulonglong2* Vs = reinterpret_cast<ulonglong2*>(panel_smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t* ring = panel_smem + (size_t)k * row_bytes + (size_t)warp * RING_DEPTH * row_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(panel_smem + (size_t)(k + PANEL_WARPS * RING_DEPTH) * row_bytes);
  int* pop_v = reinterpret_cast<int*>(bars + PANEL_WARPS * RING_DEPTH_MAX);
  const uint32_t bar0 = smem_u32(bars + warp * RING_DEPTH);
  const uint32_t ring0 = smem_u32(ring);

  const int64_t pairs = words >> 1;
  const int64_t pair0 = (int64_t)pg_panel * pg.width_pairs;
  const int valid_pairs = (int)((pairs - pair0) < pg.width_pairs ? (pairs - pair0) : pg.width_pairs);
  const uint32_t seg_bytes = (uint32_t)valid_pairs * 16u;
  const int nch = (valid_pairs + CH_PAIRS - 1) / CH_PAIRS;
  if (lane == 0) {
    for (int s = 0; s < RING_DEPTH; ++s) mbar_init(bar0 + 8u * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int e = lane; e < RING_DEPTH * panel_pairs; e += 32)       // slot tails stay zero: no column predicates below
    reinterpret_cast<ulonglong2*>(ring)[e] = make_ulonglong2(0ull, 0ull);
  fence_proxy_async();
  load_vt_panel(Vs, vt, k, words, pair0, panel_pairs, valid_pairs);
  panel_row_counts(Vs, panel_pairs, (int)k, pop_v);

  const int64_t gw = (int64_t)pg_split * PANEL_WARPS + warp;
  const int64_t nwarps = (int64_t)pg_nsplit * PANEL_WARPS;
  const int64_t blocks_total = (m + 31) >> 5;
  int my_blocks = 0, last_rows = 0;
  if (gw < blocks_total) {
    my_blocks = (int)((blocks_total - 1 - gw) / nwarps) + 1;
    const int64_t last_block = gw + (int64_t)(my_blocks - 1) * nwarps;
    last_rows = (int)((m - last_block * 32) < 32 ? (m - last_block * 32) : 32);
  }
  int to_issue = my_blocks > 0 ? ((my_blocks - 1) * 32 + last_rows) * segs : 0;   // segments not yet requested
  const uint64_t* iss_ptr = gt + 2 * pair0 + gw * 32 * words;
  const int64_t step_block = (nwarps * 32 - 31) * words;
  int iss_r = 0, iss_slot = 0;
  bool iss_z = false;                                              // next segment is the zeros half of the row
  auto issue = [&]() {
    const uint64_t* src = (ENTRIES && iss_z) ? zt + (iss_ptr - gt) : iss_ptr;
    mbar_expect_tx(bar0 + 8u * iss_slot, seg_bytes);
    bulk_load(ring0 + (uint32_t)(iss_slot * row_bytes), src, seg_bytes, bar0 + 8u * iss_slot);
    iss_slot = iss_slot == RING_DEPTH - 1 ? 0 : iss_slot + 1;
    --to_issue;
    if (ENTRIES && has_z && !iss_z) { iss_z = true; return; }
    iss_z = false;
    if (++iss_r == 32) { iss_r = 0; iss_ptr += step_block; } else { iss_ptr += words; }
  };
  if (lane == 0)
    for (int d = 0; d < RING_DEPTH && to_issue > 0; ++d) issue();

  HarleySeal8 hs_tp, hs_pd, hs_gt, hs_z;
  HarleySeal4 h4_tp;
  bool sec_tp = false, sec_pd = false, sec_gt = false, sec_z = false;
  long long n_pd = 0, n_tp = 0;
  int slot = 0;
  uint32_t phase = 0;
  const uint64_t kmask = k >= 64 ? ~0ull : ((1ull << k) - 1ull);
  const uint64_t* u_ptr = u_words + gw * 32 + lane;
  uint64_t u_next = (my_blocks > 0 && gw * 32 + lane < m) ? __ldg(u_ptr) : 0ull;
  for (int blk = 0; blk < my_blocks; ++blk) {
    const uint64_t u_cur = u_next & kmask;
    u_ptr += nwarps * 32;
    u_next = (blk + 1 < my_blocks && (gw + (int64_t)(blk + 1) * nwarps) * 32 + lane < m) ? __ldg(u_ptr) : 0ull;
    const uint64_t list = pack_selection(u_cur);                 // this lane's row, scanned once
    const uint32_t list_lo = (uint32_t)list, list_hi = (uint32_t)(list >> 32);
    int blk_pd = (!ENTRIES && (list_hi >> 24) == 1u) ? pop_v[list_lo & 0xffu] : 0, blk_tp = 0;
    const int nrows = blk + 1 < my_blocks ? 32 : last_rows;
    for (int r = 0; r < nrows; ++r) {
      const uint32_t lo = __shfl_sync(0xffffffffu, list_lo, r);
      const uint32_t hi = __shfl_sync(0xffffffffu, list_hi, r);
      const int cnt = (int)(hi >> 24);
      const ulonglong2* seg = reinterpret_cast<const ulonglong2*>(ring + (size_t)slot * row_bytes);
      mbar_wait(bar0 + 8u * slot, phase);
      const ulonglong2* zseg = nullptr;
      if (has_z) {                                               // the zeros half sits in the next slot
        if (++slot == RING_DEPTH) { slot = 0; phase ^= 1u; }
        zseg = reinterpret_cast<const ulonglong2*>(ring + (size_t)slot * row_bytes);
        mbar_wait(bar0 + 8u * slot, phase);
      }
      if (COUNT_GT || cnt != 0) {                                // a row that uses no factor predicts nothing
        for (int c = 0; c < nch; ++c) {
          const int slot0 = c * CH_PAIRS + lane;
          ulonglong2 g[4], d[4], z[4];
          uint64_t w[8];
#pragma unroll
          for (int u = 0; u < 4; ++u) g[u] = seg[slot0 + 32 * u];
          if (COUNT_GT) {
#pragma unroll
            for (int u = 0; u < 4; ++u) { w[2 * u] = g[u].x; w[2 * u + 1] = g[u].y; }
            if (!sec_gt) hs_gt.add8_first(w); else hs_gt.add8_second(w);
            sec_gt = !sec_gt;
          }
          if (has_z) {
#pragma unroll
            for (int u = 0; u < 4; ++u) { z[u] = zseg[slot0 + 32 * u]; w[2 * u] = z[u].x; w[2 * u + 1] = z[u].y; }
            if (!sec_z) hs_z.add8_first(w); else hs_z.add8_second(w);
            sec_z = !sec_z;
          }
          if (cnt != 0) {
            if (cnt <= 7) {
              panel_or_list(Vs, panel_pairs, lo, hi, cnt, slot0, d);
            } else {
              const uint64_t sel = ((uint64_t)__shfl_sync(0xffffffffu, (uint32_t)(u_cur >> 32), r) << 32) |
                                   __shfl_sync(0xffffffffu, (uint32_t)u_cur, r);
              panel_or_fast(Vs, panel_pairs, sel, slot0, d);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) { w[2 * u] = g[u].x & d[u].x; w[2 * u + 1] = g[u].y & d[u].y; }
            if (MODE == 2) {
#pragma unroll
              for (int u = 0; u < 8; ++u) blk_tp += __popcll(w[u]);
            } else if (MODE == 3) {
              h4_tp.add4(sec_tp, w[0], w[2], w[4], w[6]);
              blk_tp += __popcll(w[1]) + __popcll(w[3]) + __popcll(w[5]) + __popcll(w[7]);
              sec_tp = !sec_tp;
            } else {
              if (!sec_tp) hs_tp.add8_first(w); else hs_tp.add8_second(w);
              sec_tp = !sec_tp;
            }
            if (ENTRIES) {
              if (has_z) {
#pragma unroll
                for (int u = 0; u < 4; ++u) blk_pd += __popcll(z[u].x & d[u].x) + __popcll(z[u].y & d[u].y);
              }
            } else if (cnt != 1) {                               // one factor: |prediction| came from pop_v
              if (MODE == 0) {
#pragma unroll
                for (int u = 0; u < 4; ++u) { w[2 * u] = d[u].x; w[2 * u + 1] = d[u].y; }
                if (!sec_pd) hs_pd.add8_first(w); else hs_pd.add8_second(w);
                sec_pd = !sec_pd;
              } else {
#pragma unroll
                for (int u = 0; u < 4; ++u) blk_pd += __popcll(d[u].x) + __popcll(d[u].y);
              }
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0)                                             // refill the slot(s) of this row
        for (int q = 0; q < segs && to_issue > 0; ++q) issue();
      if (++slot == RING_DEPTH) { slot = 0; phase ^= 1u; }
    }
    n_pd += blk_pd;
    n_tp += blk_tp;
  }
  const long long t_tp = warp_sum_ll(n_tp + hs_tp.total() + h4_tp.total());
  const long long t_pd = warp_sum_ll(n_pd + hs_pd.total());
  const long long t_gt = COUNT_GT ? warp_sum_ll(hs_gt.total()) : 0;
  if (lane == 0 && (t_pd | t_gt)) {
    atomicAdd(counts + 0, (unsigned long long)t_tp);
    atomicAdd(counts + 1, (unsigned long long)t_pd);
    if (COUNT_GT) atomicAdd(counts + 2, (unsigned long long)t_gt);
  }
  if (has_z) {
    const long long t_z = warp_sum_ll(hs_z.total());
    if (lane == 0 && t_z) atomicAdd(counts + 3, (unsigned long long)t_z);
  }
}

// DYNAMIC: the warps of all CTAs of a column panel draw their 32-row blocks from one counter (sched[panel], zero at launch)
// instead of owning every (#warps)-th block.  ncu on the static form: the CTAs do equal work but live 3.6 M cycles on
// average out of 4.3 M elapsed -- SMs drain their stores at different rates, and the early finishers idle for a sixth of
// the kernel.  The counter is read two blocks ahead (atomic for block i+2 and the usage words of block i+1 are in flight
// while block i is written), so its latency is never waited for.
// RESIDUAL (get_residual): pd receives x AND NOT (the product), x with the layout of pd.  Each lane loads its four x
// pairs of the segment before the OR chain, so the load latency overlaps the panel reads, and seeds the chain with ~x:
// the store of ~(~x | product) needs no registers beyond d's (x and d held apart spill at 64 registers).  A row that uses
// no factor stores x unchanged.
template <bool DYNAMIC, bool RESIDUAL = false>
__global__ void __launch_bounds__(PRODUCT_THREADS, 1)
bool_product_panel_list_kernel(const uint64_t* __restrict__ u_words, int64_t m, const uint64_t* __restrict__ vt,
                               int64_t k, int64_t words, int panel_chunks, int store_mode, const PanelGrid pg,
                               unsigned int* __restrict__ sched, const uint64_t* __restrict__ x,
                               uint64_t* __restrict__ pd) {
  extern __shared__ __align__(128) uint8_t panel_smem[];
  ulonglong2* Vs = reinterpret_cast<ulonglong2*>(panel_smem);
  const int panel_pairs = panel_chunks * CH_PAIRS;
  const int64_t pairs = words >> 1;
  int pg_panel, pg_split, pg_nsplit;
  panel_coords(pg, pg_panel, pg_split, pg_nsplit);
  const int64_t pair0 = (int64_t)pg_panel * pg.width_pairs;
  const int valid_pairs = (int)((pairs - pair0) < pg.width_pairs ? (pairs - pair0) : pg.width_pairs);
  load_vt_panel(Vs, vt, k, words, pair0, panel_pairs, valid_pairs);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const uint64_t kmask = k >= 64 ? ~0ull : ((1ull << k) - 1ull);
  const int64_t blk_step = (int64_t)pg_nsplit * nw;
  int64_t blk = (int64_t)pg_split * nw + warp;
  unsigned int ahead = 0;                                          // lane 0: the block after next
  if (DYNAMIC) {
    unsigned int first = 0;
    if (lane == 0) { first = atomicAdd(sched + pg_panel, 1u); ahead = atomicAdd(sched + pg_panel, 1u); }
    blk = (int64_t)__shfl_sync(0xffffffffu, first, 0);
  }
  uint64_t mine = (blk * 32 + lane < m) ? __ldg(u_words + blk * 32 + lane) : 0ull;
  while (blk * 32 < m) {
    const uint64_t u_cur = mine & kmask;
    int64_t nxt = blk + blk_step;
    if (DYNAMIC) {
      nxt = (int64_t)__shfl_sync(0xffffffffu, ahead, 0);
      if (lane == 0) ahead = atomicAdd(sched + pg_panel, 1u);
    }
    mine = (nxt * 32 + lane < m) ? __ldg(u_words + nxt * 32 + lane) : 0ull;
    const uint64_t list = pack_selection(u_cur);
    const uint32_t list_lo = (uint32_t)list, list_hi = (uint32_t)(list >> 32);
    const int nrows = (m - blk * 32) < 32 ? (int)(m - blk * 32) : 32;
    ulonglong2* out = reinterpret_cast<ulonglong2*>(pd + blk * 32 * words) + pair0;
    for (int r = 0; r < nrows; ++r, out += pairs) {
      const uint32_t lo = __shfl_sync(0xffffffffu, list_lo, r);
      const uint32_t hi = __shfl_sync(0xffffffffu, list_hi, r);
      const int cnt = (int)(hi >> 24);
      for (int c = 0; c < panel_chunks; ++c) {
        const int slot0 = c * CH_PAIRS + lane;
        if (c * CH_PAIRS >= valid_pairs) break;
        ulonglong2 d[4];
        if (RESIDUAL) {
          // x at out's offset, derived rather than carried (a second row pointer spills at 64 registers)
          const ulonglong2* xin = reinterpret_cast<const ulonglong2*>(x) + (out - reinterpret_cast<ulonglong2*>(pd));
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const ulonglong2 xv = slot0 + 32 * u < valid_pairs ? __ldg(xin + slot0 + 32 * u) : make_ulonglong2(0ull, 0ull);
            d[u] = make_ulonglong2(~xv.x, ~xv.y);
          }
        }
        if (cnt == 0) {
          if (!RESIDUAL) {
#pragma unroll
            for (int u = 0; u < 4; ++u) d[u] = make_ulonglong2(0ull, 0ull);
          }
        } else if (cnt <= 7) {
          panel_or_list<RESIDUAL>(Vs, panel_pairs, lo, hi, cnt, slot0, d);
        } else {
          const uint64_t sel = ((uint64_t)__shfl_sync(0xffffffffu, (uint32_t)(u_cur >> 32), r) << 32) |
                               __shfl_sync(0xffffffffu, (uint32_t)u_cur, r);
          panel_or_fast<RESIDUAL>(Vs, panel_pairs, sel, slot0, d);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (RESIDUAL) d[u] = make_ulonglong2(~d[u].x, ~d[u].y);       // ~(~x | product) = x AND NOT product
          if (slot0 + 32 * u < valid_pairs) {
            ulonglong2* dst = out + slot0 + 32 * u;
            if (store_mode == 0) __stcs(dst, d[u]);
            else if (store_mode == 1) *dst = d[u];
            else __stwt(dst, d[u]);
          }
        }
      }
    }
    blk = nxt;
  }
}

// One zeroed counter block per (device, stream) for the dynamically scheduled kernels: launches on a stream are ordered,
// so the memset that precedes each launch cannot race with the previous launch's atomics.
static unsigned int* stream_counters(cudaStream_t st) {
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, unsigned int*> table;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  auto it = table.find({dev, st});
  if (it != table.end()) return it->second;
  unsigned int* p = nullptr;
  if (cudaMalloc(&p, 64 * sizeof(unsigned int)) != cudaSuccess) return nullptr;
  table[{dev, st}] = p;
  return p;
}

// panel geometry for k <= 64 rows of V^T: chunks (of 256 words) per panel; 0 = use the row-stream kernels
constexpr int PANEL_SMEM_BUDGET = 224 * 1024;
static inline int panel_chunks_for(int64_t k, int64_t kw, int64_t words) {
  if (k <= 0 || k > 64 || kw != 1) return 0;
  const int64_t need = ceil_div(words >> 1, CH_PAIRS);
  // two chunks only when that makes ONE balanced panel and still leaves two ring slots per warp
  if (need == 2 && (k + 2 * PANEL_WARPS) * 2 * CH_PAIRS * 16 <= PANEL_SMEM_BUDGET) return 2;
  return 1;
}
static inline int confusion_ring_depth(int64_t k, int chunks) {
  const int64_t row_bytes = (int64_t)chunks * CH_PAIRS * 16;
  int64_t depth = (PANEL_SMEM_BUDGET - k * row_bytes) / (PANEL_WARPS * row_bytes);
  if (depth > RING_DEPTH_MAX) depth = RING_DEPTH_MAX;
  return (int)depth;
}
static inline size_t confusion_panel_smem(int64_t k, int chunks, int depth) {
  return (size_t)(k + PANEL_WARPS * depth) * chunks * CH_PAIRS * 16 + PANEL_WARPS * RING_DEPTH_MAX * 8 + 64 * sizeof(int);
}
// equal-width panels, one wave of CTAs (<= #SM); BMF_PANEL_BALANCE=0 restores full-width panels + a narrow last one
static inline PanelGrid make_panel_grid(int64_t pairs, int panel_pairs, int64_t max_splits, int* total_ctas) {
  const int64_t panels = ceil_div(pairs, panel_pairs);
  const char* e = getenv("BMF_PANEL_BALANCE");
  const bool balance = !(e != nullptr && e[0] == '0');
  int64_t splits = (int64_t)num_sms() / panels;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  PanelGrid g;
  g.panels = (int)panels;
  g.splits = (int)splits;
  g.width_pairs = balance ? (int)ceil_div(pairs, panels) : panel_pairs;
  *total_ctas = g.panels * g.splits;
  return g;
}
static inline int panel_rowmap() {              // BMF_PANEL_ROWMAP=1 selects the interleaved row order (A/B experiments)
  const char* e = getenv("BMF_PANEL_ROWMAP");
  return (e != nullptr && e[0] == '1') ? 1 : 0;
}
static inline bool panel_lists() {              // BMF_PANEL_LIST=0: the bit-scan forms of the panel kernels (A/B experiments)
  const char* e = getenv("BMF_PANEL_LIST");
  return !(e != nullptr && e[0] == '0');
}
static inline int confusion_count_mode() {      // BMF_CONFUSION_COUNT = 0 (tree / tree), 1 (tree / POPC), 2 (POPC / POPC)
  const char* e = getenv("BMF_CONFUSION_COUNT");
  if (e != nullptr && e[0] >= '0' && e[0] <= '3') return e[0] - '0';   // 3 (list kernel only): half tree, half POPC for |gt & pd|
  return panel_lists() ? 3 : 1;                 // measured best (profiles/r02z_c5_list_probe.log; bit-scan form: r02_c5_knob_sweep.log)
}
static inline int product_store_mode() {        // BMF_PRODUCT_STORE = 0 (st.cs, evict first), 1 (plain st), 2 (st.wt)
  const char* e = getenv("BMF_PRODUCT_STORE");
  if (e != nullptr && e[0] >= '0' && e[0] <= '2') return e[0] - '0';
  return 0;
}
static inline bool panel_dynamic() {            // BMF_PANEL_DYNAMIC=0: static row split of the product kernel (A/B experiments)
  const char* e = getenv("BMF_PANEL_DYNAMIC");
  return !(e != nullptr && e[0] == '0');
}
static inline bool panel_disabled() {
  const char* e = getenv("BMF_NO_PANEL");
  return e != nullptr && e[0] == '1';
}

// counts = (TP, |pd|, |gt| or unused) -> (TP, FP, FN)
__global__ void confusion_finalize_kernel(long long* __restrict__ counts, long long gt_ones) {
  const long long tp = counts[0], pd = counts[1], g = gt_ones >= 0 ? gt_ones : counts[2];
  counts[1] = pd - tp;
  counts[2] = g - tp;
}

// elementwise Boolean algebra on bit rows: op 0 = OR (add), 1 = AND (multiply), 2 = AND-NOT (residual)
__global__ void __launch_bounds__(256)
bits_combine_kernel(const ulonglong2* __restrict__ a, const ulonglong2* __restrict__ b, int64_t pairs, int op,
                    ulonglong2* __restrict__ out) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < pairs; t += (int64_t)gridDim.x * blockDim.x) {
    const ulonglong2 x = __ldg(a + t), y = __ldg(b + t);
    ulonglong2 r;
    if (op == 0) { r.x = x.x | y.x; r.y = x.y | y.y; }
    else if (op == 1) { r.x = x.x & y.x; r.y = x.y & y.y; }
    else { r.x = x.x & ~y.x; r.y = x.y & ~y.y; }
    out[t] = r;
  }
}

__global__ void confusion_triplets_kernel(const int32_t* __restrict__ rows, const int32_t* __restrict__ cols,
                                          const uint8_t* __restrict__ gt, int64_t nnz,
                                          const uint64_t* __restrict__ u_words, int64_t kw,
                                          const uint64_t* __restrict__ v_words,
                                          unsigned long long* __restrict__ counts) {
  int c[4] = {0, 0, 0, 0};   // TP FP FN TN
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz;
       e += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t* uw = u_words + (int64_t)rows[e] * kw;
    const uint64_t* vw = v_words + (int64_t)cols[e] * kw;
    uint64_t hit = 0;
    for (int64_t q = 0; q < kw; ++q) hit |= uw[q] & vw[q];
    const bool pd = hit != 0, g = gt[e] != 0;
    c[g ? (pd ? 0 : 2) : (pd ? 1 : 3)] += 1;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int s = warp_sum(c[q]);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(counts + q, (unsigned long long)s);
  }
}

// AssoIter.get_refined_column in one pass (PyBMF/models/AssoIter.py:80-100)
__global__ void __launch_bounds__(256)
refine_column_kernel(const uint64_t* __restrict__ xb, int64_t m, int64_t n, int64_t words,
                     uint64_t* __restrict__ u_words, int64_t kw, const uint64_t* __restrict__ vt,
                     int64_t col, int wa, int wb, double neg_w_fp, double w_fn,
                     unsigned long long* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t pairs = words >> 1;
  const uint64_t* __restrict__ vcol = vt + col * words;
  long long t_tp = 0, t_fp = 0, t_used = 0, t_p = 0, t_n = 0;
  for (int64_t i = warp0; i < m; i += nwarps) {
    uint64_t* uw = u_words + i * kw;
    int tpo = 0, fpo = 0, P = 0, N = 0;
    for (int64_t p0 = lane; p0 < pairs; p0 += 32 * PU) {
      ulonglong2 x[PU], c[PU];
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int64_t p = p0 + 32 * u;
        x[u] = make_ulonglong2(0ull, 0ull);
        if (p < pairs) x[u] = __ldcs(reinterpret_cast<const ulonglong2*>(xb + i * words + 2 * p));
      }
      product_quad(uw, kw, vt, words, p0, pairs, col, c);               // cover without factor `col`
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int64_t p = p0 + 32 * u;
        if (p >= pairs) continue;
        const ulonglong2 v = ld_words2(vcol + 2 * p);
        tpo += __popcll(x[u].x & c[u].x) + __popcll(x[u].y & c[u].y);
        fpo += __popcll(c[u].x) + __popcll(c[u].y);                      // |c|, minus tpo below
        P += __popcll(x[u].x & ~c[u].x & v.x) + __popcll(x[u].y & ~c[u].y & v.y);
        N += __popcll(~c[u].x & v.x) + __popcll(~c[u].y & v.y);          // |v & ~c|, minus P below
      }
    }
    tpo = warp_sum(tpo); fpo = warp_sum(fpo) - tpo; P = warp_sum(P); N = warp_sum(N) - P;
    const bool use = row_uses(wa, wb, neg_w_fp, w_fn, tpo, fpo, P, N);
    __syncwarp();
    if (lane == 0) {
      const uint64_t bit = 1ull << (col & 63);
      uint64_t w = uw[col >> 6];
      w = use ? (w | bit) : (w & ~bit);                                  // AssoIter.py:60: always overwritten
      uw[col >> 6] = w;
      t_tp += tpo + (use ? P : 0);
      t_fp += fpo + (use ? N : 0);
      if (use) { t_used += 1; t_p += P; t_n += N; }
    }
    __syncwarp();
  }
  if (lane == 0) {
    atomicAdd(out + 0, (unsigned long long)t_tp);
    atomicAdd(out + 1, (unsigned long long)t_fp);
    atomicAdd(out + 2, (unsigned long long)t_used);
    atomicAdd(out + 3, (unsigned long long)t_p);
    atomicAdd(out + 4, (unsigned long long)t_n);
  }
}

// AssoIter.get_refined_column for columns col0 .. col0+ncols-1 in ONE pass over the rows.  Row i's new bit U[i, c]
// depends only on X_i, V and row i's own usage bits, so a warp walks the columns of its row in order (the bits of
// columns already refined in this sweep are read back from the usage word) and adds the row's state after column c to
// column c's counters: the sums equal what ncols successive refine_column_kernel launches accumulate.
// With A = the cover without column c, the cover before column c is A | (old bit ? v_c : 0), hence
//   TP(A) = TP - (old ? P : 0),  FP(A) = FP - (old ? N : 0),   P = |x & ~A & v_c|,  N = |~x & ~A & v_c|
// so the row's TP / FP are carried from column to column (counted once, against the starting cover) and every column
// costs two popcounts per word (P and |~A & v_c|) instead of the four of refine_column_kernel.  The data row is read
// from DRAM once and re-read from L1 / L2 for the following columns; V^T sits in shared memory when it fits (VS).
template <bool VS>
__device__ __forceinline__ ulonglong2 ld_vt2(const uint64_t* p) {
  if constexpr (VS) return *reinterpret_cast<const ulonglong2*>(p);
  else return ld_words2(p);
}

template <bool VS>
__device__ __forceinline__ void sweep_cover(const uint64_t* uw, int64_t kw, const uint64_t* V, int64_t words, int64_t p0,
                                            int64_t pairs, int64_t skip, ulonglong2 (&acc)[PU]) {
#pragma unroll
  for (int u = 0; u < PU; ++u) acc[u] = make_ulonglong2(0ull, 0ull);
  for (int64_t q = 0; q < kw; ++q) {
    uint64_t sel = uw[q];
    if ((skip >> 6) == q) sel &= ~(1ull << (skip & 63));
    while (sel) {
      const int l = __ffsll((long long)sel) - 1;
      sel &= sel - 1;
      const uint64_t* vrow = V + (q * 64 + l) * words;
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int64_t p = p0 + 32 * u;
        if (p < pairs) {
          const ulonglong2 v = ld_vt2<VS>(vrow + 2 * p);
          acc[u].x |= v.x;
          acc[u].y |= v.y;
        }
      }
    }
  }
}

template <bool VS>
__global__ void __launch_bounds__(256)
refine_sweep_kernel(const uint64_t* __restrict__ xb, int64_t m, int64_t words, uint64_t* __restrict__ u_words,
                    int64_t kw, const uint64_t* __restrict__ vt, int64_t k, int64_t col0, int64_t ncols, int wa, int wb,
                    double neg_w_fp, double w_fn, int cnt_in_smem, unsigned long long* __restrict__ out) {
  extern __shared__ __align__(16) uint64_t sweep_smem[];
  const int lane = threadIdx.x & 31;
  const int64_t pairs = words >> 1;
  const uint64_t* V = vt;
  unsigned long long* cnt = out;                                        // [ncols][5]
  if (VS) {
    for (int64_t q = threadIdx.x; q < k * pairs; q += blockDim.x)
      reinterpret_cast<ulonglong2*>(sweep_smem)[q] = ld_words2(vt + 2 * q);
    V = sweep_smem;
  }
  if (cnt_in_smem) {
    cnt = reinterpret_cast<unsigned long long*>(sweep_smem + (VS ? k * words : 0));
    for (int64_t q = threadIdx.x; q < ncols * 5; q += blockDim.x) cnt[q] = 0ull;
  }
  if (VS || cnt_in_smem) __syncthreads();
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp0; i < m; i += nwarps) {
    const uint64_t* x = xb + i * words;
    uint64_t* uw = u_words + i * kw;
    int tp = 0, pd = 0;
    for (int64_t p0 = lane; p0 < pairs; p0 += 32 * PU) {                 // TP / FP of the starting cover
      ulonglong2 c[PU];
      sweep_cover<VS>(uw, kw, V, words, p0, pairs, -1, c);
#pragma unroll
      for (int u = 0; u < PU; ++u) {
        const int64_t p = p0 + 32 * u;
        if (p >= pairs) continue;
        const ulonglong2 xv = ld_words2(x + 2 * p);
        tp += __popcll(xv.x & c[u].x) + __popcll(xv.y & c[u].y);
        pd += __popcll(c[u].x) + __popcll(c[u].y);
      }
    }
    tp = warp_sum(tp);
    int fp = warp_sum(pd) - tp;
    for (int64_t j = 0; j < ncols; ++j) {
      const int64_t col = col0 + j;
      const uint64_t* vcol = V + col * words;
      int P = 0, A = 0;
      for (int64_t p0 = lane; p0 < pairs; p0 += 32 * PU) {
        ulonglong2 c[PU];
        sweep_cover<VS>(uw, kw, V, words, p0, pairs, col, c);           // cover without factor `col`
#pragma unroll
        for (int u = 0; u < PU; ++u) {
          const int64_t p = p0 + 32 * u;
          if (p >= pairs) continue;
          const ulonglong2 xv = ld_words2(x + 2 * p);
          const ulonglong2 v = ld_vt2<VS>(vcol + 2 * p);
          const uint64_t nx = v.x & ~c[u].x, ny = v.y & ~c[u].y;
          P += __popcll(xv.x & nx) + __popcll(xv.y & ny);
          A += __popcll(nx) + __popcll(ny);                               // |v & ~c| = P + N
        }
      }
      P = warp_sum(P);
      const int N = warp_sum(A) - P;
      const uint64_t bit = 1ull << (col & 63);
      const bool old = (uw[col >> 6] & bit) != 0;
      const int tpo = tp - (old ? P : 0), fpo = fp - (old ? N : 0);
      const bool use = row_uses(wa, wb, neg_w_fp, w_fn, tpo, fpo, P, N);  // warp-uniform
      tp = tpo + (use ? P : 0);
      fp = fpo + (use ? N : 0);
      __syncwarp();
      if (lane == 0 && use != old) uw[col >> 6] ^= bit;                  // AssoIter.py:60: always overwritten
      if (lane < 5) {
        const int v = lane == 0 ? tp : lane == 1 ? fp : !use ? 0 : lane == 2 ? 1 : lane == 3 ? P : N;
        if (v) atomicAdd(cnt + j * 5 + lane, (unsigned long long)v);
      }
      __syncwarp();
    }
  }
  if (cnt_in_smem) {
    __syncthreads();
    for (int64_t q = threadIdx.x; q < ncols * 5; q += blockDim.x)
      if (cnt[q]) atomicAdd(out + q, cnt[q]);
  }
}

// =========================================================================================
// GreConD+ expansion scores (PyBMF/models/GreConDPlus.py:267-308, `_expansion`): adding `pattern` to every row that is
// not excluded, how much does each row's coverage score change?
//   delta_i = [(-w_fp)(FP_i + N_i) + w_fn (TP_i + P_i)] - [(-w_fp) FP_i + w_fn TP_i]   (fp64, the reference's order)
// with TP_i / FP_i of `old` against x and P_i / N_i the new true / false positives; excluded rows keep X_new = X_old,
// so delta_i = +0.0.  Row-wise expansion passes (X, X_old, pattern = v, exclude = u); column-wise expansion passes
// the transposed bit matrices with (pattern = u, exclude = v).  One warp per row, 128-bit row streams.
// =========================================================================================
__global__ void __launch_bounds__(256)
expand_delta_kernel(const uint64_t* __restrict__ xb, const uint64_t* __restrict__ ob, int64_t rows, int64_t words,
                    const uint64_t* __restrict__ pattern, const uint64_t* __restrict__ exclude, double neg_w_fp,
                    double w_fn, double* __restrict__ delta) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t pairs = words >> 1;
  for (int64_t i = warp0; i < rows; i += nwarps) {
    if (exclude != nullptr && ((exclude[i >> 6] >> (i & 63)) & 1ull)) {      // warp-uniform
      if (lane == 0) delta[i] = 0.0;
      continue;
    }
    int tp = 0, pd = 0, P = 0, A = 0;
    for (int64_t p = lane; p < pairs; p += 32) {
      const ulonglong2 x = ld_words2(xb + i * words + 2 * p);
      const ulonglong2 o = ld_words2(ob + i * words + 2 * p);
      const ulonglong2 v = ld_words2(pattern + 2 * p);
      tp += __popcll(x.x & o.x) + __popcll(x.y & o.y);
      pd += __popcll(o.x) + __popcll(o.y);
      P += __popcll(x.x & ~o.x & v.x) + __popcll(x.y & ~o.y & v.y);
      A += __popcll(~o.x & v.x) + __popcll(~o.y & v.y);                       // |v & ~old| = P + N
    }
    tp = warp_sum(tp); pd = warp_sum(pd); P = warp_sum(P); A = warp_sum(A);
    if (lane == 0) {
      const int fp = pd - tp, N = A - P;
      const double s_old = cover_score_f64(neg_w_fp, w_fn, fp, tp);
      const double s_new = cover_score_f64(neg_w_fp, w_fn, fp + N, tp + P);
      delta[i] = __dsub_rn(s_new, s_old);
    }
  }
}

// max and FIRST argmax of a float64 vector (numpy's d_scores.max() / d_scores.argmax()); out[0] = bits, out[1] = index
__global__ void __launch_bounds__(1024) argmax_first_f64_kernel(const double* __restrict__ v, int64_t n, long long* __restrict__ out) {
  __shared__ double s_val[32];
  __shared__ long long s_idx[32];
  double best = 0.0;
  long long idx = -1;
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
    const double x = v[j];
    if (idx < 0 || x > best) { best = x; idx = j; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (oi >= 0 && (idx < 0 || ov > best || (ov == best && oi < idx))) { best = ov; idx = oi; }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_val[warp] = best; s_idx[warp] = idx; }
  __syncthreads();
  if (warp == 0) {
    best = s_val[lane];
    idx = s_idx[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, best, o);
      const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
      if (oi >= 0 && (idx < 0 || ov > best || (ov == best && oi < idx))) { best = ov; idx = oi; }
    }
    if (lane == 0) { out[0] = __double_as_longlong(best); out[1] = idx; }
  }
}

// =========================================================================================
// Incremental GreConD+ expansion (GreConDPlus.py:207-264, `expansion`).  X_old is fixed for the whole loop, so the
// per-row TP_old / FP_old and the per-column TP_old / FP_old never change, and one iteration changes the increments by
// one bit per row (a column c joined v) or by one row's bits per column (a row r joined u).  One streaming pass
// (expand_init_kernel) produces every count; an iteration then costs O(m + n) (expand_step_rows_kernel,
// expand_step_decide_kernel), with the deltas evaluated from the same integers by the same fp64 expression as
// expand_delta_kernel, so they are bit-identical.
// =========================================================================================

// (max, FIRST argmax) merge: a candidate with a lower index wins a tie; idx < 0 is "no candidate"
__device__ __forceinline__ void better_first(double& best, long long& idx, double v, long long i) {
  if (i >= 0 && (idx < 0 || v > best || (v == best && i < idx))) { best = v; idx = i; }
}

// block-wide better_first (every thread returns the block's result); blockDim.x = 256
__device__ __forceinline__ void block_first_max(double& best, long long& idx) {
  __shared__ double s_val[8];
  __shared__ long long s_idx[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    better_first(best, idx, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, idx, o));
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) { s_val[warp] = best; s_idx[warp] = idx; }
  __syncthreads();
  best = s_val[0];
  idx = s_idx[0];
  for (int q = 1; q < 8; ++q) better_first(best, idx, s_val[q], s_idx[q]);
}

// Every block stores its (max, argmax) in partials[blockIdx.x]; the block that arrives last returns true with the
// grid's result in (best, idx) and re-arms the counter for the next launch.
__device__ __forceinline__ bool grid_first_max(double& best, long long& idx, long long* __restrict__ partials,
                                               unsigned long long* counter) {
  __shared__ int s_last;
  block_first_max(best, idx);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = __double_as_longlong(best);
    partials[2 * blockIdx.x + 1] = idx;
    __threadfence();
    s_last = atomicAdd(counter, 1ull) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  best = 0.0;
  idx = -1;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x)
    better_first(best, idx, __longlong_as_double(__ldcg(partials + 2 * b)), __ldcg(partials + 2 * b + 1));
  block_first_max(best, idx);
  if (threadIdx.x == 0) *counter = 0ull;
  return true;
}

// Bit-sliced (positional) counter of 64 columns: value of column c = sum_b bit c of plane b * 2^b.  Eight one-bit
// inputs enter a carry-save tree (ones / twos / fours, Harley-Seal); its carry of weight 8 ripples into the planes hi.
constexpr int kExpandHiPlanes = 8;                                   // <= 255 groups of 8 rows between two flushes
constexpr int kExpandRowsPerWarp = 1024;
struct PosCount {
  uint64_t ones, twos, fours, hi[kExpandHiPlanes];
  __device__ __forceinline__ void clear() {
    ones = twos = fours = 0ull;
#pragma unroll
    for (int b = 0; b < kExpandHiPlanes; ++b) hi[b] = 0ull;
  }
  __device__ __forceinline__ void add8(const uint64_t (&a)[8]) {
    uint64_t tA, tB, fA, fB, e;
    csa64(tA, ones, ones, a[0], a[1]);
    csa64(tB, ones, ones, a[2], a[3]);
    csa64(fA, twos, twos, tA, tB);
    csa64(tA, ones, ones, a[4], a[5]);
    csa64(tB, ones, ones, a[6], a[7]);
    csa64(fB, twos, twos, tA, tB);
    csa64(e, fours, fours, fA, fB);
#pragma unroll
    for (int b = 0; b < kExpandHiPlanes; ++b) {
      const uint64_t c = hi[b] & e;
      hi[b] ^= e;
      e = c;
    }
  }
  __device__ __forceinline__ unsigned value(int c) const {
    unsigned v = (unsigned)((ones >> c) & 1ull) | ((unsigned)((twos >> c) & 1ull) << 1) |
                 ((unsigned)((fours >> c) & 1ull) << 2);
#pragma unroll
    for (int b = 0; b < kExpandHiPlanes; ++b) v |= (unsigned)((hi[b] >> c) & 1ull) << (3 + b);
    return v;
  }
};

// One pass over rows [0, rows) of x / old (logical rows row0 + i).  Block (bx, by) covers words [32 bx, 32 bx + 32) of
// rows [8 rpw by, 8 rpw (by + 1)); warp q of the block the rows [rpw q, rpw (q + 1)) of that range, lane l word 32 bx + l.
//   row_cnt[i] = (TP_old, FP_old, P, N) += this window's share (two 64-bit atomics per row and window), P / N against v;
//   col_cnt[k][j] += counter k of column j over the block's rows: TP_old (x & old), FP_old (~x & old), and over the rows in
//   u: P (x & ~old), N (~x & ~old, pad bits masked).  Lanes count their 64 columns in PosCount registers, flush them
//   into the block's shared table once per warp and the block adds the table to col_cnt once.
__global__ void __launch_bounds__(256)
expand_init_kernel(const uint64_t* __restrict__ xb, const uint64_t* __restrict__ ob, int64_t rows, int64_t n,
                   int64_t words, int64_t row0, const uint64_t* __restrict__ u, const uint64_t* __restrict__ v,
                   int32_t* __restrict__ row_cnt, unsigned long long* __restrict__ col_cnt, int64_t rpw) {
  __shared__ unsigned s_cnt[4][64][32];                             // [counter][bit][lane]: conflict-free flushes
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t w0 = (int64_t)blockIdx.x * 32, w = w0 + lane;
  const bool active = w < words;
  const int64_t valid_bits = n - w * 64;
  const uint64_t colmask = !active || valid_bits <= 0 ? 0ull : valid_bits >= 64 ? ~0ull : (1ull << valid_bits) - 1ull;
  const uint64_t vw = active ? v[w] : 0ull;
  for (int e = threadIdx.x; e < 4 * 64 * 32; e += 256) (&s_cnt[0][0][0])[e] = 0u;
  __syncthreads();
  const int64_t rb = ((int64_t)blockIdx.y * 8 + warp) * rpw;
  const int64_t re = rb + rpw < rows ? rb + rpw : rows;
  if (rb < re) {
    PosCount ctp, cfp, cP, cN;
    ctp.clear(); cfp.clear(); cP.clear(); cN.clear();
    for (int64_t i0 = rb; i0 < re; i0 += 8) {
      uint64_t xw[8], ow[8], um[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int64_t i = i0 + q;
        const bool ok = i < re;
        xw[q] = ok && active ? __ldg(xb + i * words + w) : 0ull;
        ow[q] = ok && active ? __ldg(ob + i * words + w) : 0ull;
        const int64_t g = row0 + i;
        um[q] = ok ? 0ull - ((__ldg(u + (g >> 6)) >> (g & 63)) & 1ull) : 0ull;
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        unsigned t = (unsigned)__popcll(xw[q] & ow[q]) | ((unsigned)__popcll(~xw[q] & ow[q]) << 16);
        unsigned p = (unsigned)__popcll(xw[q] & ~ow[q] & vw) | ((unsigned)__popcll(~xw[q] & ~ow[q] & vw) << 16);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          t += __shfl_xor_sync(0xffffffffu, t, o);
          p += __shfl_xor_sync(0xffffffffu, p, o);
        }
        const int64_t i = i0 + q;
        if (lane == 0 && i < re) {                                   // (TP, FP) and (P, N): one 64-bit add each
          unsigned long long* rc = reinterpret_cast<unsigned long long*>(row_cnt + 4 * i);
          if (t) atomicAdd(rc, (unsigned long long)(t & 0xffffu) | ((unsigned long long)(t >> 16) << 32));
          if (p) atomicAdd(rc + 1, (unsigned long long)(p & 0xffffu) | ((unsigned long long)(p >> 16) << 32));
        }
      }
      uint64_t a[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) a[q] = xw[q] & ow[q];
      ctp.add8(a);
#pragma unroll
      for (int q = 0; q < 8; ++q) a[q] = ~xw[q] & ow[q];
      cfp.add8(a);
#pragma unroll
      for (int q = 0; q < 8; ++q) a[q] = xw[q] & ~ow[q] & um[q];
      cP.add8(a);
#pragma unroll
      for (int q = 0; q < 8; ++q) a[q] = ~xw[q] & ~ow[q] & um[q] & colmask;
      cN.add8(a);
    }
    if (active) {
      for (int c = 0; c < 64; ++c) {
        unsigned val;
        if ((val = ctp.value(c))) atomicAdd(&s_cnt[0][c][lane], val);
        if ((val = cfp.value(c))) atomicAdd(&s_cnt[1][c][lane], val);
        if ((val = cP.value(c))) atomicAdd(&s_cnt[2][c][lane], val);
        if ((val = cN.value(c))) atomicAdd(&s_cnt[3][c][lane], val);
      }
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 4 * 64 * 32; e += 256) {
    const int k = e >> 11, c = (e >> 5) & 63, l = e & 31;
    const int64_t j = (w0 + l) * 64 + c;
    const unsigned val = s_cnt[k][c][l];
    if (val && j < n) atomicAdd(col_cnt + k * n + j, (unsigned long long)val);
  }
}

// Iteration, part 1 (grid over the rank's rows).  A column c chosen by the previous decision adds bit c of x & ~old /
// ~x & ~old to every row's P / N; every row's delta is evaluated (+0.0 in u) and the last block writes the exchange
// buffer: slot `rank` = (bits of the local max, its logical row), every other slot 0, and the words of the row r chosen by
// the previous decision (x & ~old, ~x & ~old masked to n) if this rank owns r, else 0.  No-op but for zeroing the buffer
// once state[0] (stopped) is set.
__global__ void __launch_bounds__(256)
expand_step_rows_kernel(const uint64_t* __restrict__ xb, const uint64_t* __restrict__ ob, int64_t rows, int64_t n,
                        int64_t words, int64_t row0, const uint64_t* __restrict__ u, int32_t* __restrict__ row_cnt,
                        double neg_w_fp, double w_fn, long long* __restrict__ state, long long* __restrict__ partials,
                        long long* __restrict__ xbuf, int64_t world, int64_t rank) {
  const int64_t buf_len = 2 * world + 2 * words;
  if (state[0]) {
    if (blockIdx.x == 0)
      for (int64_t e = threadIdx.x; e < buf_len; e += blockDim.x) xbuf[e] = 0;
    return;
  }
  const long long c = state[2];
  double best = 0.0;
  long long idx = -1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x) {
    int4 cnt = reinterpret_cast<const int4*>(row_cnt)[i];
    if (c >= 0) {
      const uint64_t bit = 1ull << (c & 63);
      const uint64_t xw = xb[i * words + (c >> 6)], ow = ob[i * words + (c >> 6)];
      if (!(ow & bit)) {
        if (xw & bit) row_cnt[4 * i + 2] = ++cnt.z;
        else row_cnt[4 * i + 3] = ++cnt.w;
      }
    }
    const int64_t g = row0 + i;
    double d = 0.0;
    if (!((u[g >> 6] >> (g & 63)) & 1ull)) {
      const double s_old = cover_score_f64(neg_w_fp, w_fn, cnt.y, cnt.x);
      const double s_new = cover_score_f64(neg_w_fp, w_fn, cnt.y + cnt.w, cnt.x + cnt.z);
      d = __dsub_rn(s_new, s_old);
    }
    better_first(best, idx, d, g);
  }
  if (!grid_first_max(best, idx, partials, reinterpret_cast<unsigned long long*>(state + 4))) return;
  const long long r = state[1];
  const bool own = r >= row0 && r < row0 + rows;
  for (int64_t e = threadIdx.x; e < buf_len; e += blockDim.x) {
    long long val = 0;
    if (e == 2 * rank) val = __double_as_longlong(best);
    else if (e == 2 * rank + 1) val = idx;
    else if (e >= 2 * world && own) {
      const int64_t wq = (e - 2 * world) % words;
      const uint64_t xw = xb[(r - row0) * words + wq], ow = ob[(r - row0) * words + wq];
      const int64_t valid_bits = n - wq * 64;
      const uint64_t mask = valid_bits <= 0 ? 0ull : valid_bits >= 64 ? ~0ull : (1ull << valid_bits) - 1ull;
      val = (long long)(e < 2 * world + words ? xw & ~ow : ~xw & ~ow & mask);
    }
    xbuf[e] = val;
  }
}

// Iteration, part 2 (grid over the columns; after the buffers of all ranks were summed).  The row r chosen by the
// previous decision adds its words to every column's P / N; every column's delta is evaluated (+0.0 in v); the last block
// merges the rank slots (max, then the lowest logical row) and applies the reference's rule (GreConDPlus.py:221-236):
// a row if r_score > c_score and r_score > 0, a column if c_score > r_score and c_score > 0, else stop.  It sets the bit
// in u / v, appends (0 row | 1 column | 2 stop, index) to the log and updates state.
__global__ void __launch_bounds__(256)
expand_step_decide_kernel(long long* __restrict__ col_cnt, int64_t n, int64_t words, uint64_t* __restrict__ u,
                          uint64_t* __restrict__ v, double neg_w_fp, double w_fn, long long* __restrict__ state,
                          long long* __restrict__ partials, const long long* __restrict__ xbuf, int64_t world,
                          long long* __restrict__ log, int64_t log_cap) {
  if (state[0]) return;
  const long long r = state[1];
  const uint64_t* rp = reinterpret_cast<const uint64_t*>(xbuf + 2 * world);
  const uint64_t* rn = rp + words;
  double best = 0.0;
  long long idx = -1;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    const long long tp = col_cnt[j], fp = col_cnt[n + j];
    long long P = col_cnt[2 * n + j], N = col_cnt[3 * n + j];
    if (r >= 0) {
      if ((rp[j >> 6] >> (j & 63)) & 1ull) col_cnt[2 * n + j] = ++P;
      if ((rn[j >> 6] >> (j & 63)) & 1ull) col_cnt[3 * n + j] = ++N;
    }
    double d = 0.0;
    if (!((v[j >> 6] >> (j & 63)) & 1ull)) {
      const double s_old = cover_score_f64(neg_w_fp, w_fn, (int)fp, (int)tp);
      const double s_new = cover_score_f64(neg_w_fp, w_fn, (int)(fp + N), (int)(tp + P));
      d = __dsub_rn(s_new, s_old);
    }
    better_first(best, idx, d, j);
  }
  if (!grid_first_max(best, idx, partials, reinterpret_cast<unsigned long long*>(state + 5))) return;
  if (threadIdx.x != 0) return;
  double r_score = 0.0;
  long long r_index = -1;
  for (int64_t q = 0; q < world; ++q) better_first(r_score, r_index, __longlong_as_double(xbuf[2 * q]), xbuf[2 * q + 1]);
  const long long t = state[3];
  long long kind = 2, at = -1;
  if (r_score > best && r_score > 0.0) {
    kind = 0; at = r_index;
    u[r_index >> 6] |= 1ull << (r_index & 63);
    state[1] = r_index; state[2] = -1;
  } else if (best > r_score && best > 0.0) {
    kind = 1; at = idx;
    v[idx >> 6] |= 1ull << (idx & 63);
    state[1] = -1; state[2] = idx;
  } else {
    state[0] = 1;
  }
  if (t < log_cap) { log[2 * t] = kind; log[2 * t + 1] = at; }
  state[3] = t + 1;
}

// column deltas of _expansion(axis = 0) from the column counts: delta[j] = +0.0 for j in v
__global__ void __launch_bounds__(256)
expand_col_delta_kernel(const long long* __restrict__ col_cnt, int64_t n, const uint64_t* __restrict__ v, double neg_w_fp,
                        double w_fn, double* __restrict__ delta) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    double d = 0.0;
    if (!((v[j >> 6] >> (j & 63)) & 1ull)) {
      const long long tp = col_cnt[j], fp = col_cnt[n + j], P = col_cnt[2 * n + j], N = col_cnt[3 * n + j];
      d = __dsub_rn(cover_score_f64(neg_w_fp, w_fn, (int)(fp + N), (int)(tp + P)),
                    cover_score_f64(neg_w_fp, w_fn, (int)fp, (int)tp));
    }
    delta[j] = d;
  }
}

// =========================================================================================
// AssoOpt.set_optimal_row (PyBMF/models/AssoOpt.py:69-80): for data row i try all 2^k usage vectors, the score of trial
// j is (-w_fp) FP + w_fn TP of  OR_{l in bits(j)} V^T_l  against x_i, and the FIRST maximum wins (np.argmax).
// int2bin (AssoOpt.py:83-86) writes j MSB first, so factor l is bit (k - 1 - l) of j.
// One CTA per data row, trials strided over the threads; V^T sits in shared memory when it fits.
// =========================================================================================
__global__ void __launch_bounds__(256)
optimal_row_kernel(const uint64_t* __restrict__ xb, int64_t m, int64_t words, const uint64_t* __restrict__ vt, int k,
                   double neg_w_fp, double w_fn, int vt_in_smem, long long* __restrict__ best_trial,
                   double* __restrict__ best_score) {
  extern __shared__ uint64_t opt_smem[];
  __shared__ double s_val[8];
  __shared__ long long s_idx[8];
  const uint64_t* V = vt;
  if (vt_in_smem) {
    for (int64_t e = threadIdx.x; e < (int64_t)k * words; e += blockDim.x) opt_smem[e] = vt[e];
    __syncthreads();
    V = opt_smem;
  }
  const long long trials = 1ll << k;
  for (int64_t i = blockIdx.x; i < m; i += gridDim.x) {
    const uint64_t* x = xb + i * words;
    double best = 0.0;
    long long idx = -1;
    for (long long j = threadIdx.x; j < trials; j += blockDim.x) {
      int tp = 0, pd = 0;
      for (int64_t w = 0; w < words; ++w) {
        uint64_t acc = 0;
        for (int l = 0; l < k; ++l)
          if ((j >> (k - 1 - l)) & 1ll) acc |= V[(int64_t)l * words + w];
        tp += __popcll(acc & x[w]);
        pd += __popcll(acc);
      }
      const double sc = cover_score_f64(neg_w_fp, w_fn, pd - tp, tp);
      if (idx < 0 || sc > best) { best = sc; idx = j; }                    // ascending j per thread
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, best, o);
      const long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
      if (oi >= 0 && (idx < 0 || ov > best || (ov == best && oi < idx))) { best = ov; idx = oi; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) { s_val[warp] = best; s_idx[warp] = idx; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int q = 1; q < (int)(blockDim.x >> 5); ++q)
        if (s_idx[q] >= 0 && (idx < 0 || s_val[q] > best || (s_val[q] == best && s_idx[q] < idx))) { best = s_val[q]; idx = s_idx[q]; }
      best_trial[i] = idx;
      if (best_score != nullptr) best_score[i] = best;
    }
  }
}

// =========================================================================================
// On-device synthetic inputs (SURVEY section 8f rank 3): the generators' recipe -- Boolean product of two random
// factors (PyBMF/generators/BaseGenerator.py:202-221 boolean_matmul) followed by add_noise
// (PyBMF/utils/generator_utils.py:30-49: ones dropped with probability p_pos, then every entry set with probability
// p_neg) -- with a COUNTER-BASED generator: bit (i, j) of stream s is a pure function of (seed, s, i, j), so a rank that
// generates only its own row range produces exactly the rows a single GPU would.  Not bit-identical to numpy's
// Mersenne twister (validated by density / shard-independence / a fit against the CPU restatement on the same bits).
// =========================================================================================
__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// 64 Bernoulli(p) bits for global bit indices [base, base + 64): two draws per 64-bit hash (threshold = p * 2^32)
__device__ __forceinline__ uint64_t bernoulli_word(uint64_t seed, uint64_t stream, uint64_t base, uint32_t thr) {
  uint64_t w = 0;
  const uint64_t key = seed * 0x9E3779B97F4A7C15ull + stream * 0xD1B54A32D192ED03ull;
#pragma unroll 4
  for (int q = 0; q < 32; ++q) {
    const uint64_t h = splitmix64(key + (base >> 1) + (uint64_t)q);
    w |= (uint64_t)((uint32_t)h < thr) << (2 * q);
    w |= (uint64_t)((uint32_t)(h >> 32) < thr) << (2 * q + 1);
  }
  return w;
}
// out[r][w] = Bernoulli(p) bits of logical row (row0 + r), columns [64 w, 64 w + 64) of a (rows x ncols) matrix
__global__ void random_bits_kernel(uint64_t* __restrict__ out, int64_t rows, int64_t ncols, int64_t words, int64_t row0,
                                   uint64_t seed, uint64_t stream, uint32_t thr) {
  const int64_t total = rows * words;
  const int64_t cw = (ncols + 63) >> 6;                   // words that hold real columns
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / words, w = t - r * words;
    uint64_t v = 0;
    if (w < cw) {
      v = bernoulli_word(seed, stream, (uint64_t)((row0 + r) * cw + w) * 64ull, thr);
      const int64_t left = ncols - w * 64;
      if (left < 64) v &= (1ull << left) - 1ull;
    }
    out[t] = v;
  }
}
// add_noise on bit rows: x = (x & ~drop) | flip with drop ~ Bernoulli(p_pos), flip ~ Bernoulli(p_neg) per entry
__global__ void noise_bits_kernel(uint64_t* __restrict__ x, int64_t rows, int64_t ncols, int64_t words, int64_t row0,
                                  uint64_t seed, uint32_t thr_pos, uint32_t thr_neg) {
  const int64_t total = rows * words;
  const int64_t cw = (ncols + 63) >> 6;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / words, w = t - r * words;
    if (w >= cw) continue;
    const uint64_t base = (uint64_t)((row0 + r) * cw + w) * 64ull;
    uint64_t v = x[t];
    if (thr_pos) v &= ~bernoulli_word(seed, 3, base, thr_pos);
    if (thr_neg) v |= bernoulli_word(seed, 4, base, thr_neg);
    const int64_t left = ncols - w * 64;
    if (left < 64) v &= (1ull << left) - 1ull;
    x[t] = v;
  }
}
// ratio_split on bit rows (generate.ratio_split): every one of x draws u from stream s_ones and goes to val (u < t_v), test
// (u < t_v + t_t) or train; every zero inside the ncols columns draws from stream s_zeros and becomes a stored zero of val
// (u < q_v), of test (u < q_v + q_t) or stays unstored.  u is the 32-bit half of bernoulli_word's hash for the global bit
// index, so the result depends on (seed, i, j) only.  out = 5 matrices [rows][words] (train, val ones, val zeros, test
// ones, test zeros), every word written, pad bits zero.
__device__ __forceinline__ uint32_t draw32(uint64_t key, uint64_t bit) {
  const uint64_t h = splitmix64(key + (bit >> 1));
  return (bit & 1) ? (uint32_t)(h >> 32) : (uint32_t)h;
}
__global__ void __launch_bounds__(256)
split_bits_kernel(const uint64_t* __restrict__ x, int64_t rows, int64_t ncols, int64_t words, int64_t row0, uint64_t seed,
                  uint64_t s_ones, uint64_t s_zeros, uint64_t t_v, uint64_t t_vt, uint64_t q_v, uint64_t q_vt,
                  uint64_t* __restrict__ out) {
  const int64_t total = rows * words;
  const int64_t cw = (ncols + 63) >> 6;
  const uint64_t k1 = seed * 0x9E3779B97F4A7C15ull + s_ones * 0xD1B54A32D192ED03ull;
  const uint64_t k0 = seed * 0x9E3779B97F4A7C15ull + s_zeros * 0xD1B54A32D192ED03ull;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / words, w = t - r * words;
    uint64_t tr = 0, v1 = 0, v0 = 0, s1 = 0, s0 = 0;
    if (w < cw) {
      const int64_t left = ncols - w * 64;
      const uint64_t valid = left < 64 ? (1ull << left) - 1ull : ~0ull;
      const uint64_t xv = __ldcs(x + t) & valid;
      const uint64_t base = (uint64_t)((row0 + r) * cw + w) * 64ull;
      uint64_t ones = xv;
      while (ones) {                                              // a sparse X: few ones per word
        const int b = __ffsll((long long)ones) - 1;
        ones &= ones - 1;
        const uint64_t u = draw32(k1, base + b), bit = 1ull << b;
        if (u < t_v) v1 |= bit; else if (u < t_vt) s1 |= bit; else tr |= bit;
      }
      if (q_vt > 0) {
        const uint64_t zeros = ~xv & valid;
#pragma unroll 4
        for (int q = 0; q < 32; ++q) {                            // one hash serves two neighbouring bits
          if (((zeros >> (2 * q)) & 3ull) == 0) continue;
          const uint64_t h = splitmix64(k0 + (base >> 1) + (uint64_t)q);
          const uint64_t ua = (uint32_t)h, ub = (uint32_t)(h >> 32);
          const uint64_t ba = 1ull << (2 * q), bb = ba << 1;
          if (zeros & ba) { if (ua < q_v) v0 |= ba; else if (ua < q_vt) s0 |= ba; }
          if (zeros & bb) { if (ub < q_v) v0 |= bb; else if (ub < q_vt) s0 |= bb; }
        }
      }
    }
    out[t] = tr;
    out[total + t] = v1;
    out[2 * total + t] = v0;
    out[3 * total + t] = s1;
    out[4 * total + t] = s0;
  }
}
// 64 x 64 bit-block transpose in registers: lane l holds rows l (a0) and l + 32 (a1) of the block and afterwards its
// columns l and l + 32 as rows.  Six block-swap stages (Hacker's Delight, 7-3): 32 inside the thread, 16 .. 1 between
// lanes by shuffles -- about 60 instructions per warp and block instead of 64 ballots per warp.
__device__ __forceinline__ void transpose64_warp(uint64_t& a0, uint64_t& a1, int lane) {
  {
    const uint64_t t = ((a0 >> 32) ^ a1) & 0x00000000FFFFFFFFull;
    a1 ^= t;
    a0 ^= t << 32;
  }
  const uint64_t masks[5] = {0x0000FFFF0000FFFFull, 0x00FF00FF00FF00FFull, 0x0F0F0F0F0F0F0F0Full, 0x3333333333333333ull,
                             0x5555555555555555ull};
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const int j = 16 >> s;
    const bool hi = lane & j;                                  // this lane holds row k | j of each swapped pair
    const uint64_t p0 = __shfl_xor_sync(0xffffffffu, a0, j), p1 = __shfl_xor_sync(0xffffffffu, a1, j);
    const uint64_t t0 = (((hi ? p0 : a0) >> j) ^ (hi ? a0 : p0)) & masks[s];
    const uint64_t t1 = (((hi ? p1 : a1) >> j) ^ (hi ? a1 : p1)) & masks[s];
    a0 ^= hi ? t0 : (t0 << j);
    a1 ^= hi ? t1 : (t1 << j);
  }
}

// bit-matrix transpose: x [rows][words] -> xt [ncols][words_t] (bit r of xt row c = bit c of x row r).  One CTA of 256
// threads per 256-row x 512-column tile (4 x 8 blocks of 64 x 64), staged through shared memory so that the loads read
// 64 B of every row and the stores write 32 B of every output row; each warp transposes 4 blocks in registers.  Only the
// words xt[c][w] with c < ncols and 64 w < rows are written.
constexpr int kTransposeRowBlocks = 4, kTransposeColWords = 8;
__global__ void __launch_bounds__(256) transpose_bits_kernel(const uint64_t* __restrict__ x, int64_t rows, int64_t ncols,
                                                             int64_t words, uint64_t* __restrict__ xt, int64_t words_t) {
  constexpr int RB = kTransposeRowBlocks, CW = kTransposeColWords;
  __shared__ uint64_t tin[RB * 64][CW + 1];                    // +1: the column reads below hit distinct banks
  __shared__ uint64_t tout[CW * 64][RB + 1];
  const int t = threadIdx.x, lane = t & 31, wp = t >> 5;
  const int64_t w0 = (int64_t)blockIdx.x * CW, r0 = (int64_t)blockIdx.y * (RB * 64);
  const int64_t wn = (ncols + 63) >> 6;                        // words of a row that hold columns < ncols
#pragma unroll
  for (int q = 0; q < RB * 64 * CW / 256; ++q) {
    const int i = t + 256 * q, rr = i / CW, cw = i % CW;
    const int64_t r = r0 + rr, w = w0 + cw;
    tin[rr][cw] = (r < rows && w < wn) ? x[r * words + w] : 0ull;
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < RB * CW / 8; ++q) {
    const int blk = wp + 8 * q, rb = blk % RB, cw = blk / RB;
    uint64_t a0 = tin[rb * 64 + lane][cw], a1 = tin[rb * 64 + 32 + lane][cw];
    transpose64_warp(a0, a1, lane);
    tout[cw * 64 + lane][rb] = a0;
    tout[cw * 64 + 32 + lane][rb] = a1;
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < CW * 64 * RB / 256; ++q) {
    const int i = t + 256 * q, cc = i / RB, rb = i % RB;
    const int64_t col = w0 * 64 + cc, wt = (int64_t)blockIdx.y * RB + rb;
    if (col < ncols && wt * 64 < rows && wt < words_t) xt[col * words_t + wt] = tout[cc][rb];
  }
}

static inline int row_stream_grid() { return num_sms() * 8; }

}  // namespace bmf

using namespace bmf;

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" int bmf_fill_zero(void* ptr, int64_t bytes, bmf_stream_t stream) {
  BMF_REQUIRE(ptr != nullptr && bytes >= 0, "bmf_fill_zero: null pointer or negative size");
  return check_cuda(cudaMemsetAsync(ptr, 0, (size_t)bytes, as_stream(stream)), "bmf_fill_zero");
}

extern "C" int bmf_pack_csr(const int64_t* indptr, const int32_t* indices, int64_t m, int64_t n,
                            int transposed, uint64_t* bits, int64_t words, bmf_stream_t stream) {
  BMF_REQUIRE(indptr && bits && m >= 0 && n >= 0, "bmf_pack_csr: null pointer or negative shape");
  BMF_REQUIRE(words % 2 == 0 && words * 64 >= (transposed ? m : n), "bmf_pack_csr: words must be even and cover the row");
  if (m == 0) return 0;
  BMF_REQUIRE(indices != nullptr, "bmf_pack_csr: null indices");
  const int64_t blocks = ceil_div(m, 8);
  pack_csr_kernel<<<(unsigned)(blocks > 1048576 ? 1048576 : blocks), 256, 0, as_stream(stream)>>>(
      indptr, indices, m, transposed, reinterpret_cast<unsigned long long*>(bits), words);
  BMF_LAUNCH_CHECK("bmf_pack_csr");
  return 0;
}

extern "C" int bmf_expand_bits_i8(const uint64_t* bits, const uint64_t* mask_bits, int64_t rows, int64_t ncols,
                                  int64_t words, int8_t one, int8_t zero, int8_t masked, int8_t* plane,
                                  int64_t rows_pad, int64_t ld, bmf_stream_t stream) {
  BMF_REQUIRE(bits && plane, "bmf_expand_bits_i8: null pointer");
  BMF_REQUIRE(ld % 128 == 0 && ld >= ncols && rows_pad >= rows && rows >= 0, "bmf_expand_bits_i8: bad ld / rows_pad");
  if (rows_pad == 0) return 0;
  const int64_t total = rows_pad * (ld >> 4);
  int64_t blocks = ceil_div(total, 256);
  if (blocks > (int64_t)num_sms() * 64) blocks = (int64_t)num_sms() * 64;
  expand_bits_i8_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(bits, mask_bits, rows, ncols, words, one,
                                                                       zero, masked, plane, rows_pad, ld);
  BMF_LAUNCH_CHECK("bmf_expand_bits_i8");
  return 0;
}

extern "C" int bmf_assoc_counts_popc(const uint64_t* xt_bits, int64_t n, int64_t words_m, int32_t* cnt,
                                     int64_t ldc, bmf_stream_t stream) {
  BMF_REQUIRE(xt_bits && cnt && n > 0 && ldc >= n && words_m > 0, "bmf_assoc_counts_popc: bad arguments");
  dim3 grid((unsigned)ceil_div(n, PT), (unsigned)ceil_div(n, PT));
  assoc_counts_popc_kernel<<<grid, 256, 0, as_stream(stream)>>>(xt_bits, n, words_m, cnt, ldc);
  BMF_LAUNCH_CHECK("bmf_assoc_counts_popc");
  return 0;
}

extern "C" int bmf_basis_threshold(const int32_t* cnt, int64_t ldc, int64_t n, double tau,
                                   uint64_t* basis_bits, int64_t words, int8_t* cand_plane, int64_t ld,
                                   uint8_t* alive, int32_t* row_pop, bmf_stream_t stream) {
  BMF_REQUIRE(cnt && basis_bits && alive && n > 0 && ldc >= n, "bmf_basis_threshold: bad arguments");
  BMF_REQUIRE(words % 2 == 0 && words * 64 >= n, "bmf_basis_threshold: words must be even and cover n");
  BMF_REQUIRE(cand_plane == nullptr || (ld % 128 == 0 && ld >= n), "bmf_basis_threshold: bad ld");
  int64_t blocks = ceil_div(n, 8);
  basis_threshold_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(cnt, ldc, n, 0, n, 0, tau, basis_bits, words,
                                                                        cand_plane, ld, alive, row_pop);
  BMF_LAUNCH_CHECK("bmf_basis_threshold");
  return 0;
}

extern "C" int bmf_basis_threshold_rows(const int32_t* cnt_rows, int64_t ldc, int64_t n, int64_t row0, int64_t nrows,
                                        int32_t symmetric, double tau, uint64_t* basis_rows, int64_t words,
                                        uint8_t* alive_rows, int32_t* pop_rows, bmf_stream_t stream) {
  BMF_REQUIRE(cnt_rows && basis_rows && alive_rows && n > 0 && ldc >= n, "bmf_basis_threshold_rows: bad arguments");
  BMF_REQUIRE(row0 >= 0 && nrows >= 0 && row0 + nrows <= n, "bmf_basis_threshold_rows: row window outside the matrix");
  BMF_REQUIRE(words % 2 == 0 && words * 64 >= n, "bmf_basis_threshold_rows: words must be even and cover n");
  BMF_REQUIRE(!symmetric || row0 == 0, "bmf_basis_threshold_rows: the symmetric read needs the whole matrix (row0 = 0)");
  if (nrows == 0) return 0;
  const char* e = getenv("BMF_BASIS_TILES");                    // 0: the row-per-warp kernel on the symmetric matrix (A/B)
  const int64_t nb = ceil_div(n, BT);
  if (symmetric && nrows == n && nb <= 65535 && !(e != nullptr && e[0] == '0')) {
    if (pop_rows != nullptr) {                                  // the |b_i| output doubles as scratch for the minimal counts
      assoc_min_counts_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, as_stream(stream)>>>(cnt_rows, ldc, n, tau, pop_rows);
      BMF_LAUNCH_CHECK("bmf_basis_threshold_rows");
    }
    basis_threshold_tile_kernel<<<dim3((unsigned)nb, (unsigned)nb), 256, 0, as_stream(stream)>>>(cnt_rows, ldc, n, tau, pop_rows,
                                                                                               basis_rows, words);
    BMF_LAUNCH_CHECK("bmf_basis_threshold_rows");
    basis_rows_finish_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, as_stream(stream)>>>(basis_rows, n, words, nb, alive_rows,
                                                                                     pop_rows);
    BMF_LAUNCH_CHECK("bmf_basis_threshold_rows");
    return 0;
  }
  int64_t blocks = ceil_div(nrows, 8);
  basis_threshold_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(cnt_rows, ldc, n, row0, nrows, symmetric ? 1 : 0,
                                                                        tau, basis_rows, words, nullptr, 0, alive_rows,
                                                                        pop_rows);
  BMF_LAUNCH_CHECK("bmf_basis_threshold_rows");
  return 0;
}

extern "C" int bmf_cover_score_popc(const uint64_t* x_bits, const uint64_t* c_bits, int64_t m, int64_t n,
                                    int64_t words, const uint64_t* basis_bits, const uint8_t* alive,
                                    const int32_t* tp_old, const int32_t* fp_old, int32_t wa, int32_t wb,
                                    double w_fp, double w_fn, int64_t* gain_p, int64_t* gain_n,
                                    bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && c_bits && basis_bits && alive && gain_p, "bmf_cover_score_popc: null pointer");
  BMF_REQUIRE(m > 0 && n > 0 && words * 64 >= n, "bmf_cover_score_popc: bad shape");
  const bool integer_mode = (wa | wb) != 0;
  BMF_REQUIRE(integer_mode || (tp_old && fp_old && gain_n), "bmf_cover_score_popc: general mode needs tp_old/fp_old/gain_n");
  BMF_REQUIRE(wa >= 0 && wb >= 0 && wa <= 127 && wb <= 127, "bmf_cover_score_popc: integer weights out of range");
  int rc = check_cuda(cudaMemsetAsync(gain_p, 0, sizeof(int64_t) * n, as_stream(stream)), "bmf_cover_score_popc");
  if (rc) return rc;
  if (!integer_mode) {
    rc = check_cuda(cudaMemsetAsync(gain_n, 0, sizeof(int64_t) * n, as_stream(stream)), "bmf_cover_score_popc");
    if (rc) return rc;
  }
  const int64_t cand_tiles = ceil_div(n, PT), row_tiles = ceil_div(m, PT);
  int64_t splits = ceil_div((int64_t)num_sms() * 8, cand_tiles);
  if (splits > row_tiles) splits = row_tiles;
  if (splits < 1) splits = 1;
  if (splits > 65535) splits = 65535;
  dim3 grid((unsigned)cand_tiles, (unsigned)splits);
  cover_score_popc_kernel<<<grid, 256, 0, as_stream(stream)>>>(
      x_bits, c_bits, m, n, words, basis_bits, alive, tp_old, fp_old, wa, wb, -w_fp, w_fn,
      reinterpret_cast<unsigned long long*>(gain_p), reinterpret_cast<unsigned long long*>(gain_n));
  BMF_LAUNCH_CHECK("bmf_cover_score_popc");
  return 0;
}

extern "C" int bmf_select_first_max(const int64_t* gain_p, const int64_t* gain_n, const uint8_t* alive,
                                    int64_t n, int32_t wa, int32_t wb, int64_t base_int, double scale,
                                    double w_fp, double w_fn, int64_t tp_tot, int64_t fp_tot,
                                    double best_score, int64_t* record, bmf_stream_t stream) {
  BMF_REQUIRE(gain_p && alive && record && n > 0, "bmf_select_first_max: bad arguments");
  BMF_REQUIRE((wa | wb) != 0 || gain_n != nullptr, "bmf_select_first_max: general mode needs gain_n");
  select_first_max_kernel<<<1, 1024, 0, as_stream(stream)>>>(gain_p, gain_n, alive, n, wa, wb, base_int, scale,
                                                            -w_fp, w_fn, tp_tot, fp_tot, best_score, record);
  BMF_LAUNCH_CHECK("bmf_select_first_max");
  return 0;
}

static int launch_cover_apply(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                              const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                              int32_t* fp_old, int32_t wa, int32_t wb, double w_fp, double w_fn, int8_t* rows_plane,
                              int64_t ld, int covered_value, int pq_layout, uint64_t* u_bits, int64_t* totals,
                              bmf_stream_t stream, const ApplyExtra& ex = ApplyExtra{}) {
  BMF_REQUIRE(x_bits && c_bits && basis_bits && alive && winner && tp_old && fp_old && u_bits && totals,
              "bmf_cover_apply: null pointer");
  BMF_REQUIRE(m > 0 && n > 0 && words % 2 == 0 && words * 64 >= n, "bmf_cover_apply: bad shape");
  BMF_REQUIRE(rows_plane == nullptr || (ld % 128 == 0 && ld * (pq_layout >= 2 ? 2 : 1) >= words * 64),
              "bmf_cover_apply: ld must cover words*64");
  const int depth = apply_ring_depth(words);
  if (depth >= 2) {
    const size_t smem = (size_t)words * 8 + (size_t)APPLY_RING_WARPS * depth * 2 * words * 8 + APPLY_RING_WARPS * APPLY_RING_DEPTH_MAX * 8;
    int64_t ctas = ceil_div(m, APPLY_RING_WARPS);
    if (ctas > num_sms()) ctas = num_sms();
    int rc = check_cuda(cudaFuncSetAttribute(cover_apply_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                        "bmf_cover_apply");
    if (rc) return rc;
    cover_apply_ring_kernel<<<(unsigned)ctas, APPLY_RING_THREADS, smem, as_stream(stream)>>>(
        x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, wa, wb, -w_fp, w_fn, rows_plane,
        ld, covered_value, pq_layout, reinterpret_cast<unsigned long long*>(u_bits),
        reinterpret_cast<unsigned long long*>(totals), ex, depth);
    BMF_LAUNCH_CHECK("bmf_cover_apply");
    return 0;
  }
  int64_t blocks = ceil_div(m, 8);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  cover_apply_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, wa, wb, -w_fp, w_fn, rows_plane,
      ld, covered_value, pq_layout, reinterpret_cast<unsigned long long*>(u_bits),
      reinterpret_cast<unsigned long long*>(totals), ex);
  BMF_LAUNCH_CHECK("bmf_cover_apply");
  return 0;
}

extern "C" int bmf_greedy_select(const int64_t* gain_p, const int64_t* gain_n, const int64_t* tail, int64_t* tail_zero,
                                 uint8_t* alive, int64_t n, int32_t wa, int32_t wb, double scale, double w_fp,
                                 double w_fn, int32_t first, int64_t* state, int64_t* table_row, int64_t* prev_row,
                                 int64_t* record, int32_t* nused, bmf_stream_t stream) {
  BMF_REQUIRE(gain_p && alive && state && record && n > 0, "bmf_greedy_select: bad arguments");
  BMF_REQUIRE((wa | wb) != 0 || gain_n != nullptr, "bmf_greedy_select: general mode needs gain_n");
  BMF_REQUIRE(prev_row == nullptr || tail != nullptr, "bmf_greedy_select: prev_row needs the tail counters");
  greedy_select_kernel<<<1, 1024, 0, as_stream(stream)>>>(
      gain_p, gain_n, reinterpret_cast<const long long*>(tail), reinterpret_cast<long long*>(tail_zero), alive, n, wa,
      wb, scale, -w_fp, w_fn, first, reinterpret_cast<long long*>(state), reinterpret_cast<long long*>(table_row),
      reinterpret_cast<long long*>(prev_row), reinterpret_cast<long long*>(record), nused);
  BMF_LAUNCH_CHECK("bmf_greedy_select");
  return 0;
}

extern "C" int bmf_cover_apply_compact_mapped(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                              const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner,
                                              int32_t* tp_old, int32_t* fp_old, int32_t wa, int32_t wb, int32_t kind,
                                              int32_t v_one, int32_t v_zero, int32_t v_covered, uint8_t* comp_old,
                                              uint8_t* comp_new, int64_t comp_ld, int64_t comp_cap, int32_t tile_rows,
                                              int32_t* nused, uint64_t* u_bits, uint64_t* u_words, int64_t kw,
                                              int32_t factor_bit, uint64_t* vt_row, const int32_t* col_pos, int64_t* totals,
                                              bmf_stream_t stream) {
  BMF_REQUIRE((wa | wb) != 0, "bmf_cover_apply_compact: integer weights only");
  BMF_REQUIRE(col_pos == nullptr || (kind == 1 && v_zero == 0),
              "bmf_cover_apply_compact: a column map needs kind 1 (E2M1) and a zero code of 0");
  BMF_REQUIRE(kind == 0 || ((kind == 1 || kind == 2) && comp_old && comp_new && nused && comp_cap > 0 && tile_rows > 0),
              "bmf_cover_apply_compact: kind 1 (E2M1) / 2 (int8) needs the compact planes and the counter");
  BMF_REQUIRE(kind == 0 || (comp_ld % 128 == 0 && comp_ld * (kind == 1 ? 2 : 1) >= words * 64),
              "bmf_cover_apply_compact: comp_ld must cover words*64 columns");
  BMF_REQUIRE(kind != 1 || ((v_one | v_zero | v_covered) & ~7) == 0, "bmf_cover_apply_compact: E2M1 codes are 0..7");
  BMF_REQUIRE(u_words == nullptr || (kw > 0 && factor_bit >= 0 && factor_bit < kw * 64),
              "bmf_cover_apply_compact: factor_bit outside the usage words");
  ApplyExtra ex = {};
  ex.comp_old = comp_old; ex.comp_new = comp_new; ex.comp_ld = comp_ld; ex.comp_cap = comp_cap; ex.nused = nused;
  ex.comp_kind = kind; ex.v_one = v_one; ex.v_zero = v_zero; ex.v_cov = v_covered;
  ex.u_words = u_words; ex.kw = kw; ex.factor_bit = factor_bit; ex.vt_row = vt_row;
  ex.col_pos = col_pos;
  int rc = launch_cover_apply(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, wa, wb, 0.0, 0.0,
                              nullptr, 0, 0, 0, u_bits, totals, stream, ex);
  if (rc || kind == 0) return rc;
  compact_tail_zero_kernel<<<64, 256, 0, as_stream(stream)>>>(comp_old, comp_new, comp_ld, comp_cap, nused, tile_rows);
  BMF_LAUNCH_CHECK("bmf_cover_apply_compact");
  return 0;
}

extern "C" int bmf_cover_apply_compact(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                       const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner,
                                       int32_t* tp_old, int32_t* fp_old, int32_t wa, int32_t wb, int32_t kind,
                                       int32_t v_one, int32_t v_zero, int32_t v_covered, uint8_t* comp_old,
                                       uint8_t* comp_new, int64_t comp_ld, int64_t comp_cap, int32_t tile_rows,
                                       int32_t* nused, uint64_t* u_bits, uint64_t* u_words, int64_t kw,
                                       int32_t factor_bit, uint64_t* vt_row, int64_t* totals, bmf_stream_t stream) {
  return bmf_cover_apply_compact_mapped(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, wa, wb, kind,
                                        v_one, v_zero, v_covered, comp_old, comp_new, comp_ld, comp_cap, tile_rows, nused,
                                        u_bits, u_words, kw, factor_bit, vt_row, nullptr, totals, stream);
}

extern "C" int bmf_cover_apply_compact_general(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                               const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner,
                                               int32_t* tp_old, int32_t* fp_old, double w_fp, double w_fn, int32_t kind,
                                               uint8_t* comp_old, uint8_t* comp_new, int64_t comp_ld, int64_t comp_cap,
                                               int32_t* nused, int32_t* comp_tp_old, int32_t* comp_fp_old,
                                               int32_t* comp_tp_new, int32_t* comp_fp_new, uint64_t* u_bits,
                                               int64_t* totals, bmf_stream_t stream) {
  BMF_REQUIRE(kind == 0 || ((kind == 3 || kind == 4) && comp_old && comp_new && nused && comp_cap > 0 && comp_tp_old &&
                            comp_fp_old && comp_tp_new && comp_fp_new),
              "bmf_cover_apply_compact_general: kind 3 (E2M1 P/Q) / 4 (int8 P/Q) needs the compact planes, counters and counter");
  BMF_REQUIRE(kind == 0 || (comp_ld % 128 == 0 && comp_ld * (kind == 3 ? 2 : 1) >= words * 64),
              "bmf_cover_apply_compact_general: comp_ld must cover words*64 columns");
  ApplyExtra ex = {};
  ex.comp_old = comp_old; ex.comp_new = comp_new; ex.comp_ld = comp_ld; ex.comp_cap = comp_cap; ex.nused = nused;
  ex.comp_kind = kind;
  ex.comp_tp_old = comp_tp_old; ex.comp_fp_old = comp_fp_old; ex.comp_tp_new = comp_tp_new; ex.comp_fp_new = comp_fp_new;
  int rc = launch_cover_apply(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, 0, 0, w_fp, w_fn,
                              nullptr, 0, 0, 0, u_bits, totals, stream, ex);
  if (rc || kind == 0) return rc;
  compact_tail_zero_pq_kernel<<<64, 256, 0, as_stream(stream)>>>(comp_old, comp_new, comp_ld, comp_cap, nused,
                                                               kind == 3 ? 120 : 128);
  BMF_LAUNCH_CHECK("bmf_cover_apply_compact_general");
  return 0;
}

extern "C" int bmf_cover_apply(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                               const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner,
                               int32_t* tp_old, int32_t* fp_old, int32_t wa, int32_t wb, double w_fp,
                               double w_fn, int8_t* rows_plane, int64_t ld, int8_t covered_value, uint64_t* u_bits,
                               int64_t* totals, bmf_stream_t stream) {
  return launch_cover_apply(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, wa, wb, w_fp,
                            w_fn, rows_plane, ld, (int)covered_value, 0, u_bits, totals, stream);
}

extern "C" int bmf_cover_apply_general(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                       const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner,
                                       int32_t* tp_old, int32_t* fp_old, double w_fp, double w_fn, int8_t* pq_plane,
                                       int64_t ld, uint64_t* u_bits, int64_t* totals, bmf_stream_t stream) {
  BMF_REQUIRE(pq_plane != nullptr, "bmf_cover_apply_general: null pq_plane");
  return launch_cover_apply(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, 0, 0, w_fp,
                            w_fn, pq_plane, ld, 0, 1, u_bits, totals, stream);
}

extern "C" int bmf_cover_apply_f4_mapped(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                         const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                                         int32_t* fp_old, int32_t wa, int32_t wb, uint8_t* rows_plane, int64_t ld_bytes,
                                         int32_t covered_code, const int32_t* col_pos, uint64_t* u_bits, int64_t* totals,
                                         bmf_stream_t stream) {
  BMF_REQUIRE(rows_plane != nullptr && covered_code >= 0 && covered_code <= 7, "bmf_cover_apply_f4: bad plane / code");
  BMF_REQUIRE((wa | wb) != 0, "bmf_cover_apply_f4: integer weights only");
  ApplyExtra ex = {};
  ex.col_pos = col_pos;
  return launch_cover_apply(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, wa, wb, 0.0, 0.0,
                            reinterpret_cast<int8_t*>(rows_plane), ld_bytes, covered_code, 2, u_bits, totals, stream, ex);
}

extern "C" int bmf_cover_apply_f4(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                  const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                                  int32_t* fp_old, int32_t wa, int32_t wb, uint8_t* rows_plane, int64_t ld_bytes,
                                  int32_t covered_code, uint64_t* u_bits, int64_t* totals, bmf_stream_t stream) {
  return bmf_cover_apply_f4_mapped(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, wa, wb, rows_plane,
                                   ld_bytes, covered_code, nullptr, u_bits, totals, stream);
}

extern "C" int bmf_cover_apply_f4_general(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                          const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner,
                                          int32_t* tp_old, int32_t* fp_old, double w_fp, double w_fn, uint8_t* pq_plane,
                                          int64_t ld_bytes, uint64_t* u_bits, int64_t* totals, bmf_stream_t stream) {
  BMF_REQUIRE(pq_plane != nullptr, "bmf_cover_apply_f4_general: null pq_plane");
  return launch_cover_apply(x_bits, c_bits, m, n, words, basis_bits, alive, winner, tp_old, fp_old, 0, 0, w_fp, w_fn,
                            reinterpret_cast<int8_t*>(pq_plane), ld_bytes, 0, 3, u_bits, totals, stream);
}

extern "C" int bmf_expand_bits_pq_f4(const uint64_t* x_bits, const uint64_t* c_bits, int64_t rows, int64_t ncols,
                                     int64_t words, uint8_t* pq_plane, int64_t ld_bytes, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && c_bits && pq_plane, "bmf_expand_bits_pq_f4: null pointer");
  BMF_REQUIRE(rows > 0 && ld_bytes % 128 == 0 && ld_bytes * 2 >= ncols && words * 64 >= ncols, "bmf_expand_bits_pq_f4: bad shape / ld");
  const int64_t plane_rows = 2 * ceil_div(rows, 120) * 120;
  const int64_t total = plane_rows * (ld_bytes >> 4);
  int64_t blocks = ceil_div(total, 256);
  if (blocks > (int64_t)num_sms() * 64) blocks = (int64_t)num_sms() * 64;
  expand_bits_pq_f4_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(x_bits, c_bits, rows, ncols, words, pq_plane,
                                                                          plane_rows, ld_bytes);
  BMF_LAUNCH_CHECK("bmf_expand_bits_pq_f4");
  return 0;
}

extern "C" int bmf_e2m1_code(int32_t value) {
  switch (value) {
    case 0: return 0;
    case 1: return 2;
    case 2: return 4;
    case 3: return 5;
    case 4: return 6;
    case 6: return 7;
    default: return -1;
  }
}

extern "C" int bmf_expand_bits_f4_mapped(const uint64_t* bits, const uint64_t* mask_bits, int64_t rows, int64_t ncols,
                                         int64_t words, int32_t one, int32_t zero, int32_t masked, const int32_t* row_src,
                                         const int32_t* col_pos, uint8_t* plane, int64_t rows_pad, int64_t ld_bytes,
                                         bmf_stream_t stream) {
  BMF_REQUIRE(bits && plane, "bmf_expand_bits_f4: null pointer");
  BMF_REQUIRE(ld_bytes % 128 == 0 && ld_bytes * 2 >= ncols && rows_pad >= rows && rows >= 0, "bmf_expand_bits_f4: bad ld / rows_pad");
  BMF_REQUIRE(((one | zero | masked) & ~7) == 0, "bmf_expand_bits_f4: codes must be non-negative E2M1 bit patterns (0..7)");
  if (rows_pad == 0) return 0;
  if (row_src != nullptr || col_pos != nullptr) {
    BMF_REQUIRE(zero == 0, "bmf_expand_bits_f4_mapped: the zero code must be 0");
    constexpr int64_t kSmemBudget = 200 * 1024;
    BMF_REQUIRE(ld_bytes <= kSmemBudget, "bmf_expand_bits_f4_mapped: a plane row must fit in shared memory (ld_bytes <= 204800)");
    const int64_t warps = std::min<int64_t>(8, kSmemBudget / ld_bytes);
    const int smem = (int)(warps * ld_bytes);
    int rc = check_cuda(cudaFuncSetAttribute(expand_bits_f4_mapped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem),
                        "bmf_expand_bits_f4_mapped");
    if (rc) return rc;
    int64_t blocks = ceil_div(rows_pad, warps);
    if (blocks > (int64_t)num_sms() * 8) blocks = (int64_t)num_sms() * 8;
    expand_bits_f4_mapped_kernel<<<(unsigned)blocks, (unsigned)(32 * warps), smem, as_stream(stream)>>>(
        bits, mask_bits, rows, ncols, words, (uint32_t)one, (uint32_t)masked, row_src, col_pos, plane, rows_pad, ld_bytes);
    BMF_LAUNCH_CHECK("bmf_expand_bits_f4_mapped");
    return 0;
  }
  int64_t blocks = ceil_div(rows_pad, 8);
  if (blocks > (int64_t)num_sms() * 8) blocks = (int64_t)num_sms() * 8;
  expand_bits_f4_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(bits, mask_bits, rows, ncols, words, (uint32_t)one,
                                                                       (uint32_t)zero, (uint32_t)masked, plane, rows_pad,
                                                                       ld_bytes);
  BMF_LAUNCH_CHECK("bmf_expand_bits_f4");
  return 0;
}

extern "C" int bmf_expand_bits_f4(const uint64_t* bits, const uint64_t* mask_bits, int64_t rows, int64_t ncols,
                                  int64_t words, int32_t one, int32_t zero, int32_t masked, uint8_t* plane,
                                  int64_t rows_pad, int64_t ld_bytes, bmf_stream_t stream) {
  return bmf_expand_bits_f4_mapped(bits, mask_bits, rows, ncols, words, one, zero, masked, nullptr, nullptr, plane, rows_pad,
                                   ld_bytes, stream);
}

extern "C" int bmf_bits_first_set(const uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, const int32_t* row_rank,
                                  int32_t* row_first, int32_t* col_first, bmf_stream_t stream) {
  BMF_REQUIRE(bits && rows >= 0 && ncols >= 0 && words * 64 >= ncols, "bmf_bits_first_set: bad bits / shape");
  BMF_REQUIRE(col_first == nullptr || row_rank != nullptr, "bmf_bits_first_set: col_first needs row_rank");
  if (rows == 0) return 0;
  int64_t blocks = ceil_div(rows, 8);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  bits_first_set_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(bits, rows, ncols, words, row_rank, row_first,
                                                                        col_first);
  BMF_LAUNCH_CHECK("bmf_bits_first_set");
  return 0;
}

extern "C" int bmf_expand_bits_pq(const uint64_t* x_bits, const uint64_t* c_bits, int64_t rows, int64_t ncols,
                                  int64_t words, int8_t* pq_plane, int64_t ld, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && c_bits && pq_plane, "bmf_expand_bits_pq: null pointer");
  BMF_REQUIRE(rows > 0 && ld % 128 == 0 && ld >= ncols && words * 64 >= ncols, "bmf_expand_bits_pq: bad shape / ld");
  const int64_t plane_rows = 2 * ceil_div(rows, 128) * 128;
  const int64_t total = plane_rows * (ld >> 4);
  int64_t blocks = ceil_div(total, 256);
  if (blocks > (int64_t)num_sms() * 64) blocks = (int64_t)num_sms() * 64;
  expand_bits_pq_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(x_bits, c_bits, rows, ncols, words, pq_plane,
                                                                       plane_rows, ld);
  BMF_LAUNCH_CHECK("bmf_expand_bits_pq");
  return 0;
}

// The product (x == nullptr) or the residual x AND NOT product (RESIDUAL) in the panel-list form (chunks > 0: k <= 64,
// kw == 1) or the row-stream form (chunks == 0).
template <bool RESIDUAL>
static int launch_product(const uint64_t* x, const uint64_t* u_words, int64_t m, int64_t kw, const uint64_t* vt_bits,
                          int64_t k, int64_t words, int chunks, uint64_t* out, cudaStream_t st, const char* who) {
  if (chunks == 0) {
    int64_t blocks = ceil_div(m, 8);
    if (blocks > row_stream_grid()) blocks = row_stream_grid();
    bool_product_kernel<RESIDUAL><<<(unsigned)blocks, 256, 0, st>>>(u_words, m, kw, vt_bits, words, x, out);
    return check_cuda(cudaGetLastError(), who);
  }
  const size_t smem = (size_t)k * chunks * CH_PAIRS * 16;
  const int64_t max_splits = ceil_div(m, 32 * (PRODUCT_THREADS / 32));
  int ctas = 0;
  const PanelGrid pg = make_panel_grid(words >> 1, chunks * CH_PAIRS, max_splits, &ctas);
  unsigned int* sched = (panel_dynamic() && pg.panels <= 64 && m < (1ll << 36)) ? stream_counters(st) : nullptr;
  int rc = 0;
  if (sched != nullptr) {
    rc = check_cuda(cudaMemsetAsync(sched, 0, 64 * sizeof(unsigned int), st), who);
    if (rc) return rc;
    rc = check_cuda(cudaFuncSetAttribute(bool_product_panel_list_kernel<true, RESIDUAL>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), who);
    if (rc) return rc;
    bool_product_panel_list_kernel<true, RESIDUAL><<<ctas, PRODUCT_THREADS, smem, st>>>(
        u_words, m, vt_bits, k, words, chunks, product_store_mode(), pg, sched, x, out);
  } else {
    rc = check_cuda(cudaFuncSetAttribute(bool_product_panel_list_kernel<false, RESIDUAL>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), who);
    if (rc) return rc;
    bool_product_panel_list_kernel<false, RESIDUAL><<<ctas, PRODUCT_THREADS, smem, st>>>(
        u_words, m, vt_bits, k, words, chunks, product_store_mode(), pg, nullptr, x, out);
  }
  return check_cuda(cudaGetLastError(), who);
}

extern "C" int bmf_bool_product(const uint64_t* u_words, int64_t m, int64_t kw, const uint64_t* vt_bits,
                                int64_t k, int64_t words, uint64_t* pd_bits, bmf_stream_t stream) {
  BMF_REQUIRE(u_words && pd_bits && m > 0 && kw > 0 && k >= 0 && k <= kw * 64, "bmf_bool_product: bad arguments");
  BMF_REQUIRE(words > 0 && words % 2 == 0 && (k == 0 || vt_bits), "bmf_bool_product: bad words / vt_bits");
  const int chunks = panel_disabled() ? 0 : panel_chunks_for(k, kw, words);
  if (chunks > 0 && !(panel_lists() && panel_rowmap() == 0)) {
    const int panel_pairs = chunks * CH_PAIRS;
    const size_t smem = (size_t)k * panel_pairs * 16;
    const int64_t max_splits = ceil_div(m, 32 * (PRODUCT_THREADS / 32));
    int ctas = 0;
    const PanelGrid pg = make_panel_grid(words >> 1, panel_pairs, max_splits, &ctas);
    int rc = check_cuda(cudaFuncSetAttribute(bool_product_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem), "bmf_bool_product");
    if (rc) return rc;
    bool_product_panel_kernel<<<ctas, PRODUCT_THREADS, smem, as_stream(stream)>>>(u_words, m, vt_bits, k, words, chunks,
                                                                                panel_rowmap(), product_store_mode(), pg,
                                                                                pd_bits);
    BMF_LAUNCH_CHECK("bmf_bool_product");
    return 0;
  }
  return launch_product<false>(nullptr, u_words, m, kw, vt_bits, k, words, chunks, pd_bits, as_stream(stream),
                               "bmf_bool_product");
}

extern "C" int bmf_residual_factors(const uint64_t* x_bits, int64_t m, int64_t words, const uint64_t* u_words, int64_t kw,
                                    const uint64_t* vt_bits, int64_t k, uint64_t* out_bits, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && u_words && out_bits && m > 0 && kw > 0 && k >= 0 && k <= kw * 64,
              "bmf_residual_factors: bad arguments");
  BMF_REQUIRE(words > 0 && words % 2 == 0 && (k == 0 || vt_bits), "bmf_residual_factors: bad words / vt_bits");
  BMF_REQUIRE(out_bits != x_bits, "bmf_residual_factors: out_bits must not alias x_bits");
  const int chunks = panel_disabled() ? 0 : panel_chunks_for(k, kw, words);
  return launch_product<true>(x_bits, u_words, m, kw, vt_bits, k, words, chunks, out_bits, as_stream(stream),
                              "bmf_residual_factors");
}

template <bool FROM_FACTORS>
static int launch_confusion(const uint64_t* gt_bits, const uint64_t* pd_bits, int64_t m, int64_t words,
                            const uint64_t* u_words, int64_t kw, const uint64_t* vt_bits, int64_t k, int64_t gt_ones,
                            int64_t* counts, int32_t* row_tp, int32_t* row_fp, cudaStream_t st, const char* who) {
  int rc = check_cuda(cudaMemsetAsync(counts, 0, 3 * sizeof(int64_t), st), who);
  if (rc) return rc;
  unsigned long long* c = reinterpret_cast<unsigned long long*>(counts);
  if (FROM_FACTORS && row_tp == nullptr && row_fp == nullptr && !panel_disabled()) {
    const int chunks = panel_chunks_for(k, kw, words);
    if (chunks > 0) {
      const int panel_pairs = chunks * CH_PAIRS;
      const int depth = confusion_ring_depth(k, chunks);
      const size_t smem = confusion_panel_smem(k, chunks, depth);
      const int64_t max_splits = ceil_div(ceil_div(m, 32), PANEL_WARPS);
      int ctas = 0;
      const PanelGrid pg = make_panel_grid(words >> 1, panel_pairs, max_splits, &ctas);
      const int mode = confusion_count_mode();
#define BMF_CONF_LAUNCH(CG, MD)                                                                                      \
  do {                                                                                                               \
    rc = check_cuda(cudaFuncSetAttribute(confusion_panel_kernel<CG, MD>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                         (int)smem), who);                                                           \
    if (rc) return rc;                                                                                               \
    confusion_panel_kernel<CG, MD><<<ctas, PANEL_THREADS, smem, st>>>(gt_bits, m, words, u_words, vt_bits, k, chunks,  \
                                                                      depth, pg, c);                                 \
  } while (0)
#define BMF_CONF_LIST_LAUNCH(CG, MD)                                                                                      \
  do {                                                                                                                    \
    rc = check_cuda(cudaFuncSetAttribute(confusion_panel_list_kernel<CG, MD>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                         (int)smem), who);                                                                \
    if (rc) return rc;                                                                                                    \
    confusion_panel_list_kernel<CG, MD><<<ctas, PANEL_THREADS, smem, st>>>(gt_bits, nullptr, m, words, u_words, vt_bits, k, chunks,  \
                                                                           depth, pg, c);                                 \
  } while (0)
      if (panel_lists()) {
        if (gt_ones >= 0) {
          if (mode == 0) BMF_CONF_LIST_LAUNCH(false, 0); else if (mode == 1) BMF_CONF_LIST_LAUNCH(false, 1);
          else if (mode == 2) BMF_CONF_LIST_LAUNCH(false, 2); else BMF_CONF_LIST_LAUNCH(false, 3);
        } else {
          if (mode == 0) BMF_CONF_LIST_LAUNCH(true, 0); else if (mode == 1) BMF_CONF_LIST_LAUNCH(true, 1);
          else if (mode == 2) BMF_CONF_LIST_LAUNCH(true, 2); else BMF_CONF_LIST_LAUNCH(true, 3);
        }
      } else if (gt_ones >= 0) {
        if (mode == 0) BMF_CONF_LAUNCH(false, 0); else if (mode == 1) BMF_CONF_LAUNCH(false, 1); else BMF_CONF_LAUNCH(false, 2);
      } else {
        if (mode == 0) BMF_CONF_LAUNCH(true, 0); else if (mode == 1) BMF_CONF_LAUNCH(true, 1); else BMF_CONF_LAUNCH(true, 2);
      }
#undef BMF_CONF_LAUNCH
#undef BMF_CONF_LIST_LAUNCH
      rc = check_cuda(cudaGetLastError(), who);
      if (rc) return rc;
      confusion_finalize_kernel<<<1, 1, 0, st>>>(reinterpret_cast<long long*>(counts), (long long)gt_ones);
      return check_cuda(cudaGetLastError(), who);
    }
  }
  int64_t blocks = ceil_div(m, 8);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  if (gt_ones >= 0)
    confusion_kernel<FROM_FACTORS, false><<<(unsigned)blocks, 256, 0, st>>>(gt_bits, nullptr, pd_bits, m, words, u_words, kw,
                                                                          vt_bits, c, row_tp, row_fp);
  else
    confusion_kernel<FROM_FACTORS, true><<<(unsigned)blocks, 256, 0, st>>>(gt_bits, nullptr, pd_bits, m, words, u_words, kw,
                                                                         vt_bits, c, row_tp, row_fp);
  rc = check_cuda(cudaGetLastError(), who);
  if (rc) return rc;
  confusion_finalize_kernel<<<1, 1, 0, st>>>(reinterpret_cast<long long*>(counts), (long long)gt_ones);
  return check_cuda(cudaGetLastError(), who);
}

extern "C" int bmf_confusion_factors(const uint64_t* gt_bits, int64_t m, int64_t words, const uint64_t* u_words,
                                     int64_t kw, const uint64_t* vt_bits, int64_t k, int64_t gt_ones,
                                     int64_t* counts, int32_t* row_tp, int32_t* row_fp, bmf_stream_t stream) {
  BMF_REQUIRE(gt_bits && u_words && counts && m > 0 && kw > 0 && k <= kw * 64, "bmf_confusion_factors: bad arguments");
  BMF_REQUIRE(words > 0 && words % 2 == 0 && (k == 0 || vt_bits), "bmf_confusion_factors: bad words / vt_bits");
  return launch_confusion<true>(gt_bits, nullptr, m, words, u_words, kw, vt_bits, k, gt_ones, counts, row_tp, row_fp,
                                as_stream(stream), "bmf_confusion_factors");
}

extern "C" int bmf_confusion_bits(const uint64_t* gt_bits, const uint64_t* pd_bits, int64_t m, int64_t words,
                                  int64_t gt_ones, int64_t* counts, int32_t* row_tp, int32_t* row_fp,
                                  bmf_stream_t stream) {
  BMF_REQUIRE(gt_bits && pd_bits && counts && m > 0 && words > 0 && words % 2 == 0, "bmf_confusion_bits: bad arguments");
  return launch_confusion<false>(gt_bits, pd_bits, m, words, nullptr, 0, nullptr, 0, gt_ones, counts, row_tp, row_fp,
                                 as_stream(stream), "bmf_confusion_bits");
}

// Stored-entry counts (task='prediction'): counts[0..3] = (|ones & pd|, |zeros & pd|, |ones|, |zeros|) in ONE pass,
// against a materialised prediction (FROM_FACTORS false) or the product of the factors.  The panel-list form serves
// k <= 64 when its ring holds the two segments of a row, the row-stream form everything else.
template <bool FROM_FACTORS>
static int launch_confusion_entries(const uint64_t* ones, const uint64_t* zeros, const uint64_t* pd_bits, int64_t m,
                                    int64_t words, const uint64_t* u_words, int64_t kw, const uint64_t* vt_bits, int64_t k,
                                    int64_t* counts, cudaStream_t st, const char* who) {
  int rc = check_cuda(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), st), who);
  if (rc) return rc;
  unsigned long long* c = reinterpret_cast<unsigned long long*>(counts);
  if (FROM_FACTORS && !panel_disabled()) {
    const int chunks = panel_chunks_for(k, kw, words);
    const int depth = chunks > 0 ? confusion_ring_depth(k, chunks) : 0;
    if (chunks > 0 && depth >= 2) {
      const size_t smem = confusion_panel_smem(k, chunks, depth);
      const int64_t max_splits = ceil_div(ceil_div(m, 32), PANEL_WARPS);
      int ctas = 0;
      const PanelGrid pg = make_panel_grid(words >> 1, chunks * CH_PAIRS, max_splits, &ctas);
      rc = check_cuda(cudaFuncSetAttribute(confusion_panel_list_kernel<true, 3, true>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), who);
      if (rc) return rc;
      confusion_panel_list_kernel<true, 3, true><<<ctas, PANEL_THREADS, smem, st>>>(ones, zeros, m, words, u_words, vt_bits,
                                                                                 k, chunks, depth, pg, c);
      return check_cuda(cudaGetLastError(), who);
    }
  }
  int64_t blocks = ceil_div(m, 8);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  confusion_kernel<FROM_FACTORS, true, true><<<(unsigned)blocks, 256, 0, st>>>(ones, zeros, pd_bits, m, words, u_words, kw,
                                                                             vt_bits, c, nullptr, nullptr);
  return check_cuda(cudaGetLastError(), who);
}

extern "C" int bmf_confusion_entries_bits(const uint64_t* ones, const uint64_t* zeros, const uint64_t* pd_bits, int64_t m,
                                          int64_t words, int64_t* counts, bmf_stream_t stream) {
  BMF_REQUIRE(ones && pd_bits && counts && m > 0 && words > 0 && words % 2 == 0, "bmf_confusion_entries_bits: bad arguments");
  return launch_confusion_entries<false>(ones, zeros, pd_bits, m, words, nullptr, 0, nullptr, 0, counts, as_stream(stream),
                                         "bmf_confusion_entries_bits");
}

extern "C" int bmf_confusion_entries_factors(const uint64_t* ones, const uint64_t* zeros, int64_t m, int64_t words,
                                             const uint64_t* u_words, int64_t kw, const uint64_t* vt_bits, int64_t k,
                                             int64_t* counts, bmf_stream_t stream) {
  BMF_REQUIRE(ones && u_words && counts && m > 0 && kw > 0 && k >= 0 && k <= kw * 64,
              "bmf_confusion_entries_factors: bad arguments");
  BMF_REQUIRE(words > 0 && words % 2 == 0 && (k == 0 || vt_bits), "bmf_confusion_entries_factors: bad words / vt_bits");
  return launch_confusion_entries<true>(ones, zeros, nullptr, m, words, u_words, kw, vt_bits, k, counts, as_stream(stream),
                                        "bmf_confusion_entries_factors");
}

extern "C" int bmf_bits_combine(const uint64_t* a_bits, const uint64_t* b_bits, int64_t rows, int64_t words, int op,
                                uint64_t* out_bits, bmf_stream_t stream) {
  BMF_REQUIRE(a_bits && b_bits && out_bits && rows > 0 && words > 0 && words % 2 == 0, "bmf_bits_combine: bad arguments");
  BMF_REQUIRE(op >= 0 && op <= 2, "bmf_bits_combine: op must be 0 (or), 1 (and) or 2 (and-not)");
  const int64_t pairs = rows * (words >> 1);
  int64_t blocks = ceil_div(pairs, 256);
  if (blocks > row_stream_grid() * 4) blocks = row_stream_grid() * 4;
  bits_combine_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const ulonglong2*>(a_bits), reinterpret_cast<const ulonglong2*>(b_bits), pairs, op,
      reinterpret_cast<ulonglong2*>(out_bits));
  BMF_LAUNCH_CHECK("bmf_bits_combine");
  return 0;
}

extern "C" int bmf_confusion_triplets(const int32_t* rows, const int32_t* cols, const uint8_t* gt, int64_t nnz,
                                      const uint64_t* u_words, int64_t kw, const uint64_t* v_words,
                                      int64_t* counts, bmf_stream_t stream) {
  BMF_REQUIRE(counts && kw > 0 && nnz >= 0, "bmf_confusion_triplets: bad arguments");
  if (nnz == 0) return 0;
  BMF_REQUIRE(rows && cols && gt && u_words && v_words, "bmf_confusion_triplets: null pointer");
  int64_t blocks = ceil_div(nnz, 256);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  confusion_triplets_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      rows, cols, gt, nnz, u_words, kw, v_words, reinterpret_cast<unsigned long long*>(counts));
  BMF_LAUNCH_CHECK("bmf_confusion_triplets");
  return 0;
}

extern "C" int bmf_refine_column(const uint64_t* x_bits, int64_t m, int64_t n, int64_t words, uint64_t* u_words,
                                 int64_t kw, const uint64_t* vt_bits, int64_t k, int64_t col, int32_t wa,
                                 int32_t wb, double w_fp, double w_fn, int64_t* out, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && u_words && vt_bits && out, "bmf_refine_column: null pointer");
  BMF_REQUIRE(m > 0 && n > 0 && words % 2 == 0 && words * 64 >= n && kw > 0 && k <= kw * 64, "bmf_refine_column: bad shape");
  BMF_REQUIRE(col >= 0 && col < k, "bmf_refine_column: column out of range");
  int64_t blocks = ceil_div(m, 8);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  refine_column_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      x_bits, m, n, words, u_words, kw, vt_bits, col, wa, wb, -w_fp, w_fn,
      reinterpret_cast<unsigned long long*>(out));
  BMF_LAUNCH_CHECK("bmf_refine_column");
  return 0;
}

extern "C" int bmf_refine_sweep(const uint64_t* x_bits, int64_t m, int64_t n, int64_t words, uint64_t* u_words,
                                int64_t kw, const uint64_t* vt_bits, int64_t k, int64_t col0, int64_t ncols, int32_t wa,
                                int32_t wb, double w_fp, double w_fn, int64_t* out, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && u_words && vt_bits && out, "bmf_refine_sweep: null pointer");
  BMF_REQUIRE(m > 0 && n > 0 && words % 2 == 0 && words * 64 >= n && kw > 0 && k <= kw * 64, "bmf_refine_sweep: bad shape");
  BMF_REQUIRE(col0 >= 0 && ncols >= 1 && col0 + ncols <= k, "bmf_refine_sweep: columns out of range");
  const size_t vt_bytes = (size_t)k * (size_t)words * sizeof(uint64_t);
  const size_t cnt_bytes = (size_t)ncols * 5 * sizeof(unsigned long long);
  const bool vs = vt_bytes <= 96 * 1024;                // V^T in shared memory; larger V^T is read through L1 / L2
  const int cnt_in_smem = cnt_bytes <= 32 * 1024;       // per-block column counters, else atomics straight to `out`
  const size_t smem = (vs ? vt_bytes : 0) + (cnt_in_smem ? cnt_bytes : 0);
  const void* fn = vs ? (const void*)refine_sweep_kernel<true> : (const void*)refine_sweep_kernel<false>;
  int rc = check_cuda(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "bmf_refine_sweep");
  if (rc) return rc;
  int per_sm = 0;
  rc = check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 256, smem), "bmf_refine_sweep");
  if (rc) return rc;
  int64_t blocks = ceil_div(m, 8);
  const int64_t resident = (int64_t)num_sms() * (per_sm > 0 ? per_sm : 1);
  if (blocks > resident) blocks = resident;              // every block stages V^T once: no more blocks than fit at once
  if (vs)
    refine_sweep_kernel<true><<<(unsigned)blocks, 256, smem, as_stream(stream)>>>(
        x_bits, m, words, u_words, kw, vt_bits, k, col0, ncols, wa, wb, -w_fp, w_fn, cnt_in_smem,
        reinterpret_cast<unsigned long long*>(out));
  else
    refine_sweep_kernel<false><<<(unsigned)blocks, 256, smem, as_stream(stream)>>>(
        x_bits, m, words, u_words, kw, vt_bits, k, col0, ncols, wa, wb, -w_fp, w_fn, cnt_in_smem,
        reinterpret_cast<unsigned long long*>(out));
  BMF_LAUNCH_CHECK("bmf_refine_sweep");
  return 0;
}


extern "C" int bmf_expand_scores(const uint64_t* x_bits, const uint64_t* old_bits, int64_t rows, int64_t words,
                                 const uint64_t* pattern_bits, const uint64_t* exclude_bits, double w_fp, double w_fn,
                                 double* delta, int64_t* best, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && old_bits && pattern_bits && delta, "bmf_expand_scores: null pointer");
  BMF_REQUIRE(rows > 0 && words > 0 && words % 2 == 0, "bmf_expand_scores: bad shape");
  int64_t blocks = ceil_div(rows, 8);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  expand_delta_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(x_bits, old_bits, rows, words, pattern_bits,
                                                                     exclude_bits, -w_fp, w_fn, delta);
  BMF_LAUNCH_CHECK("bmf_expand_scores");
  if (best != nullptr) {
    argmax_first_f64_kernel<<<1, 1024, 0, as_stream(stream)>>>(delta, rows, reinterpret_cast<long long*>(best));
    BMF_LAUNCH_CHECK("bmf_expand_scores");
  }
  return 0;
}

static constexpr int64_t kExpandMaxBlocks = 1024;                   // grid of the step kernels (partials: 2 x 1024 pairs)

extern "C" int bmf_expand_init(const uint64_t* x_bits, const uint64_t* old_bits, int64_t rows, int64_t n, int64_t words,
                               int64_t row0, const uint64_t* u_bits, const uint64_t* v_bits, int32_t* row_cnt,
                               int64_t* col_cnt, bmf_stream_t stream) {
  BMF_REQUIRE(u_bits && v_bits && col_cnt && (rows == 0 || (x_bits && old_bits && row_cnt)), "bmf_expand_init: null pointer");
  BMF_REQUIRE(rows >= 0 && n > 0 && words * 64 >= n && words % 2 == 0 && row0 >= 0 && row0 + rows < (1ll << 31),
              "bmf_expand_init: bad shape");
  cudaStream_t s = as_stream(stream);
  int rc = check_cuda(cudaMemsetAsync(col_cnt, 0, (size_t)(4 * n) * sizeof(int64_t), s), "bmf_expand_init");
  if (rc || rows == 0) return rc;
  rc = check_cuda(cudaMemsetAsync(row_cnt, 0, (size_t)(4 * rows) * sizeof(int32_t), s), "bmf_expand_init");
  if (rc) return rc;
  // rows per warp: about four blocks per SM in all, at most kExpandRowsPerWarp (the PosCount planes' range)
  const int64_t windows = ceil_div(words, 32);
  int64_t rpw = ceil_div(ceil_div(rows * windows, (int64_t)num_sms() * 4 * 8), 8) * 8;
  rpw = rpw < 8 ? 8 : rpw > kExpandRowsPerWarp ? kExpandRowsPerWarp : rpw;
  const int64_t row_blocks = ceil_div(rows, 8 * rpw);
  BMF_REQUIRE(windows <= 0x7fffffff && row_blocks <= 65535, "bmf_expand_init: matrix too large for one launch");
  dim3 grid((unsigned)windows, (unsigned)row_blocks);
  expand_init_kernel<<<grid, 256, 0, s>>>(x_bits, old_bits, rows, n, words, row0, u_bits, v_bits, row_cnt,
                                          reinterpret_cast<unsigned long long*>(col_cnt), rpw);
  BMF_LAUNCH_CHECK("bmf_expand_init");
  return 0;
}

extern "C" int bmf_expand_step_rows(const uint64_t* x_bits, const uint64_t* old_bits, int64_t rows, int64_t n,
                                    int64_t words, int64_t row0, const uint64_t* u_bits, int32_t* row_cnt, double w_fp,
                                    double w_fn, int64_t* state, int64_t* partials, int64_t* xbuf, int64_t world,
                                    int64_t rank, bmf_stream_t stream) {
  BMF_REQUIRE(u_bits && state && partials && xbuf && (rows == 0 || (x_bits && old_bits && row_cnt)),
              "bmf_expand_step_rows: null pointer");
  BMF_REQUIRE(rows >= 0 && n > 0 && words * 64 >= n && world >= 1 && rank >= 0 && rank < world,
              "bmf_expand_step_rows: bad arguments");
  int64_t blocks = ceil_div(rows, 256);
  blocks = blocks < 1 ? 1 : blocks > kExpandMaxBlocks ? kExpandMaxBlocks : blocks;
  expand_step_rows_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      x_bits, old_bits, rows, n, words, row0, u_bits, row_cnt, -w_fp, w_fn, reinterpret_cast<long long*>(state),
      reinterpret_cast<long long*>(partials), reinterpret_cast<long long*>(xbuf), world, rank);
  BMF_LAUNCH_CHECK("bmf_expand_step_rows");
  return 0;
}

extern "C" int bmf_expand_step_decide(int64_t* col_cnt, int64_t n, int64_t words, uint64_t* u_bits, uint64_t* v_bits,
                                      double w_fp, double w_fn, int64_t* state, int64_t* partials, const int64_t* xbuf,
                                      int64_t world, int64_t* log, int64_t log_cap, bmf_stream_t stream) {
  BMF_REQUIRE(col_cnt && u_bits && v_bits && state && partials && xbuf && log, "bmf_expand_step_decide: null pointer");
  BMF_REQUIRE(n > 0 && words * 64 >= n && world >= 1 && log_cap >= 0, "bmf_expand_step_decide: bad arguments");
  int64_t blocks = ceil_div(n, 256);
  blocks = blocks > kExpandMaxBlocks ? kExpandMaxBlocks : blocks;
  expand_step_decide_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      reinterpret_cast<long long*>(col_cnt), n, words, u_bits, v_bits, -w_fp, w_fn, reinterpret_cast<long long*>(state),
      reinterpret_cast<long long*>(partials) + 2 * kExpandMaxBlocks, reinterpret_cast<const long long*>(xbuf), world,
      reinterpret_cast<long long*>(log), log_cap);
  BMF_LAUNCH_CHECK("bmf_expand_step_decide");
  return 0;
}

extern "C" int bmf_expand_col_scores(const int64_t* col_cnt, int64_t n, const uint64_t* v_bits, double w_fp, double w_fn,
                                     double* delta, int64_t* best, bmf_stream_t stream) {
  BMF_REQUIRE(col_cnt && v_bits && delta && best, "bmf_expand_col_scores: null pointer");
  BMF_REQUIRE(n > 0, "bmf_expand_col_scores: bad shape");
  int64_t blocks = ceil_div(n, 256);
  if (blocks > row_stream_grid()) blocks = row_stream_grid();
  expand_col_delta_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const long long*>(col_cnt), n,
                                                                         v_bits, -w_fp, w_fn, delta);
  BMF_LAUNCH_CHECK("bmf_expand_col_scores");
  argmax_first_f64_kernel<<<1, 1024, 0, as_stream(stream)>>>(delta, n, reinterpret_cast<long long*>(best));
  BMF_LAUNCH_CHECK("bmf_expand_col_scores");
  return 0;
}

extern "C" int bmf_optimal_rows(const uint64_t* x_bits, int64_t m, int64_t words, const uint64_t* vt_bits, int64_t k,
                                double w_fp, double w_fn, int64_t* best_trial, double* best_score, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && vt_bits && best_trial, "bmf_optimal_rows: null pointer");
  BMF_REQUIRE(m > 0 && words > 0 && k >= 1 && k <= 20, "bmf_optimal_rows: 1 <= k <= 20 (2^k trials per row)");
  const size_t vt_bytes = (size_t)k * (size_t)words * sizeof(uint64_t);
  const int in_smem = vt_bytes <= 160 * 1024;
  if (in_smem) {
    int rc = check_cuda(cudaFuncSetAttribute(optimal_row_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)vt_bytes),
                        "bmf_optimal_rows");
    if (rc) return rc;
  }
  int64_t blocks = m < (int64_t)num_sms() * 8 ? m : (int64_t)num_sms() * 8;
  optimal_row_kernel<<<(unsigned)blocks, 256, in_smem ? vt_bytes : 0, as_stream(stream)>>>(
      x_bits, m, words, vt_bits, (int)k, -w_fp, w_fn, in_smem, reinterpret_cast<long long*>(best_trial), best_score);
  BMF_LAUNCH_CHECK("bmf_optimal_rows");
  return 0;
}


static inline uint32_t bernoulli_threshold(double p) {
  if (!(p > 0.0)) return 0u;
  if (p >= 1.0) return 0xFFFFFFFFu;
  return (uint32_t)(p * 4294967296.0);
}

extern "C" int bmf_random_bits(uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, int64_t row0, uint64_t seed,
                               uint64_t stream_id, double p, bmf_stream_t stream) {
  BMF_REQUIRE(bits && rows >= 0 && ncols > 0 && words * 64 >= ncols && row0 >= 0, "bmf_random_bits: bad arguments");
  BMF_REQUIRE(p >= 0.0 && p <= 1.0, "bmf_random_bits: p must be in [0, 1]");
  if (rows == 0) return 0;
  int64_t blocks = ceil_div(rows * words, 256);
  if (blocks > (int64_t)num_sms() * 32) blocks = (int64_t)num_sms() * 32;
  random_bits_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(bits, rows, ncols, words, row0, seed, stream_id,
                                                                    bernoulli_threshold(p));
  BMF_LAUNCH_CHECK("bmf_random_bits");
  return 0;
}

extern "C" int bmf_noise_bits(uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, int64_t row0, uint64_t seed,
                              double p_pos, double p_neg, bmf_stream_t stream) {
  BMF_REQUIRE(bits && rows >= 0 && ncols > 0 && words * 64 >= ncols && row0 >= 0, "bmf_noise_bits: bad arguments");
  BMF_REQUIRE(p_pos >= 0.0 && p_pos <= 1.0 && p_neg >= 0.0 && p_neg <= 1.0, "bmf_noise_bits: probabilities must be in [0, 1]");
  if (rows == 0) return 0;
  int64_t blocks = ceil_div(rows * words, 256);
  if (blocks > (int64_t)num_sms() * 32) blocks = (int64_t)num_sms() * 32;
  noise_bits_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(bits, rows, ncols, words, row0, seed,
                                                                   bernoulli_threshold(p_pos), bernoulli_threshold(p_neg));
  BMF_LAUNCH_CHECK("bmf_noise_bits");
  return 0;
}

extern "C" int bmf_split_bits(const uint64_t* x_bits, int64_t rows, int64_t ncols, int64_t words, int64_t row0, uint64_t seed,
                              uint64_t stream_ones, uint64_t stream_zeros, uint64_t t_v, uint64_t t_t, uint64_t q_v,
                              uint64_t q_t, uint64_t* out_bits, bmf_stream_t stream) {
  BMF_REQUIRE(x_bits && out_bits && rows >= 0 && ncols > 0 && words * 64 >= ncols && row0 >= 0, "bmf_split_bits: bad arguments");
  BMF_REQUIRE(t_v <= 0xFFFFFFFFull && t_t <= 0xFFFFFFFFull && q_v <= 0xFFFFFFFFull && q_t <= 0xFFFFFFFFull,
              "bmf_split_bits: thresholds are 32-bit");
  if (rows == 0) return 0;
  int64_t blocks = ceil_div(rows * words, 256);
  if (blocks > (int64_t)num_sms() * 32) blocks = (int64_t)num_sms() * 32;
  split_bits_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(x_bits, rows, ncols, words, row0, seed, stream_ones,
                                                                   stream_zeros, t_v, t_v + t_t, q_v, q_v + q_t, out_bits);
  BMF_LAUNCH_CHECK("bmf_split_bits");
  return 0;
}

extern "C" int bmf_transpose_bits(const uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, uint64_t* bits_t,
                                  int64_t words_t, bmf_stream_t stream) {
  BMF_REQUIRE(bits && bits_t && rows > 0 && ncols > 0, "bmf_transpose_bits: bad arguments");
  BMF_REQUIRE(words * 64 >= ncols && words_t * 64 >= rows, "bmf_transpose_bits: word counts must cover the matrix");
  BMF_REQUIRE(ceil_div(rows, 64) <= 65535, "bmf_transpose_bits: more than 4.19M rows per call; transpose in row chunks");
  dim3 grid((unsigned)ceil_div(ceil_div(ncols, 64), kTransposeColWords), (unsigned)ceil_div(rows, 64 * kTransposeRowBlocks));
  transpose_bits_kernel<<<grid, 256, 0, as_stream(stream)>>>(bits, rows, ncols, words, bits_t, words_t);
  BMF_LAUNCH_CHECK("bmf_transpose_bits");
  return 0;
}
