// GreConD's concept search on bit rows (pybmf_b200/concept.py, DESIGN.md section 1 row f5).
//
// A factor is grown by the reference's first-improvement rule: with extent C, intent D and best cover `best`, the
// candidate columns j > pos, j not in D are scored as
//     C_j = C & X[:, j],   D_j = AND of the rows X[r], r in C_j (all columns when C_j is empty),
//     s_j = sum over r in C_j of popc(R[r] & D_j)         (R: the residual)
// and the FIRST j with s_j > best is accepted.  Three kernels serve both the seed search (C = all rows of one rank, one
// window of 64 columns) and the candidate rounds (C = a subset of the compact extent rows, every column):
//   concept_intents_kernel : D_j for a range of column words (+ the row count of each column when asked)
//   concept_covers_kernel  : s_j against given intents (ANDed over `parts` partial intents: one per rank in the seed)
//   concept_decide_kernel  : one block; the first j > pos, j not in D, with s_j > best; accepts it or sets `done`
// plus the extent gather (rows of one column compacted into [cap][words] buffers) and the in-place residual update.
//
// Block shape of the scoring kernels: 32 x 8 threads.  threadIdx.x is a word of the row (blockIdx.y picks a slice of 32
// words), threadIdx.y a group of 8 of the 64 columns of column word blockIdx.x; every thread keeps 8 accumulators in
// registers, so a row is read once per (column word, word slice) and never staged.  Rows whose bits in the column word
// are all outside the live candidates are skipped after one broadcast load.
#include <climits>

#include "bmf_common.cuh"

namespace bmf {
namespace {

constexpr int kSliceWords = 32;   // words of a row per block (threadIdx.x)
constexpr int kGroups = 8;        // column groups of 8 per column word (threadIdx.y)

// state[]: pos (last accepted column, or seed column - 1), best, done, number of accepted columns
enum { kPos = 0, kBest = 1, kDone = 2, kAccepted = 3 };

// Live candidate columns of column word cw: [lo, n) and not in D.
__device__ __forceinline__ uint64_t live_columns(int64_t cw, int64_t lo, int64_t n, const uint64_t* d_bits) {
  const int64_t c0 = cw * 64;
  uint64_t m = ~0ull;
  if (lo > c0) m = lo >= c0 + 64 ? 0ull : (m << (lo - c0));
  if (n < c0 + 64) m &= n <= c0 ? 0ull : (~0ull >> (c0 + 64 - n));
  if (d_bits) m &= ~d_bits[cw];
  return m;
}

// The row range [r_lo, r_hi) of this block's chunk (chunks are whole 64-row words of the row mask).
__device__ __forceinline__ void chunk_rows(int64_t rows, int64_t rows_per_chunk, int64_t* r_lo, int64_t* r_hi) {
  *r_lo = (int64_t)blockIdx.z * rows_per_chunk;
  *r_hi = *r_lo + rows_per_chunk < rows ? *r_lo + rows_per_chunk : rows;
}

__device__ __forceinline__ uint64_t mask_word(const uint64_t* row_mask, int64_t base, int64_t r_hi) {
  uint64_t mw = row_mask ? row_mask[base >> 6] : ~0ull;
  if (r_hi - base < 64) mw &= (1ull << (r_hi - base)) - 1ull;
  return mw;
}

__global__ void __launch_bounds__(256) concept_intents_kernel(const uint64_t* __restrict__ x, int64_t rows, int64_t words,
                                                              int64_t n, const uint64_t* __restrict__ row_mask,
                                                              int64_t cw0, int64_t col_lo, const long long* state,
                                                              const uint64_t* d_bits, int64_t rows_per_chunk, int atomic,
                                                              uint64_t* intents, unsigned long long* counts) {
  if (state && state[kDone]) return;
  const int64_t cw = cw0 + blockIdx.x;
  const int lane = threadIdx.x, g = threadIdx.y;
  const int64_t w = (int64_t)blockIdx.y * kSliceWords + lane;
  const uint64_t live = live_columns(cw, state ? state[kPos] + 1 : col_lo, n, d_bits);
  if (live == 0) return;                                      // block-uniform
  const bool counting = counts && blockIdx.y == 0 && lane == 0;
  uint64_t acc[8];
  int cnt[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = ~0ull, cnt[i] = 0;
  int64_t r_lo, r_hi;
  chunk_rows(rows, rows_per_chunk, &r_lo, &r_hi);
  for (int64_t base = r_lo; base < r_hi; base += 64) {
    uint64_t mw = mask_word(row_mask, base, r_hi);
    while (mw) {
      const int64_t r = base + __ffsll((long long)mw) - 1;
      mw &= mw - 1;
      const uint32_t bits = (uint32_t)((x[r * words + cw] & live) >> (8 * g)) & 0xFFu;
      if (!bits) continue;
      const uint64_t val = w < words ? x[r * words + w] : 0ull;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (bits >> i & 1u) {
          acc[i] &= val;
          cnt[i] += 1;
        }
    }
  }
  const uint32_t mine = (uint32_t)(live >> (8 * g)) & 0xFFu;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (!(mine >> i & 1u)) continue;
    const int64_t col = (cw - cw0) * 64 + 8 * g + i;
    if (w < words) {
      if (atomic)
        atomicAnd(reinterpret_cast<unsigned long long*>(intents + col * words + w), (unsigned long long)acc[i]);
      else
        intents[col * words + w] = acc[i];
    }
    if (counting && cnt[i]) atomicAdd(counts + col, (unsigned long long)cnt[i]);
  }
}

__global__ void __launch_bounds__(256) concept_covers_kernel(const uint64_t* __restrict__ x, const uint64_t* __restrict__ res,
                                                             int64_t rows, int64_t words, int64_t n,
                                                             const uint64_t* __restrict__ row_mask, int64_t cw0,
                                                             int64_t col_lo, const long long* state, const uint64_t* d_bits,
                                                             const uint64_t* __restrict__ intents, int64_t parts,
                                                             int64_t part_stride, int64_t rows_per_chunk,
                                                             unsigned long long* covers) {
  if (state && state[kDone]) return;
  const int64_t cw = cw0 + blockIdx.x;
  const int lane = threadIdx.x, g = threadIdx.y;
  const int64_t w = (int64_t)blockIdx.y * kSliceWords + lane;
  const uint64_t live = live_columns(cw, state ? state[kPos] + 1 : col_lo, n, d_bits);
  if (live == 0) return;
  uint64_t in[8];
  long long acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t col = (cw - cw0) * 64 + 8 * g + i;
    uint64_t v = ~0ull;
    if (w < words)
      for (int64_t q = 0; q < parts; ++q) v &= intents[q * part_stride + col * words + w];
    in[i] = w < words ? v : 0ull;
    acc[i] = 0;
  }
  int64_t r_lo, r_hi;
  chunk_rows(rows, rows_per_chunk, &r_lo, &r_hi);
  for (int64_t base = r_lo; base < r_hi; base += 64) {
    uint64_t mw = mask_word(row_mask, base, r_hi);
    while (mw) {
      const int64_t r = base + __ffsll((long long)mw) - 1;
      mw &= mw - 1;
      const uint32_t bits = (uint32_t)((x[r * words + cw] & live) >> (8 * g)) & 0xFFu;
      if (!bits) continue;
      const uint64_t rv = w < words ? res[r * words + w] : 0ull;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (bits >> i & 1u) acc[i] += __popcll(rv & in[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long s = warp_sum_ll(acc[i]);                  // a warp is one column group over 32 words
    if (lane == 0 && s) atomicAdd(covers + (cw - cw0) * 64 + 8 * g + i, (unsigned long long)s);
  }
}

// One block of 1024 threads.  covers / intents hold every column (column word 0 first).
__global__ void __launch_bounds__(1024) concept_decide_kernel(const uint64_t* __restrict__ xc, int64_t rows, int64_t words,
                                                              int64_t n, const long long* __restrict__ covers,
                                                              const uint64_t* __restrict__ intents, long long* state,
                                                              uint64_t* c_bits, uint64_t* d_bits) {
  __shared__ long long first_s[32];
  __shared__ long long pick;
  if (state[kDone]) return;
  const int tid = threadIdx.x;
  const long long pos = state[kPos], best = state[kBest];
  long long first = LLONG_MAX;
  for (long long j = pos + 1 + tid; j < n; j += blockDim.x)
    if (!(d_bits[j >> 6] >> (j & 63) & 1ull) && covers[j] > best) {
      first = j;
      break;
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const long long other = __shfl_xor_sync(0xffffffffu, first, o);
    first = other < first ? other : first;
  }
  if ((tid & 31) == 0) first_s[tid >> 5] = first;
  __syncthreads();
  if (tid < 32) {
    long long f = tid < (int)(blockDim.x >> 5) ? first_s[tid] : LLONG_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const long long other = __shfl_xor_sync(0xffffffffu, f, o);
      f = other < f ? other : f;
    }
    if (tid == 0) pick = f;
  }
  __syncthreads();
  const long long j = pick;
  if (j == LLONG_MAX) {
    if (tid == 0) state[kDone] = 1;
    return;
  }
  for (int64_t w = tid; w < words; w += blockDim.x) d_bits[w] = intents[j * words + w];
  // C &= X[:, j], 32 rows per warp and ballot; each warp owns whole 32-bit halves of c_bits
  uint32_t* c32 = reinterpret_cast<uint32_t*>(c_bits);
  const int64_t cw = j >> 6;
  const uint64_t jbit = 1ull << (j & 63);
  for (int64_t base = (int64_t)(tid & ~31); base < rows; base += blockDim.x) {
    const int64_t r = base + (tid & 31);
    const uint32_t half = c32[base >> 5];
    const bool keep = r < rows && (half >> (tid & 31) & 1u) && (xc[r * words + cw] & jbit);
    const uint32_t b = __ballot_sync(0xffffffffu, keep);
    if ((tid & 31) == 0) c32[base >> 5] = b;
  }
  if (tid == 0) {
    state[kPos] = j;
    state[kBest] = covers[j];
    state[kAccepted] += 1;
  }
}

// Rows of x (and of the residual) with bit `col`, compacted; idx[] gets their logical rows row0 + r.
__global__ void concept_extent_kernel(const uint64_t* __restrict__ x, const uint64_t* __restrict__ res, int64_t rows,
                                      int64_t words, int64_t row0, int64_t col, int64_t cap, uint64_t* xc, uint64_t* rc,
                                      long long* idx, unsigned long long* fill) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const uint64_t cbit = 1ull << (col & 63);
  for (int64_t base = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; base < rows;
       base += warps * 32) {
    const int64_t r = base + lane;
    const bool has = r < rows && (x[r * words + (col >> 6)] & cbit);
    uint32_t b = __ballot_sync(0xffffffffu, has);
    if (!b) continue;
    unsigned long long at = 0;
    if (lane == 0) at = atomicAdd(fill, (unsigned long long)__popc(b));
    at = __shfl_sync(0xffffffffu, at, 0);
    while (b) {
      const int k = __ffs(b) - 1;
      b &= b - 1;
      if ((int64_t)at < cap) {
        const int64_t src = base + k;
        for (int64_t w = lane; w < words; w += 32) {
          xc[(int64_t)at * words + w] = x[src * words + w];
          rc[(int64_t)at * words + w] = res[src * words + w];
        }
        if (lane == 0) idx[at] = row0 + src;
      }
      ++at;
    }
  }
}

// R[idx[c] - row0] &= ~D for the compact rows c in C whose logical row is in [row0, row1).
__global__ void concept_residual_kernel(uint64_t* res, int64_t row0, int64_t row1, int64_t words,
                                        const long long* __restrict__ idx, int64_t rows, const uint64_t* __restrict__ c_bits,
                                        const uint64_t* __restrict__ d_bits) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t c = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < rows; c += warps) {
    if (!(c_bits[c >> 6] >> (c & 63) & 1ull)) continue;
    const long long r = idx[c];
    if (r < row0 || r >= row1) continue;
    for (int64_t w = lane; w < words; w += 32) res[(r - row0) * words + w] &= ~d_bits[w];
  }
}

// Row chunks for a grid of `xy` blocks: enough blocks to fill the GPU, chunks of whole 64-row mask words.
int64_t rows_per_chunk(int64_t rows, int64_t xy) {
  int64_t chunks = ceil_div(16 * (int64_t)num_sms(), xy);
  const int64_t most = ceil_div(rows, 256);
  if (chunks > most) chunks = most;
  if (chunks < 1) chunks = 1;
  return ceil_div(ceil_div(rows, chunks), 64) * 64;
}

}  // namespace
}  // namespace bmf

using namespace bmf;

extern "C" int bmf_concept_intents(const uint64_t* x, int64_t rows, int64_t words, int64_t n, const uint64_t* row_mask,
                                   int64_t cw0, int64_t ncw, int64_t col_lo, const int64_t* state, const uint64_t* d_bits,
                                   uint64_t* intents, int64_t* counts, bmf_stream_t stream) {
  BMF_REQUIRE(x && intents, "bmf_concept_intents: null pointer");
  BMF_REQUIRE(rows >= 0 && words > 0 && n > 0 && words * 64 >= n && cw0 >= 0 && ncw >= 1 && cw0 + ncw <= words,
              "bmf_concept_intents: bad shape");
  const cudaStream_t s = as_stream(stream);
  const int64_t slices = ceil_div(words, kSliceWords);
  const int64_t rpc = rows > 0 ? rows_per_chunk(rows, ncw * slices) : 64;
  const int64_t chunks = rows > 0 ? ceil_div(rows, rpc) : 1;
  const int atomic = chunks > 1 || rows == 0;
  if (atomic) {
    int rc = check_cuda(cudaMemsetAsync(intents, 0xFF, (size_t)ncw * 64 * words * sizeof(uint64_t), s), "bmf_concept_intents");
    if (rc) return rc;
  }
  if (counts) {
    int rc = check_cuda(cudaMemsetAsync(counts, 0, (size_t)ncw * 64 * sizeof(int64_t), s), "bmf_concept_intents");
    if (rc) return rc;
  }
  if (rows == 0) return 0;
  BMF_REQUIRE(slices <= 65535 && chunks <= 65535 && ncw <= 0x7FFFFFFF, "bmf_concept_intents: grid too large");
  concept_intents_kernel<<<dim3((unsigned)ncw, (unsigned)slices, (unsigned)chunks), dim3(kSliceWords, kGroups), 0, s>>>(
      x, rows, words, n, row_mask, cw0, col_lo, reinterpret_cast<const long long*>(state), d_bits, rpc, atomic, intents,
      reinterpret_cast<unsigned long long*>(counts));
  BMF_LAUNCH_CHECK("bmf_concept_intents");
  return 0;
}

extern "C" int bmf_concept_covers(const uint64_t* x, const uint64_t* res, int64_t rows, int64_t words, int64_t n,
                                  const uint64_t* row_mask, int64_t cw0, int64_t ncw, int64_t col_lo, const int64_t* state,
                                  const uint64_t* d_bits, const uint64_t* intents, int64_t parts, int64_t part_stride,
                                  int64_t* covers, bmf_stream_t stream) {
  BMF_REQUIRE(x && res && intents && covers, "bmf_concept_covers: null pointer");
  BMF_REQUIRE(rows >= 0 && words > 0 && n > 0 && words * 64 >= n && cw0 >= 0 && ncw >= 1 && cw0 + ncw <= words,
              "bmf_concept_covers: bad shape");
  BMF_REQUIRE(parts >= 1 && (parts == 1 || part_stride >= ncw * 64 * words), "bmf_concept_covers: bad parts");
  const cudaStream_t s = as_stream(stream);
  int rc = check_cuda(cudaMemsetAsync(covers, 0, (size_t)ncw * 64 * sizeof(int64_t), s), "bmf_concept_covers");
  if (rc) return rc;
  if (rows == 0) return 0;
  const int64_t slices = ceil_div(words, kSliceWords);
  const int64_t rpc = rows_per_chunk(rows, ncw * slices);
  const int64_t chunks = ceil_div(rows, rpc);
  BMF_REQUIRE(slices <= 65535 && chunks <= 65535 && ncw <= 0x7FFFFFFF, "bmf_concept_covers: grid too large");
  concept_covers_kernel<<<dim3((unsigned)ncw, (unsigned)slices, (unsigned)chunks), dim3(kSliceWords, kGroups), 0, s>>>(
      x, res, rows, words, n, row_mask, cw0, col_lo, reinterpret_cast<const long long*>(state), d_bits, intents, parts,
      part_stride, rpc, reinterpret_cast<unsigned long long*>(covers));
  BMF_LAUNCH_CHECK("bmf_concept_covers");
  return 0;
}

extern "C" int bmf_concept_decide(const uint64_t* xc, int64_t rows, int64_t words, int64_t n, const int64_t* covers,
                                  const uint64_t* intents, int64_t* state, uint64_t* c_bits, uint64_t* d_bits,
                                  bmf_stream_t stream) {
  BMF_REQUIRE(xc && covers && intents && state && c_bits && d_bits, "bmf_concept_decide: null pointer");
  BMF_REQUIRE(rows >= 0 && words > 0 && n > 0 && words * 64 >= n, "bmf_concept_decide: bad shape");
  concept_decide_kernel<<<1, 1024, 0, as_stream(stream)>>>(xc, rows, words, n, reinterpret_cast<const long long*>(covers),
                                                           intents, reinterpret_cast<long long*>(state), c_bits, d_bits);
  BMF_LAUNCH_CHECK("bmf_concept_decide");
  return 0;
}

extern "C" int bmf_concept_extent(const uint64_t* x, const uint64_t* res, int64_t rows, int64_t words, int64_t row0,
                                  int64_t col, int64_t cap, uint64_t* xc, uint64_t* rc, int64_t* idx, int64_t* fill,
                                  bmf_stream_t stream) {
  BMF_REQUIRE(x && res && xc && rc && idx && fill, "bmf_concept_extent: null pointer");
  BMF_REQUIRE(rows >= 0 && words > 0 && col >= 0 && col < words * 64 && cap >= 0 && row0 >= 0,
              "bmf_concept_extent: bad arguments");
  const cudaStream_t s = as_stream(stream);
  int e = check_cuda(cudaMemsetAsync(fill, 0, sizeof(int64_t), s), "bmf_concept_extent");
  if (e) return e;
  if (cap > 0) {
    e = check_cuda(cudaMemsetAsync(idx, 0xFF, (size_t)cap * sizeof(int64_t), s), "bmf_concept_extent");
    if (e) return e;
  }
  if (rows == 0 || cap == 0) return 0;
  int64_t blocks = ceil_div(rows, 8 * 32);
  if (blocks > (int64_t)num_sms() * 8) blocks = (int64_t)num_sms() * 8;
  concept_extent_kernel<<<(unsigned)blocks, 256, 0, s>>>(x, res, rows, words, row0, col, cap, xc, rc,
                                                         reinterpret_cast<long long*>(idx),
                                                         reinterpret_cast<unsigned long long*>(fill));
  BMF_LAUNCH_CHECK("bmf_concept_extent");
  return 0;
}

extern "C" int bmf_concept_residual(uint64_t* res, int64_t row0, int64_t row1, int64_t words, const int64_t* idx,
                                    int64_t rows, const uint64_t* c_bits, const uint64_t* d_bits, bmf_stream_t stream) {
  BMF_REQUIRE(res && idx && c_bits && d_bits, "bmf_concept_residual: null pointer");
  BMF_REQUIRE(row0 >= 0 && row1 >= row0 && words > 0 && rows >= 0, "bmf_concept_residual: bad arguments");
  if (rows == 0 || row1 == row0) return 0;
  int64_t blocks = ceil_div(rows, 8);
  if (blocks > (int64_t)num_sms() * 8) blocks = (int64_t)num_sms() * 8;
  concept_residual_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
      res, row0, row1, words, reinterpret_cast<const long long*>(idx), rows, c_bits, d_bits);
  BMF_LAUNCH_CHECK("bmf_concept_residual");
  return 0;
}
