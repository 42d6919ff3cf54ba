// Bit-matrix transpose kernels against a device-to-device copy of the same bytes (CUDA events, 20 launches, 3 rounds):
//   old  : the former transpose_bits_kernel (one 64-thread CTA per 64 x 64 tile, 64 ballots per warp)
//   TW4  : a 256 x 256 tile staged through shared memory, still transposed by ballots
//   SHFL : the current transpose_bits_kernel (256 x 512 tile through shared memory, register transpose by shuffles)
// Outputs of TW4 and SHFL are compared word for word with old, old is spot-checked against the definition.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o transpose_probe profiles/probes/transpose_probe.cu
//   ./transpose_probe [rows ncols]        (default: the c4 shape 480189 x 17770)
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <vector>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e)); exit(1);} } while (0)

__global__ void __launch_bounds__(64) old_k(const uint64_t* __restrict__ x, int64_t rows, int64_t ncols,
                                            int64_t words, uint64_t* __restrict__ xt, int64_t words_t) {
  __shared__ uint32_t half[64][2];
  const int t = threadIdx.x, lane = t & 31, wp = t >> 5;
  const int64_t cb = blockIdx.x, rb = blockIdx.y;
  const int64_t r = rb * 64 + t;
  const uint64_t w = (r < rows) ? x[r * words + cb] : 0ull;
#pragma unroll 8
  for (int c = 0; c < 64; ++c) {
    const uint32_t b = __ballot_sync(0xffffffffu, (w >> c) & 1ull);
    if (lane == 0) half[c][wp] = b;
  }
  __syncthreads();
  const int64_t col = cb * 64 + t;
  if (col < ncols) xt[col * words_t + rb] = (uint64_t)half[t][0] | ((uint64_t)half[t][1] << 32);
}

template <int TW>
__global__ void __launch_bounds__(256) new_k(const uint64_t* __restrict__ x, int64_t rows, int64_t ncols,
                                             int64_t words, uint64_t* __restrict__ xt, int64_t words_t) {
  constexpr int TR = TW * 64;
  __shared__ uint64_t tin[TR][TW + 1];
  __shared__ uint32_t tout[TR][2 * TW + 1];
  const int t = threadIdx.x, lane = t & 31, wp = t >> 5;
  const int64_t wc0 = (int64_t)blockIdx.x * TW;
  const int64_t r0 = (int64_t)blockIdx.y * TR;
  const int64_t ww = (ncols + 63) >> 6;
  for (int i = t; i < TR * TW; i += 256) {
    const int rr = i / TW, cw = i % TW;
    const int64_t r = r0 + rr, c = wc0 + cw;
    tin[rr][cw] = (r < rows && c < ww) ? x[r * words + c] : 0ull;
  }
  __syncthreads();
  for (int p = wp; p < TW * TW * 2; p += 8) {
    const int cw = p / (2 * TW), hb = p % (2 * TW);
    const uint64_t v = tin[hb * 32 + lane][cw];
#pragma unroll 8
    for (int c = 0; c < 64; ++c) {
      const uint32_t b = __ballot_sync(0xffffffffu, (v >> c) & 1ull);
      if (lane == (c & 31)) tout[cw * 64 + c][hb] = b;
    }
  }
  __syncthreads();
  const int64_t wt0 = (int64_t)blockIdx.y * TW;
  for (int i = t; i < TR * TW; i += 256) {
    const int cc = i / TW, j = i % TW;
    const int64_t col = wc0 * 64 + cc, wt = wt0 + j;
    if (col < ncols && wt * 64 < rows && wt < words_t)
      xt[col * words_t + wt] = (uint64_t)tout[cc][2 * j] | ((uint64_t)tout[cc][2 * j + 1] << 32);
  }
}


// 64 x 64 bit-block transpose in registers: lane l holds rows l (a0) and l + 32 (a1); afterwards it holds columns l and
// l + 32 as rows.  Six swap stages (Hacker's Delight 7-3): 32 inside the thread, 16 .. 1 across lanes by shuffles.
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
    const bool hi = lane & j;
    const uint64_t p0 = __shfl_xor_sync(0xffffffffu, a0, j), p1 = __shfl_xor_sync(0xffffffffu, a1, j);
    const uint64_t t0 = (((hi ? p0 : a0) >> j) ^ (hi ? a0 : p0)) & masks[s];
    const uint64_t t1 = (((hi ? p1 : a1) >> j) ^ (hi ? a1 : p1)) & masks[s];
    a0 ^= hi ? t0 : (t0 << j);
    a1 ^= hi ? t1 : (t1 << j);
  }
}

// CTA tile: 256 rows x 512 columns (4 x 8 blocks of 64 x 64), staged through shared memory so that both the loads (64 B
// per row) and the stores (32 B per output row) are whole sectors
__global__ void __launch_bounds__(256) sh_k(const uint64_t* __restrict__ x, int64_t rows, int64_t ncols,
                                            int64_t words, uint64_t* __restrict__ xt, int64_t words_t) {
  constexpr int RB = 4, CW = 8;
  __shared__ uint64_t tin[RB * 64][CW + 1];
  __shared__ uint64_t tout[CW * 64][RB + 1];
  const int t = threadIdx.x, lane = t & 31, wp = t >> 5;
  const int64_t w0 = (int64_t)blockIdx.x * CW, r0 = (int64_t)blockIdx.y * (RB * 64);
  const int64_t wn = (ncols + 63) >> 6;
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

static int64_t words_for(int64_t n) { int64_t w = (n + 63) / 64; w += w & 1; return w < 2 ? 2 : w; }

template <typename F>
float timeit(F f, int iters) {
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  for (int i = 0; i < 3; ++i) f();
  CK(cudaDeviceSynchronize());
  cudaEventRecord(a);
  for (int i = 0; i < iters; ++i) f();
  cudaEventRecord(b); CK(cudaEventSynchronize(b));
  float ms; cudaEventElapsedTime(&ms, a, b);
  return ms / iters;
}

int main(int argc, char** argv) {
  int64_t rows = argc > 1 ? atoll(argv[1]) : 480189, ncols = argc > 2 ? atoll(argv[2]) : 17770;
  int64_t words = words_for(ncols), words_t = words_for(rows);
  size_t in_b = rows * words * 8, out_b = ncols * words_t * 8;
  std::vector<uint64_t> h(rows * words);
  uint64_t s = 88172645463325252ull;
  for (int64_t r = 0; r < rows; ++r)
    for (int64_t w = 0; w < words; ++w) {
      s ^= s << 13; s ^= s >> 7; s ^= s << 17;
      uint64_t v = s;
      int64_t left = ncols - w * 64;
      if (left <= 0) v = 0; else if (left < 64) v &= (1ull << left) - 1;
      h[r * words + w] = v;
    }
  uint64_t *x, *a, *b, *cp;
  CK(cudaMalloc(&x, in_b)); CK(cudaMalloc(&a, out_b)); CK(cudaMalloc(&b, out_b)); CK(cudaMalloc(&cp, in_b));
  CK(cudaMemcpy(x, h.data(), in_b, cudaMemcpyHostToDevice));
  CK(cudaMemset(a, 0, out_b)); CK(cudaMemset(b, 0, out_b));
  dim3 g0((unsigned)((ncols + 63) / 64), (unsigned)((rows + 63) / 64));
  dim3 g4((unsigned)(((ncols + 63) / 64 + 3) / 4), (unsigned)((rows + 255) / 256));
  auto f_old = [&] { old_k<<<g0, 64>>>(x, rows, ncols, words, a, words_t); };
  auto f_new4 = [&] { new_k<4><<<g4, 256>>>(x, rows, ncols, words, b, words_t); };
  dim3 gs((unsigned)(((ncols + 63) / 64 + 7) / 8), (unsigned)((rows + 255) / 256));
  auto f_shfl = [&] { sh_k<<<gs, 256>>>(x, rows, ncols, words, b, words_t); };
  auto f_cp = [&] { cudaMemcpyAsync(cp, x, in_b, cudaMemcpyDeviceToDevice); };
  f_old(); CK(cudaDeviceSynchronize());
  std::vector<uint64_t> ha(ncols * words_t), hb(ncols * words_t);
  CK(cudaMemcpy(ha.data(), a, out_b, cudaMemcpyDeviceToHost));
  for (int v = 0; v < 2; ++v) {
    CK(cudaMemset(b, 0, out_b));
    if (v == 0) f_new4(); else f_shfl();
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(hb.data(), b, out_b, cudaMemcpyDeviceToHost));
    size_t bad = 0;
    for (size_t i = 0; i < ha.size(); ++i) bad += ha[i] != hb[i];
    // spot-check old against the definition
    size_t bad_def = 0;
    for (int q = 0; q < 20000; ++q) {
      int64_t r = (q * 7919ll) % rows, c = (q * 104729ll) % ncols;
      uint64_t want = (h[r * words + c / 64] >> (c % 64)) & 1, got = (ha[c * words_t + r / 64] >> (r % 64)) & 1;
      bad_def += want != got;
    }
    printf("variant %s mismatches vs old: %zu, old vs definition: %zu\n", v == 0 ? "TW4" : "SHFL", bad, bad_def);
  }
  int it = 20;
  for (int rep = 0; rep < 3; ++rep) {
    float t_old = timeit(f_old, it), t4 = timeit(f_new4, it), t2 = timeit(f_shfl, it), t_cp = timeit(f_cp, it);
    double bytes = (double)in_b + (double)out_b;
    printf("rows=%lld ncols=%lld  old %.3f ms %.0f GB/s | TW4 %.3f ms %.0f GB/s | SHFL %.3f ms %.0f GB/s | copy %.3f ms %.0f GB/s (read+write)\n",
           (long long)rows, (long long)ncols, t_old, bytes / t_old / 1e6, t4, bytes / t4 / 1e6, t2, bytes / t2 / 1e6,
           t_cp, 2.0 * in_b / t_cp / 1e6);
  }
  return 0;
}
