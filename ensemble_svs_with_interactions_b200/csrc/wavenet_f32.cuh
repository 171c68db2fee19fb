// Frame tile and weight-streaming GEMM shared by the fused WaveNet block (wavenet_f32.cu) and its backward
// (wavenet_train_sm100.cu).
#pragma once
#include "svsk_common.cuh"

namespace svsk {

constexpr int kWnTT = 16;  // frames per CTA
constexpr int kWnKC = 32;  // weight rows staged per chunk

// acc[i] += sum_k w[k][col] * in[k][tg * 8 + i] for one (column, half tile) item per thread, K rows of weights streamed
// through shared memory in chunks of kWnKC rows: all threads fetch the NEXT chunk into registers (coalesced float4, many
// loads in flight) before they compute on the current one, so the L2 latency of a chunk hides behind 32 k-steps of FMAs.
// ncols is a multiple of 4; w_s holds kWnKC * ncols floats.  Must be called by all 256 threads.
__device__ __forceinline__ void wn_gemm_tile(const float* __restrict__ w, int K, int ncols, const float* in_s, float* w_s,
                                             int n_items, float (&acc)[2][8]) {
  const int vec_per_chunk = kWnKC * ncols / 4;           // float4s per chunk
  constexpr int kMaxV = 8;                               // per thread: chunk of 32 x 256 floats at most
  float4 nxt[kMaxV];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int v = 0; v < kMaxV; ++v) {
      const int i = threadIdx.x + v * 256;
      nxt[v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < vec_per_chunk) {
        const int r = (i * 4) / ncols;
        if (k0 + r < K) nxt[v] = *reinterpret_cast<const float4*>(w + (size_t)k0 * ncols + (size_t)i * 4);
      }
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < K; k0 += kWnKC) {
    __syncthreads();                                      // the previous chunk has been consumed
#pragma unroll
    for (int v = 0; v < kMaxV; ++v) {
      const int i = threadIdx.x + v * 256;
      if (i < vec_per_chunk) *reinterpret_cast<float4*>(w_s + (size_t)i * 4) = nxt[v];
    }
    __syncthreads();
    if (k0 + kWnKC < K) fetch(k0 + kWnKC);
    const int kn = min(kWnKC, K - k0);
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int item = threadIdx.x + it * 256;
      if (item >= n_items) break;
      const int col = item % ncols, tg = item / ncols;
      const float* xs = in_s + (size_t)k0 * kWnTT + tg * 8;
#pragma unroll 8
      for (int k = 0; k < kn; ++k) {
        const float wv = w_s[k * ncols + col];
        const float4 a = *reinterpret_cast<const float4*>(xs + k * kWnTT);
        const float4 c4 = *reinterpret_cast<const float4*>(xs + k * kWnTT + 4);
        acc[it][0] = fmaf(wv, a.x, acc[it][0]); acc[it][1] = fmaf(wv, a.y, acc[it][1]);
        acc[it][2] = fmaf(wv, a.z, acc[it][2]); acc[it][3] = fmaf(wv, a.w, acc[it][3]);
        acc[it][4] = fmaf(wv, c4.x, acc[it][4]); acc[it][5] = fmaf(wv, c4.y, acc[it][5]);
        acc[it][6] = fmaf(wv, c4.z, acc[it][6]); acc[it][7] = fmaf(wv, c4.w, acc[it][7]);
      }
    }
  }
}

}  // namespace svsk
