// Frame tile and weight-streaming GEMM shared by the fused WaveNet block (wavenet_f32.cu) and its backward
// (wavenet_train_sm100.cu); the sampler's weight layout, shared by the sampler (wavenet_ar_sm100.cu) and the weight-norm
// fold that writes it (wavenet_train_sm100.cu).
#pragma once
#include "svsk_common.cuh"

namespace svsk {

constexpr int kArThreads = 1024;
constexpr int kArWarps = kArThreads / 32;
constexpr int kArMaxLayers = 64;

struct ArLayout {
  long long first_w, first_b, layer0, layer_stride, w3, b3, w4, b4, total;
  long long gw, gb, sw, sb;   // offsets inside one layer block
  long long hist;             // floats of ring buffer per track
  int smem;                   // bytes of dynamic shared memory
};

// Packed weights (floats): WfT [out][R] (first_conv, transposed: one class is one contiguous row), bf [R]; per layer
// Wg [G][k R] (column j R + r = conv.weight[:, r, j]), bg [G], Wso [S + R][G/2] (rows: skip then out), bso [S + R];
// then W3 [S][S], b3 [S], W4 [out][S], b4 [out].
inline ArLayout ar_layout(int O, int R, int G, int S, int L, int stacks, int k) {
  ArLayout a = {};
  const long long Gh = G / 2, kR = (long long)k * R;
  a.first_w = 0;
  a.first_b = (long long)O * R;
  a.layer0 = a.first_b + R;
  a.gw = 0;
  a.gb = G * kR;
  a.sw = a.gb + G;
  a.sb = a.sw + (S + R) * Gh;
  a.layer_stride = a.sb + S + R;
  a.w3 = a.layer0 + L * a.layer_stride;
  a.b3 = a.w3 + (long long)S * S;
  a.w4 = a.b3 + S;
  a.b4 = a.w4 + (long long)O * S;
  a.total = a.b4 + O;
  const int per = L / stacks;
  for (int l = 0; l < L; ++l) a.hist += ((long long)(k - 1) * (1LL << (l % per)) + 1) * R;
  a.smem = (int)(((long long)L * kR + (long long)L * G + Gh + 2LL * S + 2LL * O) * sizeof(float) + 3LL * L * sizeof(int) +
                 sizeof(int));
  return a;
}

// The shapes the sampler's fixed register tiles cover (see the warp_rows instantiations in wavenet_ar_sm100.cu).
inline bool ar_supported(int O, int R, int G, int S, int L, int stacks, int k) {
  if (O < 1 || R < 1 || G < 2 || G % 2 || S < 1 || L < 1 || stacks < 1 || k < 1) return false;
  if (L > kArMaxLayers || L % stacks || L / stacks > 16) return false;
  // gate: k R <= 8 x 32 weights per lane, 2 pairs per warp; skip|out: K = G/2 <= 2 x 32, S + R <= 4 rows per warp;
  // last1: S <= 2 x 32; last3: out_dim <= 8 rows per warp
  if (k * R > 8 * 32 || G / 2 > 2 * 32 || S + R > 4 * kArWarps || S > 2 * 32 || O > 8 * kArWarps) return false;
  const ArLayout a = ar_layout(O, R, G, S, L, stacks, k);
  return a.smem <= 48 * 1024 && a.hist <= (1LL << 30) && a.total <= (1LL << 30);
}

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
