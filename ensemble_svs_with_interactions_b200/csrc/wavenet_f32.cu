// Fused WaveNet residual block in fp32 (SURVEY.md K6): replaces ResSkipBlock._forward (nnsvs/wavenet/modules.py:88-122)
// with ONE launch per layer —
//   y = causal_conv_k_dil(x) + conv1x1c(c) + b          (taps at t - (k-1-j) d, zeros before the start)
//   z = tanh(y[:G/2]) * sigmoid(y[G/2:])
//   skips (+)= conv1x1_skip(z) + b_skip ;  x_out = conv1x1_out(z) + b_out + x      (no sqrt(1/2): modules.py:119-121)
// instead of five (conv, conditioning conv, gate, skip conv, out conv).  The acoustic WaveNet is tiny (71 168 MAC per
// frame and layer, B x T = 400 frames in the reference's test): it is launch-latency bound, so the kernel stays on the
// CUDA cores in exact fp32 (this is the reference's own arithmetic; tolerance 1e-6, not a bf16 path) and spends its
// effort on having a frame tile's whole block in one CTA: inputs (all taps + conditioning) staged once in shared
// memory, the gate pre-activations and z never leave it.  Weights are pre-transposed ([K][out], folded weight norm) so
// that a warp reads 32 consecutive output channels of one k per load.
#include "wavenet_f32.cuh"

namespace svsk {

// kTrain: also writes the gate pre-activations y [B][G][T] (svsk_wavenet_block_train_f32, kept for the backward); the
// arithmetic is the same, so both instantiations give the same x_out and skips.
template <bool kTrain>
__global__ void __launch_bounds__(256) wavenet_block_f32_kernel(const svsk_wavenet_block_params p, float* __restrict__ y_out) {
  extern __shared__ float smem[];
  const int K1 = p.ksize * p.R + p.Cc, Gh = p.G / 2, O2 = p.S + p.R;
  float* in_s = smem;                                        // [K1][kWnTT]
  float* y_s = in_s + K1 * kWnTT;                            // [G][kWnTT]
  float* z_s = y_s + p.G * kWnTT;                            // [G/2][kWnTT]
  float* w_s = z_s + Gh * kWnTT;                             // [kWnKC][max(G, O2)]
  const int b = blockIdx.y, t0 = blockIdx.x * kWnTT;
  const float* xb = p.x + (size_t)b * p.R * p.T;
  const float* cb = p.c + (size_t)b * p.Cc * p.T;
  // ---- stage the inputs: row j * R + ci = x[ci][t - (k-1-j) d], rows k R .. = c
  for (int i = threadIdx.x; i < K1 * kWnTT; i += 256) {
    const int r = i / kWnTT, tt = i % kWnTT;
    const int t = t0 + tt;
    float v = 0.f;
    if (t < p.T) {
      if (r < p.ksize * p.R) {
        const int j = r / p.R, ci = r - j * p.R;
        const int u = t - (p.ksize - 1 - j) * p.dilation;
        if (u >= 0) v = xb[(size_t)ci * p.T + u];
      } else {
        v = cb[(size_t)(r - p.ksize * p.R) * p.T + t];
      }
    }
    in_s[i] = v;
  }
  // ---- gate pre-activations: item = (output channel, half tile of 8 frames), up to two items per thread
  {
    const int n_items = p.G * (kWnTT / 8);
    float acc[2][8];
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int item = threadIdx.x + it * 256;
      const float bias = (p.b1 && item < n_items) ? p.b1[item % p.G] : 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[it][i] = bias;
    }
    wn_gemm_tile(p.w1t, K1, p.G, in_s, w_s, n_items, acc);   // (its first __syncthreads also publishes in_s)
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int item = threadIdx.x + it * 256;
      if (item >= n_items) break;
      const int co = item % p.G, tg = item / p.G;
#pragma unroll
      for (int i = 0; i < 8; ++i) y_s[co * kWnTT + tg * 8 + i] = acc[it][i];
    }
  }
  __syncthreads();
  if constexpr (kTrain) {
    for (int i = threadIdx.x; i < p.G * kWnTT; i += 256) {
      const int t = t0 + i % kWnTT;
      if (t < p.T) y_out[((size_t)b * p.G + i / kWnTT) * p.T + t] = y_s[i];
    }
  }
  for (int i = threadIdx.x; i < Gh * kWnTT; i += 256) {
    const float a = y_s[i], g = y_s[Gh * kWnTT + i];
    z_s[i] = tanhf(a) * (1.f / (1.f + expf(-g)));
  }
  // ---- skip (columns [0, S)) and out (columns [S, S + R)) projections of z
  {
    const int n_items = O2 * (kWnTT / 8);
    float acc[2][8];
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int item = threadIdx.x + it * 256;
      const float bias = item < n_items ? p.b2[item % O2] : 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[it][i] = bias;
    }
    wn_gemm_tile(p.w2t, Gh, O2, z_s, w_s, n_items, acc);     // (its first __syncthreads also publishes z_s)
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int item = threadIdx.x + it * 256;
      if (item >= n_items) break;
      const int o = item % O2, tg = item / O2;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int t = t0 + tg * 8 + i;
        if (t >= p.T) break;
        if (o < p.S) {
          float* sp = p.skips + ((size_t)b * p.S + o) * p.T + t;
          *sp = p.first ? acc[it][i] : *sp + acc[it][i];
        } else {
          const size_t off = ((size_t)b * p.R + (o - p.S)) * p.T + t;
          p.x_out[off] = acc[it][i] + p.x[off];
        }
      }
    }
  }
}

}  // namespace svsk

using namespace svsk;

// Checks shared by the inference and training entries; 0 and the dynamic shared memory in *smem, or SVSK_E_ARG.
static int wavenet_block_check(const svsk_wavenet_block_params& p, size_t* smem_out) {
  SVSK_REQUIRE(p.x && p.c && p.w1t && p.w2t && p.b2 && p.x_out && p.skips, SVSK_E_ARG, "wavenet_block_f32: null tensor");
  SVSK_REQUIRE(p.B > 0 && p.B <= 65535 && p.T > 0 && p.R > 0 && p.G > 0 && p.G % 2 == 0 && p.S > 0 && p.Cc > 0 && p.ksize >= 1 &&
                   p.dilation >= 1, SVSK_E_ARG, "wavenet_block_f32: bad sizes");
  SVSK_REQUIRE(p.x != p.x_out, SVSK_E_ARG, "wavenet_block_f32: x and x_out must differ (later frames read earlier taps)");
  SVSK_REQUIRE(p.G % 4 == 0 && (p.S + p.R) % 4 == 0 && p.G <= 256 && p.S + p.R <= 256, SVSK_E_ARG,
               "wavenet_block_f32: gate channels G=%d and S + R=%d must be multiples of 4, at most 256", p.G, p.S + p.R);
  const int wcols = p.G > p.S + p.R ? p.G : p.S + p.R;
  const size_t smem = (((size_t)(p.ksize * p.R + p.Cc) + p.G + p.G / 2) * kWnTT + (size_t)kWnKC * wcols) * sizeof(float);
  SVSK_REQUIRE(smem <= 200 * 1024, SVSK_E_ARG, "wavenet_block_f32: %zu bytes of shared memory (k R + cin + 1.5 G too large)", smem);
  *smem_out = smem;
  return 0;
}

template <bool kTrain>
static int wavenet_block_launch(const svsk_wavenet_block_params& p, float* y, size_t smem, void* stream, const char* what) {
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(wavenet_block_f32_kernel<kTrain>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(e));
    smem_set = smem;
  }
  dim3 grid((unsigned)ceil_div(p.T, kWnTT), (unsigned)p.B);
  wavenet_block_f32_kernel<kTrain><<<grid, 256, smem, as_stream(stream)>>>(p, y);
  return check_launch(what);
}

extern "C" int svsk_wavenet_block_f32(const svsk_wavenet_block_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "wavenet_block_f32: null params");
  size_t smem = 0;
  if (int rc = wavenet_block_check(*pp, &smem)) return rc;
  return wavenet_block_launch<false>(*pp, nullptr, smem, stream, "wavenet_block_f32");
}

extern "C" int svsk_wavenet_block_train_f32(const svsk_wavenet_block_train_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "wavenet_block_train_f32: null params");
  SVSK_REQUIRE(pp->y != nullptr, SVSK_E_ARG, "wavenet_block_train_f32: null tensor y");
  size_t smem = 0;
  if (int rc = wavenet_block_check(pp->blk, &smem)) return rc;
  return wavenet_block_launch<true>(pp->blk, pp->y, smem, stream, "wavenet_block_train_f32");
}
