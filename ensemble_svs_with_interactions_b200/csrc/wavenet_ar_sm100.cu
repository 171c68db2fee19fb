// WaveNet autoregressive sampling in one launch, fp32 — replaces the host loop of WaveNet.inference
// (nnsvs/wavenet/wavenet.py:89-149: per step incremental_forward of every layer, softmax, OneHotCategorical draw).
//
// One CTA of 1024 threads per track runs all `steps` steps.  Per step and layer the work is two matrix-vector products
// (gate [G][k R] . taps, skip|out [S + R][G/2] . z: 32 768 weights = 128 KiB at the default widths), far too small for
// tensor cores and far too large (1.3 MiB for ten layers) to keep in one SM's shared memory.  The weights therefore
// stay in global memory, where all tracks read the same copy out of L2, and each phase is shaped so that a warp issues
// all of its weight loads before it needs any of them: one L2 round trip per phase, 2 per layer, 2 for the output convs.
// With one CTA per track the kernel runs up to one track per SM at once (148 on a B200) — a cluster that holds a
// track's weights in shared memory would need 8 SMs per track at the default widths (DESIGN §4).
//
// The dilated taps x_l[t - m d] (m = 1 .. k-1) were final at least one step earlier, so all of them, for all layers,
// are gathered at the start of a step together with the step's conditioning products, in one round trip.  They live
// in a per-track ring buffer in global memory (`hist`, (k-1) d_l + 1 frames of layer l); slots that would precede
// frame 0 read as zeros, exactly what the zero-initialised ring buffer of conv.py:21-53 gives.
#include <climits>

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

// The shapes the kernel's fixed register tiles cover (see the warp_rows instantiations below).
inline bool ar_supported(int O, int R, int G, int S, int L, int stacks, int k) {
  if (O < 1 || R < 1 || G < 2 || G % 2 || S < 1 || L < 1 || stacks < 1 || k < 1) return false;
  if (L > kArMaxLayers || L % stacks || L / stacks > 16) return false;
  // gate: k R <= 8 x 32 weights per lane, 2 pairs per warp; skip|out: K = G/2 <= 2 x 32, S + R <= 4 rows per warp;
  // last1: S <= 2 x 32; last3: out_dim <= 8 rows per warp
  if (k * R > 8 * 32 || G / 2 > 2 * 32 || S + R > 4 * kArWarps || S > 2 * 32 || O > 8 * kArWarps) return false;
  const ArLayout a = ar_layout(O, R, G, S, L, stacks, k);
  return a.smem <= 48 * 1024 && a.hist <= (1LL << 30) && a.total <= (1LL << 30);
}

__device__ __forceinline__ float warp_sum(float s) {
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}

// acc[i] = sum_{q<K} W[row_i][q] * f(v[q]) for the NR rows row_i = row_of(i) (< 0: no row), one warp per row: every
// lane first loads its NQ (K <= 32 NQ) weights of all NR rows, so the warp's whole share of the phase is in flight at
// once, then multiplies and reduces.  All lanes receive the sums.
template <int NR, int NQ, bool RELU, class RowOf>
__device__ __forceinline__ void warp_rows(const float* __restrict__ W, int K, const float* v, int lane, RowOf row_of,
                                          float (&acc)[NR]) {
  float w[NR][NQ];
#pragma unroll
  for (int i = 0; i < NR; ++i) {
    const int row = row_of(i);
#pragma unroll
    for (int j = 0; j < NQ; ++j) {
      const int q = lane + 32 * j;
      w[i][j] = (row >= 0 && q < K) ? __ldg(W + (size_t)row * K + q) : 0.f;
    }
  }
#pragma unroll
  for (int i = 0; i < NR; ++i) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < NQ; ++j) {
      const int q = lane + 32 * j;
      if (q < K) s = fmaf(w[i][j], RELU ? fmaxf(v[q], 0.f) : v[q], s);
    }
    acc[i] = warp_sum(s);
  }
}

__global__ void __launch_bounds__(kArThreads, 1) wavenet_ar_kernel(const svsk_wavenet_ar_params p, const ArLayout a) {
  extern __shared__ float smem[];
  const int O = p.out_dim, R = p.R, G = p.G, Gh = p.G / 2, S = p.S, L = p.layers, k = p.ksize, kR = k * R;
  const int tapR = (k - 1) * R;                  // taps before the current frame, per layer
  float* vin = smem;                             // [L][k R]: layer l's conv input (taps j < k-1, then x_l[t])
  float* cp = vin + L * kR;                      // [L][G]: conditioning products of frame t
  float* z = cp + L * G;                         // [G/2]
  float* skip = z + Gh;                          // [S]
  float* h3 = skip + S;                          // [S]
  float* lg = h3 + S;                            // [O] logits
  float* ex = lg + O;                            // [O] exp(logit - max)
  int* dil = reinterpret_cast<int*>(ex + O);     // [L]
  int* hoff = dil + L;                           // [L] ring offset (floats)
  int* hlen = hoff + L;                          // [L] ring length (frames)
  int* ycur = hlen + L;                          // class drawn at the previous step

  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* wp = p.wpack;
  float* hist = p.hist + (size_t)b * a.hist;
  const size_t LG = (size_t)L * G;
  const float* cpb = p.cproj + (size_t)b * LG * p.T;
  if (tid == 0) {
    const int per = L / p.stacks;
    int off = 0;
    for (int l = 0; l < L; ++l) {
      dil[l] = 1 << (l % per);
      hlen[l] = (k - 1) * dil[l] + 1;
      hoff[l] = off;
      off += hlen[l] * R;
    }
    *ycur = -1;
  }
  __syncthreads();

  for (int t = 0; t < p.steps; ++t) {
    // ---- gather: taps of every layer, conditioning products, x_0 = first_conv(onehot(y[t-1])) (bias alone at t = 0)
    for (int i = tid; i < L * tapR; i += kArThreads) {
      const int l = i / tapR, q = i - l * tapR, j = q / R, r = q - j * R;
      const int s = t - (k - 1 - j) * dil[l];
      vin[l * kR + q] = s >= 0 ? __ldcg(hist + hoff[l] + (size_t)(s % hlen[l]) * R + r) : 0.f;
    }
    for (int i = tid; i < L * G; i += kArThreads) cp[i] = __ldg(cpb + (size_t)i * p.T + t);
    if (tid < R) {
      const int y = *ycur;
      const float x0 = (y >= 0 ? __ldg(wp + a.first_w + (size_t)y * R + tid) : 0.f) + __ldg(wp + a.first_b + tid);
      vin[tapR + tid] = x0;
      hist[hoff[0] + (t % hlen[0]) * R + tid] = x0;
    }
    if (tid < S) skip[tid] = 0.f;
    __syncthreads();

    for (int l = 0; l < L; ++l) {
      const float* lw = wp + a.layer0 + (size_t)l * a.layer_stride;
      const float* xl = vin + l * kR;
      // ---- gate: warp w owns gate pairs w and w + 32 (tanh row j and sigmoid row j + G/2 together)
      {
        float acc[4];
        warp_rows<4, 8, false>(lw + a.gw, kR, xl, lane, [&](int i) {
          const int pr = warp + (i >> 1) * kArWarps;
          return pr < Gh ? pr + (i & 1) * Gh : -1;
        }, acc);
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < 4; i += 2) {
            const int pr = warp + (i >> 1) * kArWarps;
            if (pr < Gh) {
              const float ga = acc[i] + __ldg(lw + a.gb + pr) + cp[l * G + pr];
              const float gb = acc[i + 1] + __ldg(lw + a.gb + Gh + pr) + cp[l * G + Gh + pr];
              z[pr] = tanhf(ga) * (1.f / (1.f + expf(-gb)));
            }
          }
        }
      }
      __syncthreads();
      // ---- skip (rows < S) and out (rows S ..) projections of z; the last layer's x_{L} is never read
      {
        const int rows = l + 1 < L ? S + R : S;
        float acc[4];
        warp_rows<4, 2, false>(lw + a.sw, Gh, z, lane, [&](int i) {
          const int o = warp + i * kArWarps;
          return o < rows ? o : -1;
        }, acc);
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int o = warp + i * kArWarps;
            if (o >= rows) break;
            const float v = acc[i] + __ldg(lw + a.sb + o);
            if (o < S) {
              skip[o] += v;
            } else {
              const int r = o - S;
              const float xn = v + xl[tapR + r];
              vin[(l + 1) * kR + tapR + r] = xn;
              hist[hoff[l + 1] + (t % hlen[l + 1]) * R + r] = xn;
            }
          }
        }
      }
      __syncthreads();
    }
    // ---- logits = W4 relu(W3 relu(skip) + b3) + b4
    {
      float acc[2];
      warp_rows<2, 2, true>(wp + a.w3, S, skip, lane, [&](int i) {
        const int o = warp + i * kArWarps;
        return o < S ? o : -1;
      }, acc);
      if (lane == 0)
        for (int i = 0; i < 2; ++i) {
          const int o = warp + i * kArWarps;
          if (o < S) h3[o] = acc[i] + __ldg(wp + a.b3 + o);
        }
    }
    __syncthreads();
    {
      float acc[8];
      warp_rows<8, 2, true>(wp + a.w4, S, h3, lane, [&](int i) {
        const int o = warp + i * kArWarps;
        return o < O ? o : -1;
      }, acc);
      if (lane == 0)
        for (int i = 0; i < 8; ++i) {
          const int o = warp + i * kArWarps;
          if (o < O) lg[o] = acc[i] + __ldg(wp + a.b4 + o);
        }
    }
    __syncthreads();
    // ---- draw: y = smallest c with u < P_c (cumulative softmax in class order: lane chunks of consecutive classes,
    // then an exclusive scan of the chunk sums); largest c with p_c > 0 if rounding leaves none
    if (warp == 0) {
      const int per = (O + 31) / 32, c0 = min(O, lane * per), c1 = min(O, c0 + per);
      float m = -INFINITY;
      for (int c = c0; c < c1; ++c) m = fmaxf(m, lg[c]);
#pragma unroll
      for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      float part = 0.f;
      for (int c = c0; c < c1; ++c) {
        const float e = expf(lg[c] - m);
        ex[c] = e;
        part += e;
      }
      float incl = part;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      const float total = __shfl_sync(0xffffffffu, incl, 31);
      const float thr = __ldg(p.u + (size_t)b * p.steps + t) * total;
      float cum = incl - part;
      int pick = INT_MAX, last = -1;
      for (int c = c0; c < c1; ++c) {
        cum += ex[c];
        if (pick == INT_MAX && thr < cum) pick = c;
        if (ex[c] > 0.f) last = c;
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        pick = min(pick, __shfl_xor_sync(0xffffffffu, pick, o));
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
      }
      if (lane == 0) *ycur = pick != INT_MAX ? pick : last;
    }
    __syncthreads();
    const int y = *ycur;
    float* yrow = p.y + ((size_t)b * p.steps + t) * O;
    for (int c = tid; c < O; c += kArThreads) {
      yrow[c] = c == y ? 1.f : 0.f;
      if (p.logits) p.logits[((size_t)b * p.steps + t) * O + c] = lg[c];
    }
    // the next step's gather writes vin / skip only, which nothing after the barrier above reads; lg and ycur are
    // rewritten only after its first barrier
  }
}

// dst[layer * lstride + o * ostride + (j * inner + ci) * cstride] = v[layer][o][ci][j] * (g ? g[layer][o] / ||v[layer][o]|| : 1)
// and bdst[layer * lstride + o] = bias[layer][o] (0 when bias is NULL; nothing when bdst is NULL).  One CTA per row o.
__global__ void __launch_bounds__(128) wavenet_ar_fold_kernel(const float* __restrict__ v, const float* __restrict__ g,
                                                              const float* __restrict__ bias, float* __restrict__ dst,
                                                              float* __restrict__ bdst, int rows, int inner, int k,
                                                              long long lstride, int ostride, int cstride) {
  __shared__ float red[4];
  const int row = blockIdx.x, layer = row / rows, o = row - layer * rows, n = inner * k;
  const float* vr = v + (size_t)row * n;
  float scale = 1.f;
  if (g) {
    float s = 0.f;
    for (int i = threadIdx.x; i < n; i += 128) s = fmaf(vr[i], vr[i], s);
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    scale = g[row] / sqrtf(red[0] + red[1] + red[2] + red[3]);
  }
  float* d = dst + layer * lstride + (size_t)o * ostride;
  for (int i = threadIdx.x; i < n; i += 128) {
    const int ci = i / k, j = i - ci * k;
    d[(size_t)(j * inner + ci) * cstride] = vr[i] * scale;
  }
  if (bdst && threadIdx.x == 0) bdst[layer * lstride + o] = bias ? bias[row] : 0.f;
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_wavenet_ar_supported(int out_dim, int R, int G, int S, int layers, int stacks, int ksize) {
  return ar_supported(out_dim, R, G, S, layers, stacks, ksize) ? 1 : 0;
}

extern "C" int svsk_wavenet_ar_sizes(int out_dim, int R, int G, int S, int layers, int stacks, int ksize, long long* pack_floats,
                                     long long* hist_floats) {
  SVSK_REQUIRE(pack_floats && hist_floats, SVSK_E_ARG, "wavenet_ar_sizes: null output");
  SVSK_REQUIRE(ar_supported(out_dim, R, G, S, layers, stacks, ksize), SVSK_E_ARG,
               "wavenet_ar_sizes: unsupported WaveNet (out %d, R %d, G %d, S %d, layers %d, stacks %d, k %d)", out_dim, R, G,
               S, layers, stacks, ksize);
  const ArLayout a = ar_layout(out_dim, R, G, S, layers, stacks, ksize);
  *pack_floats = a.total;
  *hist_floats = a.hist;
  return 0;
}

extern "C" int svsk_wavenet_ar_pack_f32(const svsk_wavenet_ar_weights* wp, float* wpack, float* wcond, void* stream) {
  SVSK_REQUIRE(wp != nullptr && wpack && wcond, SVSK_E_ARG, "wavenet_ar_pack_f32: null argument");
  const svsk_wavenet_ar_weights& w = *wp;
  SVSK_REQUIRE(w.first_v && w.first_b && w.conv_v && w.cond_v && w.skip_v && w.skip_b && w.out_v && w.out_b && w.last1_v &&
                   w.last1_b && w.last3_v && w.last3_b, SVSK_E_ARG, "wavenet_ar_pack_f32: null weight");
  const int O = w.out_dim, R = w.R, G = w.G, Gh = w.G / 2, S = w.S, L = w.layers, k = w.ksize;
  SVSK_REQUIRE(w.cin > 0 && ar_supported(O, R, G, S, L, w.stacks, k), SVSK_E_ARG,
               "wavenet_ar_pack_f32: unsupported WaveNet (out %d, R %d, G %d, S %d, cin %d, layers %d, stacks %d, k %d)", O, R,
               G, S, w.cin, L, w.stacks, k);
  const ArLayout a = ar_layout(O, R, G, S, L, w.stacks, k);
  cudaStream_t st = as_stream(stream);
  const long long ls = a.layer_stride;
  // first_conv [R][out][1] -> WfT [out][R]
  wavenet_ar_fold_kernel<<<R, 128, 0, st>>>(w.first_v, w.first_g, w.first_b, wpack + a.first_w, wpack + a.first_b, R, O, 1, 0, 1, R);
  // conv [L][G][R][k] -> Wg [G][k R], bg
  wavenet_ar_fold_kernel<<<L * G, 128, 0, st>>>(w.conv_v, w.conv_g, w.conv_b, wpack + a.layer0 + a.gw, wpack + a.layer0 + a.gb,
                                                G, R, k, ls, k * R, 1);
  // conv1x1_skip [L][S][G/2], conv1x1_out [L][R][G/2] -> Wso rows 0 .. S-1 and S .. S+R-1
  wavenet_ar_fold_kernel<<<L * S, 128, 0, st>>>(w.skip_v, w.skip_g, w.skip_b, wpack + a.layer0 + a.sw, wpack + a.layer0 + a.sb,
                                                S, Gh, 1, ls, Gh, 1);
  wavenet_ar_fold_kernel<<<L * R, 128, 0, st>>>(w.out_v, w.out_g, w.out_b, wpack + a.layer0 + a.sw + (long long)S * Gh,
                                                wpack + a.layer0 + a.sb + S, R, Gh, 1, ls, Gh, 1);
  // last_conv_layers.1 / .3
  wavenet_ar_fold_kernel<<<S, 128, 0, st>>>(w.last1_v, w.last1_g, w.last1_b, wpack + a.w3, wpack + a.b3, S, S, 1, 0, S, 1);
  wavenet_ar_fold_kernel<<<O, 128, 0, st>>>(w.last3_v, w.last3_g, w.last3_b, wpack + a.w4, wpack + a.b4, O, S, 1, 0, S, 1);
  // conv1x1c [L][G][cin] -> wcond [L G][cin] (no bias)
  wavenet_ar_fold_kernel<<<L * G, 128, 0, st>>>(w.cond_v, w.cond_g, nullptr, wcond, nullptr, L * G, w.cin, 1, 0, w.cin, 1);
  return check_launch("wavenet_ar_pack_f32");
}

extern "C" int svsk_wavenet_ar_f32(const svsk_wavenet_ar_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "wavenet_ar_f32: null params");
  const svsk_wavenet_ar_params& p = *pp;
  SVSK_REQUIRE(p.wpack && p.cproj && p.u && p.y && p.hist, SVSK_E_ARG, "wavenet_ar_f32: null tensor");
  SVSK_REQUIRE(p.B > 0 && p.B <= (1 << 30) && p.T > 0 && p.steps > 0, SVSK_E_ARG, "wavenet_ar_f32: bad sizes B=%d T=%d steps=%d",
               p.B, p.T, p.steps);
  SVSK_REQUIRE(p.steps <= p.T, SVSK_E_ARG, "wavenet_ar_f32: steps=%d exceeds the %d conditioning frames", p.steps, p.T);
  SVSK_REQUIRE(ar_supported(p.out_dim, p.R, p.G, p.S, p.layers, p.stacks, p.ksize), SVSK_E_ARG,
               "wavenet_ar_f32: unsupported WaveNet (out %d, R %d, G %d, S %d, layers %d, stacks %d, k %d)", p.out_dim, p.R, p.G,
               p.S, p.layers, p.stacks, p.ksize);
  const ArLayout a = ar_layout(p.out_dim, p.R, p.G, p.S, p.layers, p.stacks, p.ksize);
  wavenet_ar_kernel<<<p.B, kArThreads, a.smem, as_stream(stream)>>>(p, a);
  return check_launch("wavenet_ar_f32");
}
