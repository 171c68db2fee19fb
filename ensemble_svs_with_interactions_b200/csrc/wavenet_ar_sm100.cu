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

#include "wavenet_f32.cuh"

namespace svsk {

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
