// WaveNet training backward, fp32 on the CUDA cores (the forward is wavenet_f32.cu's block kernel with kTrain, which also
// keeps the gate pre-activations y).  Per training step, with L layers:
//   svsk_wavenet_train_pack_f32     1 launch   weight-norm fold of every weight, written in all the layouts used below
//   svsk_wavenet_dgrad_f32          L + 1      launch l: g_l = dL/dx_l for a 16-frame tile, then dy_{l-1} for the same tile
//   svsk_wavenet_wgrad_f32          1 or 2     every weight / bias gradient: 64 x 64 output tiles reduced over (b, t)
//   svsk_wavenet_wnorm_grad_f32     1          dg and dv of the weight-normed weights from the effective weights' gradients
// plus svsk_conv1d_f32 for the transposed 1x1s of the head, of first_conv (dx) and of all conditioning convs at once (dc),
// and svsk_relu_mask_f32 for the head's two ReLU derivatives.  Nothing uses atomics: every output element is written by
// one thread, and every sum runs in a fixed order, so gradients are bit-reproducible.
// The weight-norm fold here is the library's only one: the inference forward uses the same pack, and
// svsk_wavenet_ar_pack_f32 runs it with the sampler's layout.
#include "wavenet_f32.cuh"

namespace svsk {

// ------------------------------------------------------------------------------------------------------------------
// Layouts of the weight pack and the gradient arena (include/svsk.h); ops.py mirrors them.
// ------------------------------------------------------------------------------------------------------------------
struct WnTrainDims {
  long long out, R, G, G2, S, cin, L, k, Rp, G2p, K1;
  // pack
  long long w1t, w2t, wT, wB, wcT, first, firstT, last1, last1T, last3, last3T, pack_floats;
  // gradient arena
  long long conv, conv_b, cond, skip, skip_b, outw, out_b, gfirst, first_b, glast1, last1_b, glast3, last3_b, grad_floats;
};

static WnTrainDims train_dims(int out_dim, int R, int G, int S, int cin, int layers, int ksize) {
  WnTrainDims d{};
  d.out = out_dim; d.R = R; d.G = G; d.G2 = G / 2; d.S = S; d.cin = cin; d.L = layers; d.k = ksize;
  d.Rp = (R + 3) / 4 * 4; d.G2p = (d.G2 + 3) / 4 * 4; d.K1 = (long long)ksize * R + cin;
  long long o = 0;
  d.w1t = o;    o += d.L * d.K1 * G;
  d.w2t = o;    o += d.L * d.G2 * (S + R);
  d.wT = o;     o += d.L * d.k * G * d.Rp;
  d.wB = o;     o += d.L * (R + S) * d.G2p;
  d.wcT = o;    o += d.cin * d.L * G;
  d.first = o;  o += d.R * d.out;
  d.firstT = o; o += d.R * d.out;
  d.last1 = o;  o += d.S * d.S;
  d.last1T = o; o += d.S * d.S;
  d.last3 = o;  o += d.out * d.S;
  d.last3T = o; o += d.out * d.S;
  d.pack_floats = o;
  o = 0;
  d.conv = o;    o += d.L * G * R * d.k;
  d.conv_b = o;  o += d.L * G;
  d.cond = o;    o += d.L * G * d.cin;
  d.skip = o;    o += d.L * S * d.G2;
  d.skip_b = o;  o += d.L * S;
  d.outw = o;    o += d.L * R * d.G2;
  d.out_b = o;   o += d.L * R;
  d.gfirst = o;  o += d.R * d.out;
  d.first_b = o; o += d.R;
  d.glast1 = o;  o += d.S * d.S;
  d.last1_b = o; o += d.S;
  d.glast3 = o;  o += d.out * d.S;
  d.last3_b = o; o += d.out;
  d.grad_floats = o;
  return d;
}

// the shapes svsk_wavenet_block_f32 accepts (wavenet_f32.cu), for a whole network
static int train_shape_check(const char* what, int out_dim, int R, int G, int S, int cin, int layers, int ksize) {
  SVSK_REQUIRE(out_dim > 0 && R > 0 && G > 0 && S > 0 && cin > 0 && layers > 0 && ksize >= 1, SVSK_E_ARG, "%s: bad sizes", what);
  SVSK_REQUIRE(G % 4 == 0 && (S + R) % 4 == 0 && G <= 256 && S + R <= 256, SVSK_E_ARG,
               "%s: gate channels G=%d and S + R=%d must be multiples of 4, at most 256", what, G, S + R);
  const int wcols = G > S + R ? G : S + R;
  const size_t smem = (((size_t)ksize * R + cin + G + G / 2) * kWnTT + (size_t)kWnKC * wcols) * sizeof(float);
  SVSK_REQUIRE(smem <= 200 * 1024, SVSK_E_ARG, "%s: %zu bytes of shared memory for the block (k R + cin + 1.5 G too large)", what,
               smem);
  return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// Weight-norm fold and its gradient: one 256-thread CTA per output row of every weight.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kWnormBlock = 256;
constexpr int kWnGroups = 7;

struct WnDst {
  float* base;            // NULL: unused; element (layer l, row ro, input channel ci, tap j) goes to
  long long ls, rs, cs, js;  // base[l ls + ro rs + ci cs + j js]
};
struct WnBias {
  const float* src;       // NULL: zeros
  float* dst;             // NULL: no copy; row r (layer l, row ro) writes dst[l ls + ro] = src[r]
  long long ls;
};
struct WnGroup {
  const float* v;
  const float* g;         // NULL: no weight norm (w = v)
  int rows, rowsize, rpl, k;  // rows = layers * rpl; rowsize = cin * k (flat [ci][j] as in the conv weight)
  WnDst d[2];
  WnBias b;               // the sampler's pack writes its biases in the same launch
  long long dw, dg;       // offsets in the gradient arena / the dg vector (svsk_wavenet_wnorm_grad_f32)
};
struct WnGroups {
  WnGroup g[kWnGroups];
  int n;
  int row0[kWnGroups + 1];
};

// sum over the row of a[i] * b[i] in the order of torch's weight_norm_fwd_first_dim_kernel (256 threads, strided
// per-thread fma sums, shared-memory tree down to 64, then one warp): the fold gives the same bits as
// torch._weight_norm(v, g, 0) on CUDA, which the module's eval path uses.
__device__ __forceinline__ float wn_row_dot(const float* __restrict__ a, const float* __restrict__ b, int n, float* s) {
  const int tid = threadIdx.x;
  float ts = 0.f;
  for (int i = tid; i < n; i += kWnormBlock) ts = fmaf(a[i], b[i], ts);
  s[tid] = ts;
  __syncthreads();
#pragma unroll
  for (int i = kWnormBlock / 2; i >= 64; i >>= 1) {
    if (tid < i) s[tid] = s[tid] + s[tid + i];
    __syncthreads();
  }
  if (tid < 32) {
    float f = s[tid] + s[tid + 32];
#pragma unroll
    for (int i = 16; i >= 1; i >>= 1) f = f + __shfl_down_sync(0xffffffffu, f, i);
    if (tid == 0) s[0] = f;
  }
  __syncthreads();
  const float r = s[0];
  __syncthreads();  // s is reused by the next reduction
  return r;
}

__device__ __forceinline__ int wn_group_of(const WnGroups& G, int row) {
  int gi = 0;
  while (gi + 1 < G.n && row >= G.row0[gi + 1]) ++gi;
  return gi;
}

__global__ void __launch_bounds__(kWnormBlock) wavenet_wnorm_fold_kernel(const WnGroups G) {
  __shared__ float s[kWnormBlock];
  const int gi = wn_group_of(G, blockIdx.x);
  const WnGroup& q = G.g[gi];
  const int r = blockIdx.x - G.row0[gi];
  const float* v = q.v + (size_t)r * q.rowsize;
  float gg = 1.f, rnorm = 1.f;
  if (q.g) {
    const float nrm = sqrtf(wn_row_dot(v, v, q.rowsize, s));
    rnorm = 1.f / nrm;
    gg = q.g[r];
  }
  const int l = r / q.rpl, ro = r - l * q.rpl;
  for (int i = threadIdx.x; i < q.rowsize; i += kWnormBlock) {
    const float val = v[i];
    const float w = q.g ? gg * val * rnorm : val;
    const int ci = i / q.k, j = i - ci * q.k;
#pragma unroll
    for (int d = 0; d < 2; ++d)
      if (q.d[d].base) q.d[d].base[l * q.d[d].ls + ro * q.d[d].rs + ci * q.d[d].cs + j * q.d[d].js] = w;
  }
  if (q.b.dst && threadIdx.x == 0) q.b.dst[l * q.b.ls + ro] = q.b.src ? q.b.src[r] : 0.f;
}

__global__ void __launch_bounds__(kWnormBlock) wavenet_wnorm_grad_kernel(const WnGroups G, float* __restrict__ dW,
                                                                          float* __restrict__ dg) {
  __shared__ float s[kWnormBlock];
  const int gi = wn_group_of(G, blockIdx.x);
  const WnGroup& q = G.g[gi];
  const int r = blockIdx.x - G.row0[gi];
  const float* v = q.v + (size_t)r * q.rowsize;
  float* dw = dW + q.dw + (size_t)r * q.rowsize;
  const float nrm = sqrtf(wn_row_dot(v, v, q.rowsize, s));
  const float dgr = wn_row_dot(dw, v, q.rowsize, s) / nrm;   // <dw, v / ||v||>
  if (threadIdx.x == 0) dg[q.dg + r] = dgr;
  const float scale = q.g[r] / nrm;
  for (int i = threadIdx.x; i < q.rowsize; i += kWnormBlock) dw[i] = scale * (dw[i] - dgr * (v[i] / nrm));
}

static void wn_add(WnGroups& G, const float* v, const float* g, long long rows, long long rowsize, long long rpl, long long k,
                   WnDst d0, WnDst d1, WnBias b, long long dw, long long dg) {
  WnGroup& q = G.g[G.n];
  q.v = v; q.g = g; q.rows = (int)rows; q.rowsize = (int)rowsize; q.rpl = (int)rpl; q.k = (int)k;
  q.d[0] = d0; q.d[1] = d1; q.b = b; q.dw = dw; q.dg = dg;
  G.row0[G.n + 1] = G.row0[G.n] + (int)rows;
  ++G.n;
}

// The seven weights of svsk_wavenet_ar_weights as fold / gradient groups.  pack == NULL: no destinations (gradient).
static WnGroups wn_groups(const svsk_wavenet_ar_weights& w, const WnTrainDims& d, float* pack, bool only_normed) {
  WnGroups G{};
  auto add = [&](const float* v, const float* g, long long rows, long long rowsize, long long rpl, long long k, WnDst d0,
                 WnDst d1, long long dw, long long dg) {
    if (!only_normed || g) wn_add(G, v, g, rows, rowsize, rpl, k, d0, d1, {}, dw, dg);
  };
  auto P = [&](long long off) { return pack ? pack + off : nullptr; };
  const long long L = d.L, R = d.R, G_ = d.G, G2 = d.G2, S = d.S, k = d.k, out = d.out, cin = d.cin;
  long long dg = 0;
  // first [R][out]: natural, and transposed [out][R]
  add(w.first_v, w.first_g, R, out, R, 1, {P(d.first), 0, out, 1, 0}, {P(d.firstT), 0, 1, R, 0}, d.gfirst, dg);
  dg += R;
  // conv [L][G][R][k] -> w1t[l][(j R + ci)][co], wT[l][(j G + co)][ci]
  add(w.conv_v, w.conv_g, L * G_, R * k, G_, k, {P(d.w1t), d.K1 * G_, 1, G_, R * G_}, {P(d.wT), k * G_ * d.Rp, d.Rp, 1, G_ * d.Rp},
      d.conv, dg);
  dg += L * G_;
  // cond [L][G][cin] -> w1t[l][k R + cc][co], wcT[cc][l G + co]
  add(w.cond_v, w.cond_g, L * G_, cin, G_, 1, {P(d.w1t) ? P(d.w1t) + k * R * G_ : nullptr, d.K1 * G_, 1, G_, 0},
      {P(d.wcT), G_, 1, L * G_, 0}, d.cond, dg);
  dg += L * G_;
  // skip [L][S][G2] -> w2t[l][c2][s], wB[l][R + s][c2]
  add(w.skip_v, w.skip_g, L * S, G2, S, 1, {P(d.w2t), G2 * (S + R), 1, S + R, 0},
      {P(d.wB) ? P(d.wB) + R * d.G2p : nullptr, (R + S) * d.G2p, d.G2p, 1, 0}, d.skip, dg);
  dg += L * S;
  // out [L][R][G2] -> w2t[l][c2][S + o], wB[l][o][c2]
  add(w.out_v, w.out_g, L * R, G2, R, 1, {P(d.w2t) ? P(d.w2t) + S : nullptr, G2 * (S + R), 1, S + R, 0},
      {P(d.wB), (R + S) * d.G2p, d.G2p, 1, 0}, d.outw, dg);
  dg += L * R;
  add(w.last1_v, w.last1_g, S, S, S, 1, {P(d.last1), 0, S, 1, 0}, {P(d.last1T), 0, 1, S, 0}, d.glast1, dg);
  dg += S;
  add(w.last3_v, w.last3_g, out, S, out, 1, {P(d.last3), 0, S, 1, 0}, {P(d.last3T), 0, 1, out, 0}, d.glast3, dg);
  return G;
}

static int weights_check(const char* what, const svsk_wavenet_ar_weights* w) {
  SVSK_REQUIRE(w != nullptr, SVSK_E_ARG, "%s: null weights", what);
  SVSK_REQUIRE(w->first_v && w->conv_v && w->cond_v && w->skip_v && w->out_v && w->last1_v && w->last3_v, SVSK_E_ARG,
               "%s: null weight tensor", what);
  return train_shape_check(what, w->out_dim, w->R, w->G, w->S, w->cin, w->layers, w->ksize);
}

// ------------------------------------------------------------------------------------------------------------------
// dgrad: launch l of the backward through the blocks (svsk.h).  Shared memory: one tap of dy_l [G][16], [g_l ; dS]
// [R + S][16], weight chunk [32][max(Rp, G2p)].
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) wavenet_dgrad_kernel(const svsk_wavenet_dgrad_params p) {
  extern __shared__ float smem[];
  const int G2 = p.G / 2, Rp = (p.R + 3) / 4 * 4, G2p = (G2 + 3) / 4 * 4, KB = p.R + p.S;
  float* in_s = smem;
  float* gd_s = in_s + p.G * kWnTT;
  float* w_s = gd_s + KB * kWnTT;
  const int b = blockIdx.y, t0 = blockIdx.x * kWnTT;
  // ---- g_l = g_{l+1} + transposed dilated conv of dy_l: dx(t) gathers dy(t + (k-1-j) d) through tap j
  float acc[2][8];
#pragma unroll
  for (int it = 0; it < 2; ++it)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[it][i] = 0.f;
  if (p.dy_in) {
    const float* dyb = p.dy_in + (size_t)b * p.dy_bstride;
    for (int j = 0; j < p.ksize; ++j) {
      if (j) __syncthreads();                               // the previous tap has been consumed
      const long long sh = (long long)(p.ksize - 1 - j) * p.dilation;
      for (int i = threadIdx.x; i < p.G * kWnTT; i += 256) {
        const int co = i / kWnTT;
        const long long t = t0 + i % kWnTT + sh;
        in_s[i] = t < p.T ? dyb[(size_t)co * p.T + t] : 0.f;
      }
      wn_gemm_tile(p.wT + (size_t)j * p.G * Rp, p.G, Rp, in_s, w_s, 2 * Rp, acc);
    }
  }
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int item = threadIdx.x + it * 256;
    if (item >= 2 * Rp) break;
    const int r = item % Rp, tg = item / Rp;
    if (r >= p.R) continue;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int tt = tg * 8 + i, t = t0 + tt;
      float gv = 0.f;
      if (t < p.T) {
        const size_t off = ((size_t)b * p.R + r) * p.T + t;
        gv = acc[it][i] + (p.g_next ? p.g_next[off] : 0.f);
        p.g_out[off] = gv;
      }
      gd_s[r * kWnTT + tt] = gv;
    }
  }
  if (!p.y_prev) return;
  for (int i = threadIdx.x; i < p.S * kWnTT; i += 256) {
    const int s = i / kWnTT, t = t0 + i % kWnTT;
    gd_s[p.R * kWnTT + i] = t < p.T ? p.dS[((size_t)b * p.S + s) * p.T + t] : 0.f;
  }
  // ---- dz = [W_out ; W_skip]^T [g_l ; dS], then the gate derivative with block l-1's pre-activations
#pragma unroll
  for (int it = 0; it < 2; ++it)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[it][i] = 0.f;
  wn_gemm_tile(p.wB, KB, G2p, gd_s, w_s, 2 * G2p, acc);      // (its first __syncthreads also publishes gd_s)
  float* dyo = p.dy_out + (size_t)b * p.dy_bstride;
  const float* yb = p.y_prev + (size_t)b * p.G * p.T;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int item = threadIdx.x + it * 256;
    if (item >= 2 * G2p) break;
    const int c2 = item % G2p, tg = item / G2p;
    if (c2 >= G2) continue;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int t = t0 + tg * 8 + i;
      if (t >= p.T) break;
      const float a = yb[(size_t)c2 * p.T + t], g = yb[(size_t)(G2 + c2) * p.T + t];
      const float th = tanhf(a), sg = 1.f / (1.f + expf(-g));
      const float dz = acc[it][i];
      dyo[(size_t)c2 * p.T + t] = dz * sg * (1.f - th * th);
      dyo[(size_t)(G2 + c2) * p.T + t] = dz * th * sg * (1.f - sg);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// wgrad: out[m][n] = sum over (b, t) of P[b][m][t] Q[b][n][t], one 64 x 64 tile of one job per CTA, 32-frame chunks
// staged in shared memory (prefetched into registers one chunk ahead), 4 x 4 outputs per thread.
// Jobs, per layer l: A (P = dy_l; Q = x_l taps, c, ones -> conv, cond, conv_b), O (P = g_{l+1}; Q = z_l, ones -> out,
// out_b), K (P = dS; Q = z_l, ones -> skip, skip_b); then the head: H3 (P = dL/dlogits; Q = relu(h1), ones), H1
// (P = dh1; Q = relu(skips), ones), F (P = g_0; Q = x_in, ones).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kWgT = 64, kWgF = 32, kWgPitch = kWgT + 4;
enum { kQPlain = 0, kQRelu = 1, kQGate = 2, kQOnes = 3 };

struct WgCol {
  const float* q;     // row of Q at b = 0
  long long bstride;  // floats between tracks
  long long out;      // arena offset of (m = 0, this column); element m at out + m * ms
  int ms;
  int shift;          // Q read at t + shift (zero outside [0, T))
  int mode;
  int aux;            // kQGate: floats from the tanh row to the sigmoid row
};

struct WgArgs {
  svsk_wavenet_wgrad_params p;
  long long o_conv, o_conv_b, o_cond, o_skip, o_skip_b, o_out, o_out_b, o_first, o_first_b, o_last1, o_last1_b, o_last3, o_last3_b;
  long long grad_floats;
  int tA, tO, tK, tH3, tH1, tF;  // tiles per job
  int nnA, nnO, nnK, nnH3, nnH1, nnF;  // column tiles per job
};

__device__ __forceinline__ int wg_tiles(int M, int N) { return ((M + kWgT - 1) / kWgT) * ((N + kWgT - 1) / kWgT); }

__global__ void __launch_bounds__(256) wavenet_wgrad_kernel(const WgArgs A) {
  __shared__ __align__(16) float Ps[kWgF * kWgPitch];
  __shared__ __align__(16) float Qs[kWgF * kWgPitch];
  __shared__ WgCol cols[kWgT];
  const svsk_wavenet_wgrad_params& p = A.p;
  const int T = p.T, R = p.R, G = p.G, G2 = p.G / 2, S = p.S, L = p.layers, k = p.ksize;
  const size_t BT = (size_t)p.B * T;
  // ---- which job, which tile
  int tile = blockIdx.x, kind, l = 0, M, N, nn;
  const int per_layer = A.tA + A.tO + A.tK;
  if (tile < L * per_layer) {
    l = tile / per_layer;
    tile -= l * per_layer;
    if (tile < A.tA) { kind = 0; M = G; N = k * R + p.cin + 1; nn = A.nnA; }
    else if ((tile -= A.tA) < A.tO) { kind = 1; M = R; N = G2 + 1; nn = A.nnO; }
    else { tile -= A.tO; kind = 2; M = S; N = G2 + 1; nn = A.nnK; }
  } else {
    tile -= L * per_layer;
    if (tile < A.tH3) { kind = 3; M = p.out_dim; N = S + 1; nn = A.nnH3; }
    else if ((tile -= A.tH3) < A.tH1) { kind = 4; M = S; N = S + 1; nn = A.nnH1; }
    else { tile -= A.tH1; kind = 5; M = R; N = p.out_dim + 1; nn = A.nnF; }
  }
  const int m0 = (tile / nn) * kWgT, n0 = (tile % nn) * kWgT;
  const float* P;
  long long pb;
  switch (kind) {
    case 0: P = p.dy + (size_t)l * G * T; pb = (long long)L * G * T; break;
    case 1: P = p.gs + (size_t)(l + 1) * BT * R; pb = (long long)R * T; break;
    case 2: P = p.dS; pb = (long long)S * T; break;
    case 3: P = p.glog; pb = (long long)p.out_dim * T; break;
    case 4: P = p.dh1; pb = (long long)S * T; break;
    default: P = p.gs; pb = (long long)R * T; break;
  }
  // ---- column descriptors of this tile
  if (threadIdx.x < kWgT) {
    const int n = n0 + threadIdx.x;
    WgCol c{nullptr, 0, 0, 0, 0, kQPlain, 0};
    if (n < N) {
      const bool ones = n == N - 1;
      switch (kind) {
        case 0:
          if (ones) { c.mode = kQOnes; c.out = A.o_conv_b + (long long)l * G; c.ms = 1; }
          else if (n < k * R) {
            const int j = n / R, ci = n - j * R;
            c.q = p.xs + (size_t)l * BT * R + (size_t)ci * T; c.bstride = (long long)R * T;
            c.shift = -(k - 1 - j) * p.dilations[l];
            c.out = A.o_conv + (long long)l * G * R * k + (long long)ci * k + j; c.ms = R * k;
          } else {
            const int cc = n - k * R;
            c.q = p.c + (size_t)cc * T; c.bstride = (long long)p.cin * T;
            c.out = A.o_cond + (long long)l * G * p.cin + cc; c.ms = p.cin;
          }
          break;
        case 1:
        case 2: {
          const long long ow = kind == 1 ? A.o_out + (long long)l * R * G2 : A.o_skip + (long long)l * S * G2;
          const long long obias = kind == 1 ? A.o_out_b + (long long)l * R : A.o_skip_b + (long long)l * S;
          if (ones) { c.mode = kQOnes; c.out = obias; c.ms = 1; }
          else {
            c.mode = kQGate; c.q = p.ys + (size_t)l * BT * G + (size_t)n * T; c.bstride = (long long)G * T; c.aux = G2 * T;
            c.out = ow + n; c.ms = G2;
          }
          break;
        }
        case 3:
        case 4: {
          const float* src = kind == 3 ? p.h1 : p.skips;
          if (ones) { c.mode = kQOnes; c.out = kind == 3 ? A.o_last3_b : A.o_last1_b; c.ms = 1; }
          else {
            c.mode = kQRelu; c.q = src + (size_t)n * T; c.bstride = (long long)S * T;
            c.out = (kind == 3 ? A.o_last3 : A.o_last1) + n; c.ms = S;
          }
          break;
        }
        default:
          if (ones) { c.mode = kQOnes; c.out = A.o_first_b; c.ms = 1; }
          else { c.q = p.x_in + (size_t)n * T; c.bstride = (long long)p.out_dim * T; c.out = A.o_first + n; c.ms = p.out_dim; }
          break;
      }
    }
    cols[threadIdx.x] = c;
  }
  __syncthreads();
  // ---- this split's share of the (b, 32-frame chunk) sequence
  const int tch = (T + kWgF - 1) / kWgF;
  const long long nch = (long long)p.B * tch;
  const long long c_beg = nch * blockIdx.y / p.splits, c_end = nch * (blockIdx.y + 1) / p.splits;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // raw loads only (all in flight at once); the ReLU / gate transforms run when the chunk is staged
  float np_[8], nqa[8], nqb[8];
  auto fetch = [&](long long ch) {
    const int b = (int)(ch / tch);
    const int t = (int)(ch - (long long)b * tch) * kWgF + lane;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int m = m0 + warp + 8 * i;
      np_[i] = (m < M && t < T) ? P[(size_t)b * pb + (size_t)m * T + t] : 0.f;
      const WgCol& c = cols[warp + 8 * i];
      const int u = t + c.shift;
      const bool in = c.q && t < T && u >= 0 && u < T;
      const float* q = c.q + (size_t)b * c.bstride + u;
      nqa[i] = in ? q[0] : 0.f;
      nqb[i] = (in && c.mode == kQGate) ? q[c.aux] : 0.f;
    }
  };
  auto qval = [&](int i, int t) {
    const WgCol& c = cols[warp + 8 * i];
    if (c.mode == kQOnes) return t < T ? 1.f : 0.f;
    if (c.mode == kQRelu) return fmaxf(nqa[i], 0.f);
    if (c.mode == kQGate) return tanhf(nqa[i]) * (1.f / (1.f + expf(-nqb[i])));
    return nqa[i];
  };
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int tm = (threadIdx.x & 15) * 4, tn = (threadIdx.x >> 4) * 4;
  if (c_beg < c_end) fetch(c_beg);
  for (long long ch = c_beg; ch < c_end; ++ch) {
    __syncthreads();                                            // the previous chunk has been consumed
    const int tl = (int)(ch % tch) * kWgF + lane;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      Ps[lane * kWgPitch + warp + 8 * i] = np_[i];
      Qs[lane * kWgPitch + warp + 8 * i] = qval(i, tl);
    }
    __syncthreads();
    if (ch + 1 < c_end) fetch(ch + 1);
#pragma unroll 4
    for (int f = 0; f < kWgF; ++f) {
      const float4 a = *reinterpret_cast<const float4*>(Ps + f * kWgPitch + tm);
      const float4 q = *reinterpret_cast<const float4*>(Qs + f * kWgPitch + tn);
      const float av[4] = {a.x, a.y, a.z, a.w}, qv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], qv[j], acc[i][j]);
    }
  }
  float* dst = p.splits > 1 ? p.ws + (size_t)blockIdx.y * A.grad_floats : p.dW;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int nl = tn + j;
    if (n0 + nl >= N) break;
    const WgCol& c = cols[nl];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + tm + i;
      if (m < M) dst[c.out + (long long)m * c.ms] = acc[i][j];
    }
  }
}

__global__ void wavenet_wgrad_sum_kernel(const float* __restrict__ ws, float* __restrict__ dW, long long n, int splits) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float s = ws[i];
    for (int k = 1; k < splits; ++k) s += ws[(size_t)k * n + i];
    dW[i] = s;
  }
}

__global__ void relu_mask_kernel(const float* __restrict__ x, const float* __restrict__ m, float* y, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = m[i] > 0.f ? x[i] : 0.f;
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_wavenet_train_sizes(int out_dim, int R, int G, int S, int cin, int layers, int ksize, long long* pack_floats,
                                        long long* grad_floats) {
  if (int rc = train_shape_check("wavenet_train_sizes", out_dim, R, G, S, cin, layers, ksize)) return rc;
  const WnTrainDims d = train_dims(out_dim, R, G, S, cin, layers, ksize);
  if (pack_floats) *pack_floats = d.pack_floats;
  if (grad_floats) *grad_floats = d.grad_floats;
  return 0;
}

extern "C" int svsk_wavenet_train_pack_f32(const svsk_wavenet_ar_weights* w, float* pack, void* stream) {
  if (int rc = weights_check("wavenet_train_pack_f32", w)) return rc;
  SVSK_REQUIRE(pack != nullptr, SVSK_E_ARG, "wavenet_train_pack_f32: null pack");
  const WnTrainDims d = train_dims(w->out_dim, w->R, w->G, w->S, w->cin, w->layers, w->ksize);
  cudaStream_t st = as_stream(stream);
  if (d.Rp != d.R || d.G2p != d.G2) {   // zero padding columns of wT and wB (contiguous in the pack)
    cudaError_t e = cudaMemsetAsync(pack + d.wT, 0, (size_t)(d.wcT - d.wT) * sizeof(float), st);
    if (e != cudaSuccess) return fail((int)e, "wavenet_train_pack_f32: cudaMemsetAsync: %s", cudaGetErrorString(e));
  }
  const WnGroups G = wn_groups(*w, d, pack, false);
  wavenet_wnorm_fold_kernel<<<G.row0[G.n], kWnormBlock, 0, st>>>(G);
  return check_launch("wavenet_train_pack_f32");
}

// The sampler's pack (ArLayout, wavenet_f32.cuh): the same fold, so its weights are the forward's bits.
extern "C" int svsk_wavenet_ar_pack_f32(const svsk_wavenet_ar_weights* wp, float* wpack, float* wcond, void* stream) {
  SVSK_REQUIRE(wp != nullptr && wpack && wcond, SVSK_E_ARG, "wavenet_ar_pack_f32: null argument");
  const svsk_wavenet_ar_weights& w = *wp;
  SVSK_REQUIRE(w.first_v && w.first_b && w.conv_v && w.cond_v && w.skip_v && w.skip_b && w.out_v && w.out_b && w.last1_v &&
                   w.last1_b && w.last3_v && w.last3_b, SVSK_E_ARG, "wavenet_ar_pack_f32: null weight");
  const int O = w.out_dim, R = w.R, G = w.G, Gh = w.G / 2, S = w.S, L = w.layers, k = w.ksize, cin = w.cin;
  SVSK_REQUIRE(cin > 0 && ar_supported(O, R, G, S, L, w.stacks, k), SVSK_E_ARG,
               "wavenet_ar_pack_f32: unsupported WaveNet (out %d, R %d, G %d, S %d, cin %d, layers %d, stacks %d, k %d)", O, R,
               G, S, cin, L, w.stacks, k);
  const ArLayout a = ar_layout(O, R, G, S, L, w.stacks, k);
  const long long ls = a.layer_stride;
  float* lay = wpack + a.layer0;
  WnGroups Q{};
  // first_conv [R][out] -> WfT [out][R], bf
  wn_add(Q, w.first_v, w.first_g, R, O, R, 1, {wpack + a.first_w, 0, 1, R, 0}, {}, {w.first_b, wpack + a.first_b, 0}, 0, 0);
  // conv [L][G][R][k] -> Wg [G][k R] (column j R + r), bg
  wn_add(Q, w.conv_v, w.conv_g, (long long)L * G, R * k, G, k, {lay + a.gw, ls, k * R, 1, R}, {}, {w.conv_b, lay + a.gb, ls}, 0, 0);
  // conv1x1_skip [L][S][G/2], conv1x1_out [L][R][G/2] -> Wso rows 0 .. S-1 and S .. S+R-1, bso
  wn_add(Q, w.skip_v, w.skip_g, (long long)L * S, Gh, S, 1, {lay + a.sw, ls, Gh, 1, 0}, {}, {w.skip_b, lay + a.sb, ls}, 0, 0);
  wn_add(Q, w.out_v, w.out_g, (long long)L * R, Gh, R, 1, {lay + a.sw + (long long)S * Gh, ls, Gh, 1, 0}, {},
         {w.out_b, lay + a.sb + S, ls}, 0, 0);
  // last_conv_layers.1 / .3
  wn_add(Q, w.last1_v, w.last1_g, S, S, S, 1, {wpack + a.w3, 0, S, 1, 0}, {}, {w.last1_b, wpack + a.b3, 0}, 0, 0);
  wn_add(Q, w.last3_v, w.last3_g, O, S, O, 1, {wpack + a.w4, 0, S, 1, 0}, {}, {w.last3_b, wpack + a.b4, 0}, 0, 0);
  // conv1x1c [L][G][cin] -> wcond [L G][cin] (no bias)
  wn_add(Q, w.cond_v, w.cond_g, (long long)L * G, cin, G, 1, {wcond, (long long)G * cin, cin, 1, 0}, {}, {}, 0, 0);
  wavenet_wnorm_fold_kernel<<<Q.row0[Q.n], kWnormBlock, 0, as_stream(stream)>>>(Q);
  return check_launch("wavenet_ar_pack_f32");
}

extern "C" int svsk_wavenet_wnorm_grad_f32(const svsk_wavenet_ar_weights* w, float* dW, float* dg, void* stream) {
  if (int rc = weights_check("wavenet_wnorm_grad_f32", w)) return rc;
  SVSK_REQUIRE(dW && dg, SVSK_E_ARG, "wavenet_wnorm_grad_f32: null dW or dg");
  const WnTrainDims d = train_dims(w->out_dim, w->R, w->G, w->S, w->cin, w->layers, w->ksize);
  const WnGroups G = wn_groups(*w, d, nullptr, true);
  if (G.n == 0) return 0;               // no weight norm anywhere: dW already is the parameters' gradient
  wavenet_wnorm_grad_kernel<<<G.row0[G.n], kWnormBlock, 0, as_stream(stream)>>>(G, dW, dg);
  return check_launch("wavenet_wnorm_grad_f32");
}

extern "C" int svsk_wavenet_dgrad_f32(const svsk_wavenet_dgrad_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "wavenet_dgrad_f32: null params");
  const svsk_wavenet_dgrad_params& p = *pp;
  SVSK_REQUIRE(p.g_out && p.dS, SVSK_E_ARG, "wavenet_dgrad_f32: null g_out or dS");
  SVSK_REQUIRE((p.dy_in == nullptr) == (p.wT == nullptr), SVSK_E_ARG, "wavenet_dgrad_f32: dy_in and wT go together");
  SVSK_REQUIRE(!p.y_prev || (p.wB && p.dy_out), SVSK_E_ARG, "wavenet_dgrad_f32: y_prev needs wB and dy_out");
  SVSK_REQUIRE(p.B > 0 && p.B <= 65535 && p.T > 0 && p.ksize >= 1 && p.dilation >= 1, SVSK_E_ARG, "wavenet_dgrad_f32: bad sizes");
  SVSK_REQUIRE(p.R > 0 && p.S > 0 && p.G > 0 && p.G % 4 == 0 && (p.S + p.R) % 4 == 0 && p.G <= 256 && p.S + p.R <= 256, SVSK_E_ARG,
               "wavenet_dgrad_f32: gate channels G=%d and S + R=%d must be multiples of 4, at most 256", p.G, p.S + p.R);
  SVSK_REQUIRE(p.dy_bstride >= (long long)p.G * p.T, SVSK_E_ARG, "wavenet_dgrad_f32: dy_bstride %lld < G T", p.dy_bstride);
  const int Rp = (p.R + 3) / 4 * 4, G2p = (p.G / 2 + 3) / 4 * 4;
  const int wcols = Rp > G2p ? Rp : G2p;
  const size_t smem = ((size_t)(p.G + p.R + p.S) * kWnTT + (size_t)kWnKC * wcols) * sizeof(float);
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(wavenet_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "wavenet_dgrad_f32: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    smem_set = smem;
  }
  dim3 grid((unsigned)ceil_div(p.T, kWnTT), (unsigned)p.B);
  wavenet_dgrad_kernel<<<grid, 256, smem, as_stream(stream)>>>(p);
  return check_launch("wavenet_dgrad_f32");
}

extern "C" int svsk_wavenet_wgrad_f32(const svsk_wavenet_wgrad_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "wavenet_wgrad_f32: null params");
  const svsk_wavenet_wgrad_params& p = *pp;
  SVSK_REQUIRE(p.x_in && p.c && p.xs && p.ys && p.gs && p.dy && p.dS && p.skips && p.h1 && p.dh1 && p.glog && p.dilations && p.dW,
               SVSK_E_ARG, "wavenet_wgrad_f32: null tensor");
  if (int rc = train_shape_check("wavenet_wgrad_f32", p.out_dim, p.R, p.G, p.S, p.cin, p.layers, p.ksize)) return rc;
  SVSK_REQUIRE(p.B > 0 && p.T > 0 && p.splits >= 1 && p.splits <= 65535, SVSK_E_ARG, "wavenet_wgrad_f32: bad sizes");
  SVSK_REQUIRE(p.splits == 1 || p.ws, SVSK_E_ARG, "wavenet_wgrad_f32: splits > 1 needs the workspace ws");
  const WnTrainDims d = train_dims(p.out_dim, p.R, p.G, p.S, p.cin, p.layers, p.ksize);
  WgArgs A{};
  A.p = p;
  A.o_conv = d.conv; A.o_conv_b = d.conv_b; A.o_cond = d.cond; A.o_skip = d.skip; A.o_skip_b = d.skip_b; A.o_out = d.outw;
  A.o_out_b = d.out_b; A.o_first = d.gfirst; A.o_first_b = d.first_b; A.o_last1 = d.glast1; A.o_last1_b = d.last1_b;
  A.o_last3 = d.glast3; A.o_last3_b = d.last3_b; A.grad_floats = d.grad_floats;
  auto tiles = [](long long M, long long N, int* nn) { *nn = (int)ceil_div_ll(N, kWgT); return (int)(ceil_div_ll(M, kWgT) * *nn); };
  A.tA = tiles(p.G, (long long)p.ksize * p.R + p.cin + 1, &A.nnA);
  A.tO = tiles(p.R, p.G / 2 + 1, &A.nnO);
  A.tK = tiles(p.S, p.G / 2 + 1, &A.nnK);
  A.tH3 = tiles(p.out_dim, p.S + 1, &A.nnH3);
  A.tH1 = tiles(p.S, p.S + 1, &A.nnH1);
  A.tF = tiles(p.R, p.out_dim + 1, &A.nnF);
  const long long total = (long long)p.layers * (A.tA + A.tO + A.tK) + A.tH3 + A.tH1 + A.tF;
  SVSK_REQUIRE(total < (1ll << 31), SVSK_E_ARG, "wavenet_wgrad_f32: too many tiles");
  cudaStream_t st = as_stream(stream);
  wavenet_wgrad_kernel<<<dim3((unsigned)total, (unsigned)p.splits), 256, 0, st>>>(A);
  if (int rc = check_launch("wavenet_wgrad_f32")) return rc;
  if (p.splits == 1) return 0;
  const long long blocks = ceil_div_ll(d.grad_floats, 256);
  wavenet_wgrad_sum_kernel<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, st>>>(p.ws, p.dW, d.grad_floats, p.splits);
  return check_launch("wavenet_wgrad_f32 (split sum)");
}

extern "C" int svsk_relu_mask_f32(const float* x, const float* m, float* y, long long n, void* stream) {
  SVSK_REQUIRE(x && m && y, SVSK_E_ARG, "relu_mask_f32: null tensor");
  SVSK_REQUIRE(n > 0, SVSK_E_ARG, "relu_mask_f32: bad size");
  const long long blocks = ceil_div_ll(n, 256);
  relu_mask_kernel<<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, as_stream(stream)>>>(x, m, y, n);
  return check_launch("relu_mask_f32");
}
