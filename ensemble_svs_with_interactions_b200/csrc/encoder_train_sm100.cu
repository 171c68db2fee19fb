// FFConvLSTM encoder backward, fp32 on the CUDA cores (the training forward is fp32: svsk_conv1d_f32, the BatchNorm batch
// statistics of encoder_sm100.cu and svsk_lstm_train_f32).  Per training step with three conv layers and two LSTM layers:
//   svsk_wgrad_f32           every weight and bias gradient: Linear / Conv1d k = 7 / W_ih / W_hh (one launch each, plus a
//                            fixed-order reduction of the frame splits)
//   svsk_bn_relu_bwd_f32     BatchNorm1d (batch statistics) + ReLU backward, one launch per conv layer
//   svsk_reflect_fold_f32    ReflectionPad1d backward: the padded rows of the k = 7 conv's data gradient, folded back
//   svsk_lstm_bwd_f32        the recurrences (lstm_train_sm100.cu)
// The data gradients of the Linears / convs / input projections are svsk_conv1d_f32 with transposed (flipped) weights and
// svsk_relu_mask_f32.  Nothing uses atomics and every sum runs in a fixed order: gradients are bit-reproducible.
#include "svsk_common.cuh"

namespace svsk {

// ------------------------------------------------------------------------------------------------------------------
// dW[n][c] = sum_b sum_t dY[b][n][t] X~[b][c][t] over 64 x 64 output tiles, c = k * ksize + j with
// X~[b][c][t] = X[b][k][t + j - origin] (zero or reflected outside [0, T)), and c = K * ksize the bias column (X~ = 1).
// Split s reduces the 32-frame chunks [s * nch / splits, (s+1) * nch / splits) of the (b, t) chunk list.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kWgTile = 64, kWgChunk = 32;

struct WgradArgs {
  const float* dy;
  const float* x;
  float* dw;
  float* db;
  float* ws;
  long long dy_sb, x_sb;
  int B, N, K, T, ksize, origin, reflect, splits, KK, ncols;
};

__device__ __forceinline__ int wg_src(int u, int T, int reflect) {
  if (u >= 0 && u < T) return u;
  if (!reflect) return -1;
  return u < 0 ? -u : 2 * (T - 1) - u;
}

__global__ void __launch_bounds__(256) wgrad_kernel(const WgradArgs a) {
  __shared__ float sdy[kWgChunk][kWgTile + 4];
  __shared__ float sx[kWgChunk][kWgTile + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n0 = blockIdx.y * kWgTile, c0 = blockIdx.x * kWgTile, split = blockIdx.z;
  const int tch = (a.T + kWgChunk - 1) / kWgChunk, nch = a.B * tch;
  const int ch0 = (int)((long long)split * nch / a.splits), ch1 = (int)((long long)(split + 1) * nch / a.splits);
  float acc[4][4] = {};
  for (int ch = ch0; ch < ch1; ++ch) {
    const int b = ch / tch, t0 = (ch % tch) * kWgChunk;
    __syncthreads();
    for (int i = tid; i < kWgTile * kWgChunk; i += 256) {
      const int r = i / kWgChunk, tt = i % kWgChunk, t = t0 + tt;
      const int n = n0 + r, cc = c0 + r;
      float vy = 0.f, vx = 0.f;
      if (t < a.T) {
        if (n < a.N) vy = a.dy[(size_t)b * a.dy_sb + (size_t)n * a.T + t];
        if (cc < a.KK) {
          const int k = cc / a.ksize, j = cc % a.ksize;
          const int u = wg_src(t + j - a.origin, a.T, a.reflect);
          if (u >= 0) vx = a.x[(size_t)b * a.x_sb + (size_t)k * a.T + u];
        } else if (cc == a.KK && a.db) {
          vx = 1.f;
        }
      }
      sdy[tt][r] = vy;
      sx[tt][r] = vx;
    }
    __syncthreads();
#pragma unroll 8
    for (int tt = 0; tt < kWgChunk; ++tt) {
      const float4 yv = *reinterpret_cast<const float4*>(&sdy[tt][ty * 4]);
      const float4 xv = *reinterpret_cast<const float4*>(&sx[tt][tx * 4]);
      const float ys[4] = {yv.x, yv.y, yv.z, yv.w}, xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ys[i], xs[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n >= a.N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cc = c0 + tx * 4 + j;
      if (cc >= a.ncols) continue;
      if (a.splits > 1) a.ws[((size_t)split * a.N + n) * a.ncols + cc] = acc[i][j];
      else if (cc < a.KK) a.dw[(size_t)n * a.KK + cc] = acc[i][j];
      else a.db[n] = acc[i][j];
    }
  }
}

__global__ void wgrad_reduce_kernel(const WgradArgs a) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, per = (size_t)a.N * a.ncols;
  if (i >= per) return;
  float s = 0.f;
  for (int sp = 0; sp < a.splits; ++sp) s += a.ws[sp * per + i];
  const int n = (int)(i / a.ncols), cc = (int)(i % a.ncols);
  if (cc < a.KK) a.dw[(size_t)n * a.KK + cc] = s;
  else a.db[n] = s;
}

// ------------------------------------------------------------------------------------------------------------------
// BatchNorm1d (batch statistics) + ReLU backward, one CTA per channel over all B*T positions, padded frames included:
//   dz = dy [y > 0] ;  dbeta = sum dz ;  dgamma = sum dz xhat ;  dx = gamma rstd (dz - (dbeta + xhat dgamma) / N)
// xhat from the BatchNorm input x and the forward's mean / var with the forward's rstd = 1 / sqrtf(var + eps).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bn_relu_bwd_kernel(const float* dy, const float* __restrict__ y, const float* __restrict__ x,
                                                          const float* __restrict__ mean, const float* __restrict__ var,
                                                          const float* __restrict__ gamma, float eps, float* dx,
                                                          float* __restrict__ dgamma, float* __restrict__ dbeta, int B, int C,
                                                          int T) {
  const int c = blockIdx.x;
  const float m = mean[c], rstd = 1.0f / sqrtf(var[c] + eps);
  double sb = 0.0, sg = 0.0;
  for (int b = 0; b < B; ++b) {
    const size_t row = ((size_t)b * C + c) * T;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
      const float dz = y[row + t] > 0.f ? dy[row + t] : 0.f;
      const float xh = (x[row + t] - m) * rstd;
      sb += dz;
      sg += (double)dz * xh;
    }
  }
  __shared__ double sh[2][8];
  __shared__ float res[2];
  for (int o = 16; o > 0; o >>= 1) {
    sb += __shfl_xor_sync(0xffffffffu, sb, o);
    sg += __shfl_xor_sync(0xffffffffu, sg, o);
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = sb; sh[1][threadIdx.x >> 5] = sg; }
  __syncthreads();
  if (threadIdx.x == 0) {
    sb = sg = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { sb += sh[0][w]; sg += sh[1][w]; }
    res[0] = (float)sb;
    res[1] = (float)sg;
    dbeta[c] = res[0];
    dgamma[c] = res[1];
  }
  __syncthreads();
  const float db = res[0], dg = res[1], inv_n = 1.0f / ((float)B * (float)T), gr = gamma[c] * rstd;
  for (int b = 0; b < B; ++b) {
    const size_t row = ((size_t)b * C + c) * T;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
      const float dz = y[row + t] > 0.f ? dy[row + t] : 0.f;
      const float xh = (x[row + t] - m) * rstd;
      dx[row + t] = gr * (dz - fmaf(xh, dg, db) * inv_n);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// ReflectionPad1d(pad) backward for a Conv1d(k = 2 pad + 1) whose data gradient dx = conv(dY, W flipped / transposed)
// already holds the centre rows: adds the 2 pad padded rows, dXp[p] = sum_j W[:, ci, j]^T dY[p - j] (p < pad or
// p >= T + pad), into the frames they were reflected from: p -> pad - p and T + pad + e -> T - 2 - e.  One warp per
// (b, ci): lanes split the output channels, a fixed butterfly sums them, lane 0 adds the rows in order.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kFoldMaxPad = 4;

__global__ void __launch_bounds__(256) reflect_fold_kernel(float* dx, const float* __restrict__ dy, const float* __restrict__ w,
                                                           int B, int Cin, int Cout, int T, int pad) {
  const int gw = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (gw >= B * Cin) return;
  const int b = gw / Cin, ci = gw % Cin, ks = 2 * pad + 1;
  float acc[2 * kFoldMaxPad] = {};
  for (int co = lane; co < Cout; co += 32) {
    const float* wr = w + ((size_t)co * Cin + ci) * ks;
    const float* yr = dy + ((size_t)b * Cout + co) * T;
#pragma unroll
    for (int p = 0; p < kFoldMaxPad; ++p) {
      if (p >= pad) break;
      float s = 0.f, e = 0.f;
      for (int j = 0; j <= p; ++j) s = fmaf(wr[j], yr[p - j], s);                    // padded row p
      for (int j = pad + p + 1; j < ks; ++j) e = fmaf(wr[j], yr[T + pad + p - j], e);  // padded row T + pad + p
      acc[p] += s;
      acc[kFoldMaxPad + p] += e;
    }
  }
#pragma unroll
  for (int i = 0; i < 2 * kFoldMaxPad; ++i)
    for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
  if (lane == 0) {
    float* row = dx + ((size_t)b * Cin + ci) * T;
    for (int p = 0; p < pad; ++p) row[pad - p] += acc[p];
    for (int p = 0; p < pad; ++p) row[T - 2 - p] += acc[kFoldMaxPad + p];
  }
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_wgrad_f32(const svsk_wgrad_f32_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "wgrad_f32: null params");
  const svsk_wgrad_f32_params& p = *pp;
  SVSK_REQUIRE(p.dy && p.x && p.dw, SVSK_E_ARG, "wgrad_f32: null tensor");
  SVSK_REQUIRE(p.B > 0 && p.N > 0 && p.K > 0 && p.T > 0 && p.ksize > 0 && p.splits > 0 && p.splits <= 1024, SVSK_E_ARG,
               "wgrad_f32: bad sizes B=%d N=%d K=%d T=%d ksize=%d splits=%d", p.B, p.N, p.K, p.T, p.ksize, p.splits);
  SVSK_REQUIRE(p.dy_batch_stride >= (long long)p.N * p.T && p.x_batch_stride >= (long long)p.K * p.T, SVSK_E_ARG,
               "wgrad_f32: batch strides must cover N T / K T");
  SVSK_REQUIRE(p.pad_mode == SVSK_PAD_ZEROS || p.pad_mode == SVSK_PAD_REFLECT, SVSK_E_ARG, "wgrad_f32: pad_mode must be zeros or reflect");
  SVSK_REQUIRE(p.pad_mode != SVSK_PAD_REFLECT || (p.origin < p.T && p.ksize - 1 - p.origin < p.T && p.origin >= 0 && p.origin < p.ksize),
               SVSK_E_ARG, "wgrad_f32: reflect padding needs 0 <= origin < ksize and a reach below T");
  SVSK_REQUIRE(p.splits == 1 || p.ws, SVSK_E_ARG, "wgrad_f32: splits > 1 needs a workspace");
  if (int rc = require_sm100()) return rc;
  WgradArgs a = {};
  a.dy = p.dy; a.x = p.x; a.dw = p.dw; a.db = p.db; a.ws = p.ws;
  a.dy_sb = p.dy_batch_stride; a.x_sb = p.x_batch_stride;
  a.B = p.B; a.N = p.N; a.K = p.K; a.T = p.T; a.ksize = p.ksize; a.origin = p.origin;
  a.reflect = p.pad_mode == SVSK_PAD_REFLECT; a.splits = p.splits;
  a.KK = p.K * p.ksize;
  a.ncols = a.KK + (p.db ? 1 : 0);
  cudaStream_t st = as_stream(stream);
  dim3 grid((unsigned)ceil_div(a.ncols, kWgTile), (unsigned)ceil_div(a.N, kWgTile), (unsigned)a.splits);
  wgrad_kernel<<<grid, 256, 0, st>>>(a);
  if (int rc = check_launch("wgrad_f32")) return rc;
  if (a.splits > 1) {
    const long long n = (long long)a.N * a.ncols;
    wgrad_reduce_kernel<<<(unsigned)ceil_div_ll(n, 256), 256, 0, st>>>(a);
    return check_launch("wgrad_f32: reduce");
  }
  return 0;
}

extern "C" int svsk_bn_relu_bwd_f32(const float* dy, const float* y, const float* x, const float* mean, const float* var,
                                    const float* gamma, float eps, float* dx, float* dgamma, float* dbeta, int B, int C, int T,
                                    void* stream) {
  SVSK_REQUIRE(dy && y && x && mean && var && gamma && dx && dgamma && dbeta, SVSK_E_ARG, "bn_relu_bwd_f32: null tensor");
  SVSK_REQUIRE(B > 0 && C > 0 && T > 0 && eps > 0.f, SVSK_E_ARG, "bn_relu_bwd_f32: bad B/C/T/eps");
  if (int rc = require_sm100()) return rc;
  bn_relu_bwd_kernel<<<(unsigned)C, 256, 0, as_stream(stream)>>>(dy, y, x, mean, var, gamma, eps, dx, dgamma, dbeta, B, C, T);
  return check_launch("bn_relu_bwd_f32");
}

extern "C" int svsk_reflect_fold_f32(float* dx, const float* dy, const float* w, int B, int Cin, int Cout, int T, int pad,
                                     void* stream) {
  SVSK_REQUIRE(dx && dy && w, SVSK_E_ARG, "reflect_fold_f32: null tensor");
  SVSK_REQUIRE(B > 0 && Cin > 0 && Cout > 0 && pad >= 1 && pad <= kFoldMaxPad, SVSK_E_ARG,
               "reflect_fold_f32: bad sizes (pad must be 1..%d)", kFoldMaxPad);
  SVSK_REQUIRE(T > pad, SVSK_E_ARG, "reflect_fold_f32: reflect padding %d needs T > %d (T=%d)", pad, pad, T);
  if (int rc = require_sm100()) return rc;
  const long long threads = (long long)B * Cin * 32;
  reflect_fold_kernel<<<(unsigned)ceil_div_ll(threads, 256), 256, 0, as_stream(stream)>>>(dx, dy, w, B, Cin, Cout, T, pad);
  return check_launch("reflect_fold_f32");
}
