// Backward of the bidirectional LSTM recurrence (lstm_sm100.cu), one thread-block cluster per (track, direction) like the
// forward.  Given dH_ext = dL/dh from the layer above and the gates i, f, g, o and cells c_t that svsk_lstm_train_f32
// kept, it walks each direction's own scan in reverse:
//   dh = dH_ext[t] + dh_rec ;  dc = dc' + dh o (1 - tanh^2 c_t)
//   da = [dc g i(1-i), dc c_{t-1} f(1-f), dc i (1-g^2), dh tanh(c_t) o(1-o)] ;  dc' <- dc f ;  dh_rec <- W_hh^T da
// and writes da = dL/dpre for every frame (0 for frames >= length).  The weight gradients are separate GEMMs
// (svsk_wgrad_f32); this kernel is only the sequential part.
//
// Same structure as the forward: the unit's slice of W_hh^T lives in registers — a thread owns ONE hidden unit j and one
// column segment of the 4H-long da vector (the four gate rows of L units: w[g][i] = W_hh[g*H + k*L + i][j]), so the
// per-step dot reads 4 x 32 values from shared memory; the CS partial sums of a unit meet in a butterfly of shuffles
// (fixed order, so every lane ends with the same bits); the input-gate lane of each unit does the cell algebra; every
// warp sends the da of its units to all CTAs as 16-byte st.async messages (one gate of four consecutive units each) that
// complete a transaction barrier in the receiver.  The per-frame inputs of step s-1 are loaded while step s computes.
#include "lstm_sm100.cuh"

namespace svsk {

struct LstmBwdArgs {
  const float* dh;        // [B][ndir*H][T]
  const float* gates;     // [B][ndir*4H][T]
  const float* cell;      // [B][ndir*H][T]
  const float* w_hh;      // [ndir][4H][H]
  const int32_t* lengths;
  float* dpre;            // [B][ndir*4H][T]
  int B, T, H, ndir;
  int NC, U, L;
};

template <int CS, int KSEG>
__global__ void __launch_bounds__(kLstmMaxThreads, 1) lstm_backward_kernel(const LstmBwdArgs a) {
  constexpr int kPitch = KSEG + 4;
  __shared__ __align__(16) float dbuf[2][4][CS * kPitch];
  __shared__ __align__(8) uint64_t dbar[2];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (int)ptx::cluster_ctarank();
  const int cluster_id = blockIdx.x / a.NC;
  const int b = cluster_id / a.ndir, d = cluster_id % a.ndir;
  const int U = a.U, H = a.H, L = a.L, T = a.T;
  const int k = tid % CS, u = tid / CS;
  const bool active = u < U;
  const int unit = c * U + (active ? u : 0);
  const int len = a.lengths ? min(max(a.lengths[b], 0), T) : T;

  float w[4][KSEG];  // W_hh^T: gate rows k*L .. k*L+L-1 of each gate, column `unit` (zeros past L)
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float* src = a.w_hh + ((size_t)d * 4 * H + (size_t)g * H + (size_t)k * L) * H + unit;
#pragma unroll
    for (int i = 0; i < KSEG; ++i) w[g][i] = (active && i < L) ? src[(size_t)i * H] : 0.f;
  }
  for (int i = tid; i < 2 * 4 * CS * kPitch; i += blockDim.x) (&dbuf[0][0][0])[i] = 0.f;
  if (tid == 0) {
    ptx::mbar_init(&dbar[0], 1);
    ptx::mbar_init(&dbar[1], 1);
    ptx::fence_mbar_init();
  }
  __syncthreads();
  ptx::cluster_sync_all();

  const bool cell_thread = active && k == 0;
  const size_t col = (size_t)d * H + unit;
  const float* dh_row = a.dh + ((size_t)b * a.ndir * H + col) * T;
  const float* c_row = a.cell + ((size_t)b * a.ndir * H + col) * T;
  const size_t gstride = (size_t)H * T;
  const size_t grow0 = ((size_t)b * a.ndir * 4 * H + (size_t)d * 4 * H + unit) * T;
  const float* g_row = a.gates + grow0;
  float* da_row = a.dpre + grow0;
  auto frame_of = [&](int step) { return d == 0 ? step : len - 1 - step; };

  // messages: one gate of a quad of four consecutive units of this warp, to one CTA (QW * NC * 4 <= 32, checked at launch)
  constexpr int UW = 32 / CS, QW = UW / 4;
  const int mq = lane % QW, mdst = (lane / QW) % a.NC, mg = lane / (QW * a.NC);
  const int mu0 = warp * UW + 4 * mq;
  const bool sender = lane < QW * a.NC * 4 && mu0 < U;
  const int mug = c * U + mu0;
  const uint32_t mpos = (uint32_t)((mg * CS * kPitch) + (mug / L) * kPitch + (mug % L)) * 4u;
  const uint32_t mdata0 = ptx::mapa(ptx::smem_u32(&dbuf[0][0][0]) + mpos, (uint32_t)(sender ? mdst : 0));
  const uint32_t mbar0 = ptx::mapa(ptx::smem_u32(&dbar[0]), (uint32_t)(sender ? mdst : 0));

  // per-frame inputs of the current step (loaded one step ahead on the cell lanes)
  float gi = 0.f, gf = 0.f, gg = 0.f, go = 0.f, ct = 0.f, cp = 0.f, dx = 0.f;
  auto load = [&](int s, float& i_, float& f_, float& g_, float& o_, float& c_, float& p_, float& h_) {
    const int fr = frame_of(s);
    i_ = g_row[fr];
    f_ = g_row[gstride + fr];
    g_ = g_row[2 * gstride + fr];
    o_ = g_row[3 * gstride + fr];
    c_ = c_row[fr];
    p_ = s > 0 ? c_row[frame_of(s - 1)] : 0.f;
    h_ = dh_row[fr];
  };
  if (cell_thread && len > 0) load(len - 1, gi, gf, gg, go, ct, cp, dx);
  float dcc = 0.f;

#pragma unroll 1
  for (int j = 0; j < len; ++j) {
    const int s = len - 1 - j;
    const int cur = j & 1, nxt = cur ^ 1;
    if (tid == 0 && j + 1 < len) ptx::mbar_arrive_expect_tx(&dbar[nxt], (uint32_t)H * 16u);
    float ni = 0.f, nf = 0.f, ng = 0.f, no = 0.f, nc = 0.f, np = 0.f, nx = 0.f;
    if (cell_thread && s > 0) load(s - 1, ni, nf, ng, no, nc, np, nx);
    // everything of the cell algebra that does not depend on dh_rec, before the wait
    const float tc = tanhf(ct);
    const float kc = go * (1.f - tc * tc);
    const float ka[4] = {gg * gi * (1.f - gi), cp * gf * (1.f - gf), gi * (1.f - gg * gg), tc * go * (1.f - go)};
    float dh_rec = 0.f;
    if (j > 0) {
      ptx::mbar_wait(&dbar[cur], ((j - 1) >> 1) & 1);  // da of step s+1 complete in dbuf[cur]
      float acc[4][2];
#pragma unroll
      for (int g = 0; g < 4; ++g) acc[g][0] = acc[g][1] = 0.f;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const float* ds = &dbuf[cur][g][k * kPitch];
#pragma unroll
        for (int i = 0; i < KSEG; i += 4) {
          const float4 v = *reinterpret_cast<const float4*>(ds + i);
          float& q = acc[g][(i >> 2) & 1];
          q = fmaf(w[g][i], v.x, q);
          q = fmaf(w[g][i + 1], v.y, q);
          q = fmaf(w[g][i + 2], v.z, q);
          q = fmaf(w[g][i + 3], v.w, q);
        }
      }
      dh_rec = ((acc[0][0] + acc[0][1]) + (acc[1][0] + acc[1][1])) + ((acc[2][0] + acc[2][1]) + (acc[3][0] + acc[3][1]));
#pragma unroll
      for (int o = 1; o < CS; o <<= 1) dh_rec += __shfl_xor_sync(0xffffffffu, dh_rec, o);
    }
    // cell algebra (meaningful on the input-gate lane of each unit)
    const float dhh = dx + dh_rec;
    const float dc = fmaf(dhh, kc, dcc);
    float da[4] = {dc * ka[0], dc * ka[1], dc * ka[2], dhh * ka[3]};
    dcc = dc * gf;
    if (cell_thread) {
      const int fr = frame_of(s);
#pragma unroll
      for (int g = 0; g < 4; ++g) da_row[g * gstride + fr] = da[g];
    }
    if (j + 1 < len) {
      float m[4];
#pragma unroll
      for (int g = 0; g < 4; ++g)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const float v = __shfl_sync(0xffffffffu, da[g], ((4 * mq + r) * CS) & 31);
          if (g == mg) m[r] = v;
        }
      if (sender) st_async_v4(mdata0 + (uint32_t)(nxt * 4 * CS * kPitch) * 4u, m[0], m[1], m[2], m[3], mbar0 + (uint32_t)nxt * 8u);
    }
    gi = ni; gf = nf; gg = ng; go = no; ct = nc; cp = np; dx = nx;
  }

  // frames past the end of the packed sequence take no part: their gradient is zero
  for (int i = tid; i < (T - len) * U * 4; i += blockDim.x) {
    const int fr = len + i / (U * 4), r = i % (U * 4), g = r / U, uu = c * U + r % U;
    a.dpre[((size_t)b * a.ndir * 4 * H + (size_t)d * 4 * H + (size_t)g * H + uu) * T + fr] = 0.f;
  }
  ptx::cluster_sync_all();
}

template <int CS, int KSEG>
static int launch_lstm_bwd(const LstmBwdArgs& a, int threads, cudaStream_t st) {
  return launch_cluster(lstm_backward_kernel<CS, KSEG>, a, a.B * a.ndir * a.NC, a.NC, threads, st, "lstm_bwd_f32");
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_lstm_bwd_f32(const svsk_lstm_bwd_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "lstm_bwd_f32: null params");
  const svsk_lstm_bwd_params& p = *pp;
  SVSK_REQUIRE(p.dh && p.gates && p.cell && p.w_hh && p.dpre, SVSK_E_ARG, "lstm_bwd_f32: null tensor");
  SVSK_REQUIRE(p.B > 0 && p.T > 0 && (p.ndir == 1 || p.ndir == 2), SVSK_E_ARG, "lstm_bwd_f32: B=%d T=%d ndir=%d", p.B, p.T, p.ndir);
  LstmBwdArgs a = {};
  int CS = 1;
  SVSK_REQUIRE(lstm_layout(p.H, &a.NC, &a.U, &CS, &a.L), SVSK_E_ARG,
               "lstm_bwd_f32: hidden size %d has no cluster layout (need H <= 256 and H %% (4 * 2^k) == 0 with H / 2^k <= 32, k <= 3)", p.H);
  SVSK_REQUIRE(a.NC <= CS, SVSK_E_ARG, "lstm_bwd_f32: H=%d: more CTAs than column segments", p.H);
  const int threads = (a.U * CS + 31) & ~31;
  SVSK_REQUIRE(threads <= kLstmMaxThreads, SVSK_E_ARG, "lstm_bwd_f32: %d threads", threads);
  if (int rc = require_sm100()) return rc;
  a.dh = p.dh; a.gates = p.gates; a.cell = p.cell; a.w_hh = p.w_hh; a.lengths = p.lengths; a.dpre = p.dpre;
  a.B = p.B; a.T = p.T; a.H = p.H; a.ndir = p.ndir;
  cudaStream_t st = as_stream(stream);
  if (CS == 8) return launch_lstm_bwd<8, 32>(a, threads, st);
  if (CS == 4) return launch_lstm_bwd<4, 32>(a, threads, st);
  if (CS == 2) return launch_lstm_bwd<2, 32>(a, threads, st);
  if (a.L <= 8) return launch_lstm_bwd<1, 8>(a, threads, st);
  if (a.L <= 16) return launch_lstm_bwd<1, 16>(a, threads, st);
  return launch_lstm_bwd<1, 32>(a, threads, st);
}
