// Bidirectional LSTM recurrence, one thread-block cluster per (track, direction) — the sequential part of the
// FFConvLSTM encoder in front of the denoiser (nnsvs/model.py:861-868,917-919; SURVEY.md §8(f) row 1).
//
// The input half of the gates (W_ih x_t + b_ih + b_hh, all frames, both directions) is a plain GEMM done beforehand; this
// kernel runs   a_t = pre_t + W_hh h_{t-1};  c_t = s(f) c_{t-1} + s(i) tanh(g);  h_t = s(o) tanh(c_t)   (gate rows in
// torch order i, f, g, o) over the first `length` frames of each track, from the last of them for the reverse direction;
// frames beyond `length` are written as zeros (pack_padded_sequence / pad_packed_sequence semantics).
//
// Latency is everything here (T dependent steps), so nothing is re-read and nothing waits on more than it must:
//  * the 4H x H recurrent matrix of one direction is split over the NC <= 8 CTAs of a cluster (H/NC units each) and lives
//    in REGISTERS: a thread owns the four gate rows of ONE unit over one column segment of <= 32 (4 x 32 fp32 weights),
//    so it reads only 32 values of h per step (8 LDS.128 — the first version read whole rows and was bound by the
//    shared-memory pipe, not by the FMAs);
//  * the CS = H/32 column segments of a unit sit in neighbouring lanes: a transposing shuffle reduction leaves each lane
//    with the complete sum of ONE gate, which it activates; three more shuffles bring f, g, o to the input-gate lane for
//    the cell update;
//  * h_{t-1} sits in shared memory of every CTA (two buffers, by step parity); every warp sends the new h of its own
//    units to all CTAs of the cluster as 16-byte st.async messages that complete a transaction barrier in the
//    receiver — no __syncthreads and no cluster-wide barrier inside the loop;
//  * the gate pre-activations of step t+3 are fetched while step t computes (register ring, loop unrolled by four).
#include "lstm_sm100.cuh"

namespace svsk {

struct LstmArgs {
  const float* pre;
  const float* w_hh;
  const int32_t* lengths;
  float* h_f32;
  __nv_bfloat16* h_bf16;
  float* gates;           // kTrain: [B][ndir*4H][T] activated gates i, f, g, o of every frame < length
  float* cell;            // kTrain: [B][ndir*H][T] cell state c_t
  long long pre_sb, pre_st, pre_sr, hf_sb, hf_st, hf_sr, hb_sb, hb_st;
  int B, T, H, ndir;
  int NC, U, L;           // CTAs per cluster, units per CTA, real elements per column segment (H / CS)
};

// CS column segments per unit (lanes unit*CS .. unit*CS+CS-1), KSEG = padded segment length.  kTrain: the input-gate lane
// of each unit also stores the four activated gates and c_t of every frame (what svsk_lstm_bwd_f32 needs); the arithmetic
// is the same instruction for instruction, so h is bit-identical to the inference kernel's.
template <int CS, int KSEG, bool kTrain>
__global__ void __launch_bounds__(kLstmMaxThreads, 1) lstm_recurrence_kernel(const LstmArgs a) {
  constexpr int kPitch = KSEG + 4;  // neighbouring segments start 4 banks apart: the CS broadcasts of a warp do not collide
  constexpr int NG = CS >= 4 ? 1 : 4 / CS;  // gates a lane owns after the reduction
  __shared__ __align__(16) float hbuf[2][CS * kPitch];
  __shared__ __align__(8) uint64_t hbar[2];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (int)ptx::cluster_ctarank();
  const int cluster_id = blockIdx.x / a.NC;
  const int b = cluster_id / a.ndir, d = cluster_id % a.ndir;
  const int U = a.U, H = a.H, L = a.L;
  const int k = tid % CS, u = tid / CS;              // column segment, unit within the CTA
  const bool active = u < U;                         // the block is padded to whole warps
  const int unit = c * U + (active ? u : 0);
  const int len = a.lengths ? min(max(a.lengths[b], 0), a.T) : a.T;
  // gate(s) whose complete sum lands on this lane: CS >= 4 -> one, bit-reversed (lanes 0..3 = i, g, f, o);
  // CS == 2 -> lane 0: i, f / lane 1: g, o;  CS == 1 -> all four
  const int g0 = CS >= 4 ? (((k & 1) << 1) | ((k >> 1) & 1)) : (CS == 2 ? 2 * k : 0);

  float w[4][KSEG];  // recurrent weights of this unit's four gate rows over this column segment (zeros past L)
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float* src = a.w_hh + ((size_t)d * 4 * H + (size_t)g * H + unit) * H + k * L;
#pragma unroll
    for (int i = 0; i < KSEG; ++i) w[g][i] = (active && i < L) ? src[i] : 0.f;
  }
  for (int i = tid; i < 2 * CS * kPitch; i += blockDim.x) (&hbuf[0][0])[i] = 0.f;
  if (tid == 0) {
    ptx::mbar_init(&hbar[0], 1);
    ptx::mbar_init(&hbar[1], 1);
    ptx::fence_mbar_init();
  }
  __syncthreads();
  ptx::cluster_sync_all();  // every CTA's buffers and barriers exist before anybody sends

  const bool gate_thread = active && k < 4;          // lanes that hold complete gate sums (CS == 8: lanes 4..7 mirror 0..3)
  const bool cell_thread = active && k == 0;
  const float* pre = a.pre + (size_t)b * a.pre_sb + ((size_t)d * 4 * H + unit) * a.pre_sr;
  auto frame_of = [&](int step) { return d == 0 ? step : len - 1 - step; };
  // pre-activations of steps t .. t+3 in a register ring (slot = step & 3): the load for step t+3 is issued at step t and
  // first touched three steps later, so its DRAM latency never meets the critical path
  float q[4][NG];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int n = 0; n < NG; ++n) q[i][n] = 0.f;
  auto fetch = [&](int step, float (&dst)[NG]) {
    const float* row = pre + (size_t)frame_of(step) * a.pre_st;
#pragma unroll
    for (int n = 0; n < NG; ++n) dst[n] = row[(size_t)(g0 + n) * H * a.pre_sr];
  };
  if (gate_thread) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
      if (i < len) fetch(i, q[i]);
  }
  float cell = 0.f;
  const uint32_t hbuf_addr = ptx::smem_u32(&hbuf[0][0]);
  const uint32_t hbar_addr = ptx::smem_u32(&hbar[0]);
  // messages of this warp: its 32/CS units = QW quads of four, each quad to every CTA of the cluster
  constexpr int UW = 32 / CS, QW = UW / 4;
  const int mq = lane % QW, mdst = lane / QW;                       // quad and destination of the message this lane sends
  const int mu0 = warp * UW + 4 * mq;                               // first unit (within the CTA) of that quad
  const bool sender = lane < QW * a.NC && mu0 < U;
  const int mug = c * U + mu0;
  const uint32_t mpos = (uint32_t)((mug / L) * kPitch + (mug % L)) * 4u;
  const uint32_t mdata0 = ptx::mapa(hbuf_addr + mpos, (uint32_t)(sender ? mdst : 0));
  const uint32_t mbar0 = ptx::mapa(hbar_addr, (uint32_t)(sender ? mdst : 0));
  const int ubase = lane & ~(CS - 1);                               // lane of this unit's input gate
  const int col = d * H + unit;

#pragma unroll 1
  for (int t0 = 0; t0 < len; t0 += 4) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int t = t0 + j;
      if (t >= len) break;
      const int cur = j & 1, nxt = cur ^ 1;
      if (tid == 0 && t + 1 < len) ptx::mbar_arrive_expect_tx(&hbar[nxt], (uint32_t)H * 4u);
      if (gate_thread && t + 3 < len) fetch(t + 3, q[(j + 3) & 3]);
      if (t > 0) ptx::mbar_wait(&hbar[cur], ((t - 1) >> 1) & 1);   // h_{t-1} complete in hbuf[cur]

      const float* hs = &hbuf[cur][k * kPitch];
      float acc[4][2];
#pragma unroll
      for (int g = 0; g < 4; ++g) acc[g][0] = acc[g][1] = 0.f;
#pragma unroll
      for (int i = 0; i < KSEG; i += 4) {
        const float4 hv = *reinterpret_cast<const float4*>(hs + i);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float& s = acc[g][(i >> 2) & 1];
          s = fmaf(w[g][i], hv.x, s);
          s = fmaf(w[g][i + 1], hv.y, s);
          s = fmaf(w[g][i + 2], hv.z, s);
          s = fmaf(w[g][i + 3], hv.w, s);
        }
      }
      float s0 = acc[0][0] + acc[0][1], s1 = acc[1][0] + acc[1][1], s2 = acc[2][0] + acc[2][1], s3 = acc[3][0] + acc[3][1];

      // transposing reduction over the unit's CS lanes, then activation of the gate(s) this lane ends up with
      float gi, gf, gg, go;
      if constexpr (CS == 1) {
        const float* p = q[j];
        gi = sigmoid_fast(s0 + p[0]);
        gf = sigmoid_fast(s1 + p[1]);
        gg = tanh_fast(s2 + p[2]);
        go = sigmoid_fast(s3 + p[3]);
      } else {
        const bool hi = k & 1;                                        // odd lanes keep g, o; even lanes keep i, f
        const float r0 = __shfl_xor_sync(0xffffffffu, hi ? s0 : s2, 1);
        const float r1 = __shfl_xor_sync(0xffffffffu, hi ? s1 : s3, 1);
        float a0 = (hi ? s2 : s0) + r0, a1 = (hi ? s3 : s1) + r1;     // (i, f) or (g, o)
        if constexpr (CS == 2) {
          const float* p = q[j];
          const float x0 = hi ? tanh_fast(a0 + p[0]) : sigmoid_fast(a0 + p[0]);
          const float x1 = sigmoid_fast(a1 + p[1]);
          gi = x0;
          gf = x1;
          gg = __shfl_sync(0xffffffffu, x0, ubase + 1);
          go = __shfl_sync(0xffffffffu, x1, ubase + 1);
        } else {
          const bool hi2 = k & 2;                                     // lanes 0..3 end with i, g, f, o
          const float r = __shfl_xor_sync(0xffffffffu, hi2 ? a0 : a1, 2);
          float v = (hi2 ? a1 : a0) + r;
          if constexpr (CS == 8) v += __shfl_xor_sync(0xffffffffu, v, 4);
          v += q[j][0];
          const float x = (g0 == 2) ? tanh_fast(v) : sigmoid_fast(v);
          gi = x;
          gg = __shfl_sync(0xffffffffu, x, ubase + 1);
          gf = __shfl_sync(0xffffffffu, x, ubase + 2);
          go = __shfl_sync(0xffffffffu, x, ubase + 3);
        }
      }
      cell = fmaf(gf, cell, gi * gg);                                 // meaningful on the input-gate lane of each unit
      const float h = go * tanh_fast(cell);
      // four consecutive units' h -> one 16-byte message per (quad, destination CTA)
      const float m0 = __shfl_sync(0xffffffffu, h, (4 * mq + 0) * CS);
      const float m1 = __shfl_sync(0xffffffffu, h, (4 * mq + 1) * CS);
      const float m2 = __shfl_sync(0xffffffffu, h, (4 * mq + 2) * CS);
      const float m3 = __shfl_sync(0xffffffffu, h, (4 * mq + 3) * CS);
      if (sender && t + 1 < len)
        st_async_v4(mdata0 + (uint32_t)(nxt * CS * kPitch) * 4u, m0, m1, m2, m3, mbar0 + (uint32_t)nxt * 8u);
      if (cell_thread) {
        const int frame = frame_of(t);
        if (a.h_f32) a.h_f32[(size_t)b * a.hf_sb + (size_t)frame * a.hf_st + (size_t)col * a.hf_sr] = h;
        if (a.h_bf16) a.h_bf16[(size_t)b * a.hb_sb + (size_t)frame * a.hb_st + col] = __float2bfloat16_rn(h);
        if constexpr (kTrain) {
          float* gp = a.gates + ((size_t)b * a.ndir * 4 + (size_t)d * 4) * H * a.T + (size_t)unit * a.T + frame;
          gp[0] = gi;
          gp[(size_t)H * a.T] = gf;
          gp[(size_t)2 * H * a.T] = gg;
          gp[(size_t)3 * H * a.T] = go;
          a.cell[((size_t)b * a.ndir * H + col) * a.T + frame] = cell;
        }
      }
    }
  }

  // frames past the end of the packed sequence read as zeros
  for (int i = tid; i < (a.T - len) * U; i += blockDim.x) {
    const int frame = len + i / U, zc = d * H + c * U + i % U;
    if (a.h_f32) a.h_f32[(size_t)b * a.hf_sb + (size_t)frame * a.hf_st + (size_t)zc * a.hf_sr] = 0.f;
    if (a.h_bf16) a.h_bf16[(size_t)b * a.hb_sb + (size_t)frame * a.hb_st + zc] = __float2bfloat16_rn(0.f);
    if constexpr (kTrain) {
      for (int g = 0; g < 4; ++g) a.gates[((size_t)b * a.ndir * 4 * H + (size_t)d * 4 * H + g * H + c * U + i % U) * a.T + frame] = 0.f;
      a.cell[((size_t)b * a.ndir * H + zc) * a.T + frame] = 0.f;
    }
  }
  ptx::cluster_sync_all();  // nobody leaves while a peer may still address its shared memory
}

template <int CS, int KSEG, bool kTrain>
static int launch_lstm(const LstmArgs& a, int threads, cudaStream_t st) {
  return launch_cluster(lstm_recurrence_kernel<CS, KSEG, kTrain>, a, a.B * a.ndir * a.NC, a.NC, threads, st, "lstm_f32");
}

template <bool kTrain>
static int launch_lstm_any(const LstmArgs& a, int CS, int threads, cudaStream_t st) {
  if (CS == 8) return launch_lstm<8, 32, kTrain>(a, threads, st);
  if (CS == 4) return launch_lstm<4, 32, kTrain>(a, threads, st);
  if (CS == 2) return launch_lstm<2, 32, kTrain>(a, threads, st);
  if (a.L <= 8) return launch_lstm<1, 8, kTrain>(a, threads, st);
  if (a.L <= 16) return launch_lstm<1, 16, kTrain>(a, threads, st);
  return launch_lstm<1, 32, kTrain>(a, threads, st);
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_lstm_supported(int H) {
  int NC, U, CS, L;
  return lstm_layout(H, &NC, &U, &CS, &L) ? 1 : 0;
}

// Argument checks shared by both entries, then the kernel arguments; 0 or an SVSK_E_* code (nothing launched).
static int lstm_args(const svsk_lstm_params* pp, const char* what, LstmArgs* a, int* CS, int* threads) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "%s: null params", what);
  const svsk_lstm_params& p = *pp;
  SVSK_REQUIRE(p.pre && p.w_hh && (p.h_f32 || p.h_bf16), SVSK_E_ARG, "%s: null tensor", what);
  SVSK_REQUIRE(p.B > 0 && p.T > 0 && (p.ndir == 1 || p.ndir == 2), SVSK_E_ARG, "%s: B=%d T=%d ndir=%d", what, p.B, p.T, p.ndir);
  *a = LstmArgs{};
  SVSK_REQUIRE(lstm_layout(p.H, &a->NC, &a->U, CS, &a->L), SVSK_E_ARG,
               "%s: hidden size %d has no cluster layout (need H <= 256 and H %% (4 * 2^k) == 0 with H / 2^k <= 32, k <= 3)", what, p.H);
  a->pre = p.pre; a->w_hh = p.w_hh; a->lengths = p.lengths; a->h_f32 = p.h_f32; a->h_bf16 = reinterpret_cast<__nv_bfloat16*>(p.h_bf16);
  a->pre_sb = p.pre_stride_b; a->pre_st = p.pre_stride_t; a->pre_sr = p.pre_stride_r;
  a->hf_sb = p.hf_stride_b; a->hf_st = p.hf_stride_t; a->hf_sr = p.hf_stride_c;
  a->hb_sb = p.hb_stride_b; a->hb_st = p.hb_stride_t;
  a->B = p.B; a->T = p.T; a->H = p.H; a->ndir = p.ndir;
  *threads = (a->U * *CS + 31) & ~31;
  SVSK_REQUIRE(*threads <= kLstmMaxThreads, SVSK_E_ARG, "%s: %d threads", what, *threads);
  return 0;
}

extern "C" int svsk_lstm_f32(const svsk_lstm_params* pp, void* stream) {
  LstmArgs a;
  int CS = 1, threads = 0;
  if (int rc = lstm_args(pp, "lstm_f32", &a, &CS, &threads)) return rc;
  if (int rc = require_sm100()) return rc;
  return launch_lstm_any<false>(a, CS, threads, as_stream(stream));
}

extern "C" int svsk_lstm_train_f32(const svsk_lstm_params* pp, float* gates, float* cell, void* stream) {
  LstmArgs a;
  int CS = 1, threads = 0;
  if (int rc = lstm_args(pp, "lstm_train_f32", &a, &CS, &threads)) return rc;
  SVSK_REQUIRE(gates && cell, SVSK_E_ARG, "lstm_train_f32: null gates / cell");
  if (int rc = require_sm100()) return rc;
  a.gates = gates;
  a.cell = cell;
  return launch_lstm_any<true>(a, CS, threads, as_stream(stream));
}
