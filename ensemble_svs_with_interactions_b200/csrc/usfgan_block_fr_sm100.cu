// Fused uSFGAN / QPPWG residual block with the aux projection taken at FRAME rate (usfgan_fr.cuh) — the variant
// svsk_usfgan_block_bf16 runs when the caller passes aux_u / aux_q.  Same arithmetic per block as usfgan_block_sm100.cu
// (nnsvs/usfgan/layers/residual_block.py:123-157, 198-234; nnsvs/usfgan/utils/index.py:12-54):
//
//   D1[t][128] = [x(tap0) ; x(t) ; x(tap2)] . W1p^T  +  U[t][16] . Q[fbase .. fbase+15][128]      K = 192 + 16
//   z = tanh(D1[:, :64] + b) * sigmoid(D1[:, 64:] + b)
//   D2[t][64]  = z . Wout^T ;   x'(t) = (D2 + bout + x(t)) * sqrt(1/2)
//
// What differs from the sample-rate kernel, and why (profiles/r01n_ablate_usfgan_noprof.log: the MMA-issuing thread, the
// epilogue chain and the data skeleton were all within 3.1-4.9 k cycles per tile):
//   * no sample-rate aux stream: 256 instead of 416 DRAM bytes per sample, 13 instead of 17 MMAs per tile, the block's
//     resident weights shrink from 88 to 56 KB;
//   * the freed shared memory holds TWO whole-tile operand stages (4 x 16 KB: tap0, centre, tap2, aux) with ONE full and
//     ONE empty barrier per tile, so the MMA thread does 2 barrier waits and 2 commits per tile instead of 5 + 6 — a wait
//     whose result is needed at once stalls that thread ~160 cycles even when the phase completed long ago;
//   * the residual add runs on the tensor cores: the GEMM1 thread also issues D2 = X_centre . I (four N = 64 MMAs against
//     a resident 64 x 64 identity tile, exact in the fp32 accumulator) and GEMM2 accumulates onto it — the epilogue's
//     per-row residual loads are gone.  Thread = row epilogue accesses to GLOBAL memory touch 32 different 128-byte
//     lines per warp instruction; ncu showed the LSU data pipe at 78 % of its peak with them (residual loads + direct
//     stores: 3.4 -> 2.7 k cycles per tile when either was ablated), while TMA traffic does not pass through that pipe;
//   * two epilogue groups of 8 warps, group p owning the tiles n with n & 1 == p together with D1[p], G[p] and two D2
//     accumulators: while one group waits for its GEMM2 or its TMA store the other one gates.
//
//   warp 0      TMA producer: centre tap, and both side taps of interior fixed-block tiles
//   warp 1      MMA issuer (tcgen05.mma cta_group::1, M=128): per tile GEMM2 (N=64) of the tile two back, then GEMM1
//               (N=128) and the residual's identity MMAs of this one — one thread, so their order in the tensor pipe is
//               fixed; + TMEM owner
//   warp 6      idle (was the GEMM2 issuer)
//   warps 2-5   gather producers (thread = row): the aux operands U (rows = samples) and Q (rows = gate channels) of
//               every tile by 16-byte cp.async into the swizzled tiles (completion through
//               cp.async.mbarrier.arrive.noinc on the tile's full barrier), and the side taps of adaptive blocks /
//               reflected boundary tiles: one 1 KB TMA box per 8-row group whose sources are consecutive rows, cp.async
//               rows for the rest
//   warps 7-22  epilogue: two groups of 8 warps (thread = sample, two warps per TMEM lane quarter alternating 16-column
//               chunks); gate -> G[p] (bf16, swizzled smem) -> GEMM2 -> output rows into the same buffer -> one TMA store
//               per lane quarter
// TMEM: two D1 (2 x 128 columns, one per epilogue group) and four D2 (4 x 64, two per group: the residual's identity
// MMAs of the group's next tile are issued while the current one is still being read) = 512 columns.
#include <cuda_bf16.h>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"
#include "tma_util.cuh"
#include "usfgan_fr.cuh"

namespace svsk {

constexpr int kFTile = 128 * 128;     // 128 rows x 64 bf16
constexpr int kFStage = 4 * kFTile;   // tap0, centre, tap2, aux
constexpr int kFThreads = 736;  // producer, GEMM1, 4 gather, GEMM2, 2 x 8 epilogue warps

struct UsfganFrArgs {
  const __nv_bfloat16* xb_in;
  __nv_bfloat16* xb_out;
  const float* bias1;
  const float* bout;
  const int32_t* idx_past;
  const int32_t* idx_future;
  const __nv_bfloat16* aux_u;  // [ceil128(T)][16]
  const __nv_bfloat16* aux_q;  // this block's 128 rows of track 0; row n of track b at aux_q + b * q_batch_stride + n * q_ld
  long long q_batch_stride;
  int q_ld, q_fpad, hop, reach;
  int B, T, dilation, adaptive, tiles_per_row, total_tiles;
  float out_scale;
  int out_relu;
};

struct __align__(8) UsfganFrBarriers {
  uint64_t full[2];   // 1 TMA arrival (+ tx bytes) + 128 gather arrivals per tile
  uint64_t empty[2];  // GEMM1 of the tile has read the stage
  uint64_t d1_full[2], g_full[2], d2_full[4];
  uint64_t w_full;
  uint32_t tmem_base;
};

__device__ __forceinline__ void fr_cp_async_16(void* dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ptx::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void fr_cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(ptx::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fr_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(ptx::smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool fr_tile_needs_gather(int t0, int T, int d, int adaptive) {
  if (adaptive) return true;
  const int last = min(t0 + 127, T - 1);
  return (t0 - d < 0) || (last + d >= T);  // a reflected tap: rows are not a shifted copy any more
}

// kWindow (fixed blocks with dilation <= 8, i.e. 34 of the recipe's 35): the three taps of an interior tile are ONE
// (128 + 16)-row window load and three row offsets of the A descriptor (as in the DiffNet kernels) instead of three
// 16 KB loads of the same rows shifted by -d / 0 / +d: 18 instead of 48 KB per tile from L2 into shared memory.  Tiles at
// a track's ends (reflected taps) keep the gathered layout.
constexpr int kFWinRows = 128 + 16;
constexpr int kFWinBytes = kFWinRows * 128;  // 18 KB: the tap0 tile of the stage + the first 2 KB of its centre tile

template <bool kWindow>
__global__ void __launch_bounds__(kFThreads, 1)
usfgan_block_fr_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w1,
                       const __grid_constant__ CUtensorMap tm_wout, const __grid_constant__ CUtensorMap tm_xout,
                       const __grid_constant__ CUtensorMap tm_x8, const __grid_constant__ CUtensorMap tm_xw,
                       const UsfganFrArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w1_s = smem;                       // 3 tiles of [128 rows][64]
  uint8_t* wout_s = w1_s + 3 * kFTile;        // [64 rows][64] = 8 KB
  uint8_t* stages = wout_s + 8192;            // 2 x {tap0, centre, tap2, aux}
  uint8_t* gbuf = stages + 2 * kFStage;       // 2 x 16 KB: G, then the output rows, of the tile of epilogue group p
  uint8_t* ident_s = gbuf + 2 * kFTile;       // [64 rows][64] identity, 8 KB
  float* bias_s = reinterpret_cast<float*>(ident_s + 8192);  // [128] gate biases, [64] output biases
  UsfganFrBarriers* bars = reinterpret_cast<UsfganFrBarriers*>(bias_s + 192);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = a.T;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_x);
    ptx::prefetch_tmap(&tm_w1);
    ptx::prefetch_tmap(&tm_wout);
    ptx::prefetch_tmap(&tm_xout);
    ptx::prefetch_tmap(&tm_x8);
    if (kWindow) ptx::prefetch_tmap(&tm_xw);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->full[i], 129);
      ptx::mbar_init(&bars->empty[i], 1);
      ptx::mbar_init(&bars->d1_full[i], 1);
      ptx::mbar_init(&bars->g_full[i], 256);
    }
    for (int i = 0; i < 4; ++i) ptx::mbar_init(&bars->d2_full[i], 1);
    ptx::mbar_init(&bars->w_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 192; i += kFThreads) bias_s[i] = i < 128 ? a.bias1[i] : a.bout[i - 128];
  // identity tile in the swizzled K-major layout: row n holds 1.0 at K = n (chunk n >> 3 of the row, element n & 7)
  for (int i = threadIdx.x; i < 8192 / 16; i += kFThreads) {
    const uint32_t row = (uint32_t)i >> 3, pos = (uint32_t)i & 7u;           // physical 16-byte chunk `pos` of row `row`
    const uint32_t chunk = pos ^ (row & 7u);                                  // logical chunk stored there
    const uint32_t one = (chunk == (row >> 3)) ? (0x3f80u << (16 * (row & 1u))) : 0u;
    const uint32_t w = (row & 7u) >> 1;
    ptx::st_shared_v4(ident_s + i * 16, w == 0 ? one : 0u, w == 1 ? one : 0u, w == 2 ? one : 0u, w == 3 ? one : 0u);
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      ptx::mbar_arrive_expect_tx(&bars->w_full, 3 * kFTile + 8192);
      for (int kb = 0; kb < 3; ++kb) ptx::tma_load_2d(w1_s + kb * kFTile, &tm_w1, &bars->w_full, kb * 64, 0);
      ptx::tma_load_2d(wout_s, &tm_wout, &bars->w_full, 0, 0);
      int n = 0;
      for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++n) {
        const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
        const bool gather = fr_tile_needs_gather(t0, T, a.dilation, a.adaptive);
        const int st = n & 1;
        ptx::mbar_wait(&bars->empty[st], ((n >> 1) & 1) ^ 1);
        uint8_t* slot = stages + st * kFStage;
        if (kWindow && !gather) {
          ptx::mbar_arrive_expect_tx(&bars->full[st], kFWinBytes);
          ptx::tma_load_3d(slot, &tm_xw, &bars->full[st], 0, t0 - 8, b);
        } else {
          ptx::mbar_arrive_expect_tx(&bars->full[st], gather ? kFTile : 3 * kFTile);
          ptx::tma_load_3d(slot + kFTile, &tm_x, &bars->full[st], 0, t0, b);
          if (!gather) {
            ptx::tma_load_3d(slot, &tm_x, &bars->full[st], 0, t0 - a.dilation, b);
            ptx::tma_load_3d(slot + 2 * kFTile, &tm_x, &bars->full[st], 0, t0 + a.dilation, b);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ GEMM1 issuer
    if (lane == 0) {
      const uint32_t idesc1 = ptx::umma_idesc_bf16_f32(128, 128);
      ptx::mbar_wait(&bars->w_full, 0);
      ptx::tc_fence_after();
      const uint32_t idesc2 = ptx::umma_idesc_bf16_f32(128, 64);
      const uint32_t st_lo = ptx::umma_desc_lo(ptx::smem_u32(stages)), w1_lo = ptx::umma_desc_lo(ptx::smem_u32(w1_s));
      const uint32_t id_lo = ptx::umma_desc_lo(ptx::smem_u32(ident_s));
      constexpr uint32_t kT16 = kFTile >> 4;
      // The barriers of tile n+1 are probed while the MMAs of tile n are issued (ptx::umma_bf16_x4_probe): no phase can
      // complete twice in between, because the stage's next producer waits for this thread's commit.
      bool full_ready = false, g_ready = false;
      const uint32_t wo_lo = ptx::umma_desc_lo(ptx::smem_u32(wout_s)), g_lo = ptx::umma_desc_lo(ptx::smem_u32(gbuf));
      // GEMM2 of this CTA's m-th tile: D2 += G . Wout^T onto the residual the identity MMAs left there
      auto issue_gemm2 = [&](int m) {
        const int pm = m & 1, j = pm * 2 + ((m >> 1) & 1);  // D2 accumulator: two per epilogue group, alternating
        const uint32_t gl = g_lo + pm * (kFTile >> 4);
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) ptx::umma_bf16_lo(tmem + 256 + j * 64, gl + 2 * k4, wo_lo + 2 * k4, idesc2, 1);
        ptx::umma_commit(&bars->d2_full[j]);
      };
      int n = 0;
      int tt = (int)blockIdx.x % a.tiles_per_row;  // tile index within its track (kWindow: which operand layout the stage holds)
      for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++n) {
        const int p = n & 1;
        // D1[p] is free once the epilogue has gated tile n - 2 out of it — the same event makes G[p] of tile n - 2 ready
        // for GEMM2, which is therefore issued HERE, ahead of this tile's GEMM1.  With a thread of its own for GEMM2 both
        // woke on the same barrier, and whenever GEMM1's 17 MMAs won the race the epilogue group waited for four N = 64
        // MMAs queued behind them: 381 -> 365 us per fixed block.  (Measured and not kept: this thread as an event loop
        // polling both groups' g_full while it waits, so that neither group's GEMM2 waits for the other's gating — 377 us;
        // the polls cost more than the head-of-line blocking they remove.)
        if (n >= 2) {
          if (!g_ready) ptx::mbar_wait(&bars->g_full[p], ((n - 2) >> 1) & 1);
          ptx::tc_fence_after();
          issue_gemm2(n - 2);
        }
        if (!full_ready) ptx::mbar_wait(&bars->full[p], (n >> 1) & 1);
        ptx::fence_proxy_async_smem();  // the gather warps' cp.async writes -> tensor-core (async proxy) reads
        ptx::tc_fence_after();
        const uint32_t s_lo = st_lo + p * (kFStage >> 4);
        // operand rows: three tiles of the stage, or (window) three row offsets of one tile
        uint32_t a_t0 = s_lo, a_c = s_lo + kT16, a_t2 = s_lo + 2 * kT16;
        if (kWindow) {
          if (!fr_tile_needs_gather(tt * 128, T, a.dilation, 0)) {
            a_t0 = s_lo + (uint32_t)(8 - a.dilation) * 8u;
            a_c = s_lo + 64u;
            a_t2 = s_lo + (uint32_t)(8 + a.dilation) * 8u;
          }
          tt += (int)gridDim.x;
          while (tt >= a.tiles_per_row) tt -= a.tiles_per_row;
        }
        const uint32_t d1 = tmem + p * 128;
        uint64_t* nfull = &bars->full[p ^ 1];
        const uint32_t nfull_par = ((n + 1) >> 1) & 1;
        uint64_t* ng = &bars->g_full[p ^ 1];
        const uint32_t ng_par = ((n - 1) >> 1) & 1;  // meaningful for n >= 1
        (void)ptx::umma_bf16_x4_probe(d1, a_t0, w1_lo, idesc1, 0, 4, nfull, nfull_par);
        const bool r1 = ptx::umma_bf16_x4_probe(d1, a_c, w1_lo + kT16, idesc1, 1, 4, ng, ng_par);
        const bool r2 = ptx::umma_bf16_x4_probe(d1, a_t2, w1_lo + 2 * kT16, idesc1, 1, 4, nfull, nfull_par);
        // aux: A = U (K columns 0..15 of the aux tile's rows), B = Q (K columns 16..31 of the same rows)
        ptx::umma_bf16_lo(d1, s_lo + 3 * kT16, s_lo + 3 * kT16 + 2, idesc1, 1);
        // residual: D2 = X_centre . I, GEMM2 accumulates onto it.  This D2 accumulator was last read by the residual
        // epilogue of tile n - 4, which its group finished before it gated tile n - 2 (waited for above).
        const uint32_t d2 = tmem + 256 + (p * 2 + ((n >> 1) & 1)) * 64;
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) ptx::umma_bf16_lo(d2, a_c + 2 * k4, id_lo + 2 * k4, idesc2, k4 != 0);
        ptx::umma_commit(&bars->empty[p]);
        ptx::umma_commit(&bars->d1_full[p]);
        full_ready = r2;
        g_ready = r1 && n >= 1;
      }
      for (int m = n >= 2 ? n - 2 : 0; m < n; ++m) {  // GEMM2 of the last two tiles
        ptx::mbar_wait(&bars->g_full[m & 1], (m >> 1) & 1);
        ptx::tc_fence_after();
        issue_gemm2(m);
      }
    }
  } else if (warp < 6) {
    // ------------------------------------------------------------------ gather producers (thread = row of the tiles)
    const int r = threadIdx.x - 64;
    // This row's two tap indices are requested one tile ahead, so that their (L2) latency is off the stage's chain.
    auto load_idx = [&](int tile, int& ip_, int& ifu_) {
      ip_ = ifu_ = -1;
      if (a.adaptive && tile < a.total_tiles) {
        const int b_ = tile / a.tiles_per_row, t_ = (tile - b_ * a.tiles_per_row) * 128 + r;
        if (t_ < T) {
          ip_ = __ldg(a.idx_past + (size_t)b_ * T + t_);
          ifu_ = __ldg(a.idx_future + (size_t)b_ * T + t_);
        }
      }
    };
    int ip_next, ifu_next;
    load_idx(blockIdx.x, ip_next, ifu_next);
    int n = 0;
    for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++n) {
      const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
      const bool gather = fr_tile_needs_gather(t0, T, a.dilation, a.adaptive);
      const int t = t0 + r;
      const int ip = ip_next, ifu = ifu_next;
      load_idx(tile + gridDim.x, ip_next, ifu_next);
      const int st = n & 1;
      ptx::mbar_wait_warp(&bars->empty[st], ((n >> 1) & 1) ^ 1);
      uint8_t* slot = stages + st * kFStage;
      {
        uint8_t* aux_s = slot + 3 * kFTile;
        const uint8_t* us = reinterpret_cast<const uint8_t*>(a.aux_u + (size_t)t * 16);
        const int fb = usfgan_frame_base(t0, a.reach, a.hop);
        const uint8_t* qs = reinterpret_cast<const uint8_t*>(a.aux_q + (size_t)b * a.q_batch_stride + (size_t)r * a.q_ld +
                                                             (a.q_fpad + fb));
        fr_cp_async_16(aux_s + ptx::sw128_offset((uint32_t)r, 0u), us, 16u);
        fr_cp_async_16(aux_s + ptx::sw128_offset((uint32_t)r, 1u), us + 16, 16u);
        fr_cp_async_16(aux_s + ptx::sw128_offset((uint32_t)r, 2u), qs, 16u);
        fr_cp_async_16(aux_s + ptx::sw128_offset((uint32_t)r, 3u), qs + 16, 16u);
      }
      if (gather) {
#pragma unroll
        for (int side = 0; side < 2; ++side) {
          int src = -1;
          if (t < T) {
            if (a.adaptive) {
              src = side == 0 ? ip : ifu;
            } else {
              src = t + (side == 0 ? -a.dilation : a.dilation);
              if (src < 0) src = -src;
              if (src >= T) src = 2 * (T - 1) - src;
            }
          }
          const bool ok = src >= 0 && src < T;
          uint8_t* dst = slot + side * 2 * kFTile;
          // F0 is constant over a hop, so the pitch-dependent taps of most 8-row groups are 8 CONSECUTIVE source rows:
          // such a group (one 1 KB swizzle atom of the tile) travels as one TMA box issued by its first lane — its bytes
          // are added to the phase's expected count before this thread's own arrival, so the phase cannot close early —
          // and only the groups that straddle a frame boundary, a reflection or the end of the track are gathered row by
          // row (16 cp.async per thread and tile were 1.7 k of the adaptive blocks' 4.1 k cycles per tile).
          const int base = __shfl_sync(0xffffffffu, src, lane & ~7);
          const unsigned lin = __ballot_sync(0xffffffffu, ok && src == base + (lane & 7));
          if (((lin >> (lane & ~7)) & 0xffu) == 0xffu) {
            if ((lane & 7) == 0) {
              fr_mbar_expect_tx(&bars->full[st], 1024u);
              ptx::tma_load_3d(dst + (r >> 3) * 1024, &tm_x8, &bars->full[st], 0, base, b);
            }
          } else {
            const uint8_t* g = reinterpret_cast<const uint8_t*>(a.xb_in + ((size_t)b * T + (ok ? src : 0)) * 64);
#pragma unroll
            for (int c = 0; c < 8; ++c)
              fr_cp_async_16(dst + ptx::sw128_offset((uint32_t)r, (uint32_t)c), g + c * 16, ok ? 16u : 0u);
          }
        }
      }
      fr_cp_async_arrive_noinc(&bars->full[st]);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else if (warp == 6) {
    // (idle: GEMM2 is issued by the GEMM1 thread, see there)
  } else {
    // ------------------------------------------------------------------ epilogue: two groups of 8 warps; group p owns the
    // tiles n with n & 1 == p and with them D1[p], G[p] and the D2 pair 2p, 2p+1 — the groups share no buffer.
    // (Measured and not kept: ONE group of 16 warps, one 16-column chunk per thread, software-pipelined gate(n) ;
    // residual(n - 1) — no idle waits left (D1 0.3 k + D2 0.25 k cycles per tile), but the phases do not get twice as fast
    // with twice the warps (gate 2.55 k -> 1.79 k, residual 1.70 k -> 1.00 k: barrier, TMEM-load and fence latencies and the
    // 1.0 k-cycle MUFU floor of a tile's gate do not divide), and serialised they cost more than two half-width groups that
    // overlap each other: 400 vs 365 us per fixed block; adaptive blocks, bound by the gather, 421 vs 440 us.)
    // Thread = one sample, half the columns (two warps per TMEM lane quarter alternating 16-column chunks).
    const int e = warp - 7;
    const int p = e >> 3;
    const int sub = (e >> 2) & 1;  // 0: 16-column chunks 0 and 2, 1: chunks 1 and 3
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    const bool qlead = (sub == 0 && lane == 0);  // issues the TMA stores of this lane quarter's 32 rows
    const uint32_t qbar = 1 + p * 4 + q;         // named barrier of the quarter's two warps
    const int my_tiles = a.total_tiles > (int)blockIdx.x ? (a.total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int own = my_tiles > p ? (my_tiles - 1 - p) / 2 + 1 : 0;  // tiles of this group
    uint8_t* gb = gbuf + p * kFTile;
    for (int k = 0; k < own; ++k) {
      const int n = p + 2 * k;
      const int tile = blockIdx.x + n * gridDim.x;
      const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
      ptx::mbar_wait_warp(&bars->d1_full[p], k & 1);
      ptx::tc_fence_after();
      if (k >= 1) {  // this quarter's rows of G[p] held the previous output tile: its TMA store must have read them
        if (qlead) ptx::bulk_wait_read_all();
        ptx::named_bar_sync(qbar, 64);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c0 = 16 * (2 * i + sub);
        uint32_t ra[16], rb[16];
        ptx::tmem_ld16(tmem + tlane + p * 128 + c0, ra);
        ptx::tmem_ld16(tmem + tlane + p * 128 + 64 + c0, rb);
        ptx::tmem_ld_wait();
        uint32_t o[8];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const uint4 ba = ptx::ld_shared_v4(bias_s + c0 + 4 * v), bb = ptx::ld_shared_v4(bias_s + 64 + c0 + 4 * v);
          const float fa[4] = {__uint_as_float(ba.x), __uint_as_float(ba.y), __uint_as_float(ba.z), __uint_as_float(ba.w)};
          const float fb[4] = {__uint_as_float(bb.x), __uint_as_float(bb.y), __uint_as_float(bb.z), __uint_as_float(bb.w)};
          float z[4];
          // column pairs: FADD2 / FMUL2 / FFMA2 — same arithmetic per lane as tanh_approx(ya) * sigmoid_approx(yb)
#pragma unroll
          for (int j = 0; j < 4; j += 2) {
            const uint64_t ya = ptx::f2_add(ptx::f2_pack(__uint_as_float(ra[4 * v + j]), __uint_as_float(ra[4 * v + j + 1])), ptx::f2_pack(fa[j], fa[j + 1]));
            const uint64_t yb = ptx::f2_add(ptx::f2_pack(__uint_as_float(rb[4 * v + j]), __uint_as_float(rb[4 * v + j + 1])), ptx::f2_pack(fb[j], fb[j + 1]));
            ptx::f2_unpack(ptx::f2_gate(yb, ya), z[j], z[j + 1]);
          }
          o[2 * v] = ptx::pack_bf16(z[0], z[1]);
          o[2 * v + 1] = ptx::pack_bf16(z[2], z[3]);
        }
        ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3)), o[0], o[1], o[2], o[3]);
        ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3) + 1), o[4], o[5], o[6], o[7]);
      }
      ptx::tc_fence_before();
      ptx::fence_proxy_async_smem();
      ptx::mbar_arrive(&bars->g_full[p]);
      const int j2 = p * 2 + (k & 1);
      ptx::mbar_wait_warp(&bars->d2_full[j2], (k >> 1) & 1);  // D2 = x + G . Wout^T is there, GEMM2 has read G[p]
      ptx::tc_fence_after();
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c0 = 16 * (2 * i + sub);
        uint32_t rd[16];
        ptx::tmem_ld16(tmem + tlane + 256 + j2 * 64 + c0, rd);
        ptx::tmem_ld_wait();
        uint32_t o[8];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const uint4 bo = ptx::ld_shared_v4(bias_s + 128 + c0 + 4 * v);
          const float fo[4] = {__uint_as_float(bo.x), __uint_as_float(bo.y), __uint_as_float(bo.z), __uint_as_float(bo.w)};
          float y[4];
          const uint64_t sc2 = ptx::f2_pack(a.out_scale, a.out_scale);
#pragma unroll
          for (int j = 0; j < 4; j += 2) {
            const uint64_t y2 = ptx::f2_mul(ptx::f2_add(ptx::f2_pack(__uint_as_float(rd[4 * v + j]), __uint_as_float(rd[4 * v + j + 1])), ptx::f2_pack(fo[j], fo[j + 1])), sc2);
            ptx::f2_unpack(y2, y[j], y[j + 1]);
          }
          if (a.out_relu) {
#pragma unroll
            for (int j = 0; j < 4; ++j) y[j] = fmaxf(y[j], 0.f);
          }
          o[2 * v] = ptx::pack_bf16(y[0], y[1]);
          o[2 * v + 1] = ptx::pack_bf16(y[2], y[3]);
        }
        ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3)), o[0], o[1], o[2], o[3]);
        ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3) + 1), o[4], o[5], o[6], o[7]);
      }
      ptx::tc_fence_before();
      ptx::fence_proxy_async_smem();
      // each TMEM lane quarter (two warps, 32 rows of the tile) stores its own rows
      ptx::named_bar_sync(qbar, 64);
      if (qlead) {
        ptx::tma_store_3d(&tm_xout, gb + q * 4096, 0, t0 + q * 32, b);
        ptx::bulk_commit_group();
      }
    }
    if (qlead) ptx::bulk_wait_read_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem, 512);
}

// Called by svsk_usfgan_block_bf16 (usfgan_block_sm100.cu) after the common argument checks.
int usfgan_block_fr_launch(const svsk_usfgan_block_params& p, void* stream) {
  SVSK_REQUIRE(p.aux_u && p.aux_q, SVSK_E_ARG, "usfgan_block_bf16: frame-rate aux needs both aux_u and aux_q");
  SVSK_REQUIRE(p.hop >= 1 && p.reach >= 0 && (127 + 2 * (long long)p.reach) / p.hop <= 7, SVSK_E_ARG,
               "usfgan_block_bf16: a 128-sample tile must reach at most 8 frames (hop=%d reach=%d)", p.hop, p.reach);
  SVSK_REQUIRE(p.q_ld > 0 && p.q_ld % 8 == 0 && p.q_fpad >= 0 && p.q_fpad % 8 == 0 && p.q_batch_stride % 8 == 0 &&
                   (reinterpret_cast<uintptr_t>(p.aux_q) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.aux_u) & 15) == 0,
               SVSK_E_ALIGN, "usfgan_block_bf16: aux_q rows / aux_u must be 16-byte aligned (q_ld=%d q_fpad=%d)", p.q_ld, p.q_fpad);
  const int tiles_per_row = (p.T + 127) / 128;
  const int fb_first = usfgan_frame_base(0, p.reach, p.hop), fb_last = usfgan_frame_base((tiles_per_row - 1) * 128, p.reach, p.hop);
  SVSK_REQUIRE(p.q_fpad + fb_first >= 0 && p.q_fpad + fb_last + 16 <= p.q_ld, SVSK_E_ARG,
               "usfgan_block_bf16: aux_q rows hold columns 0..%d, the tiles read %d..%d", p.q_ld - 1, p.q_fpad + fb_first,
               p.q_fpad + fb_last + 15);
  int rc;
  CUtensorMap tm_x, tm_w1, tm_wout, tm_xout, tm_x8, tm_xw;
  {
    uint64_t dims[3] = {64, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {128, (uint64_t)p.T * 128};
    uint32_t box[3] = {64, 128, 1};
    uint32_t box_q[3] = {64, 32, 1};  // stores go out per TMEM lane quarter: 32 rows
    uint32_t box_8[3] = {64, 8, 1};   // side taps of gathered tiles: one swizzle atom (8 consecutive source rows)
    if ((rc = make_tmap_bf16(&tm_x, p.xb_in, 3, dims, str, box))) return rc;
    if ((rc = make_tmap_bf16(&tm_x8, p.xb_in, 3, dims, str, box_8))) return rc;
    uint32_t box_w[3] = {64, (uint32_t)kFWinRows, 1};  // an interior tile's rows t0 - 8 .. t0 + 135 (window mode)
    if ((rc = make_tmap_bf16(&tm_xw, p.xb_in, 3, dims, str, box_w))) return rc;
    if ((rc = make_tmap_bf16(&tm_xout, p.xb_out, 3, dims, str, box_q))) return rc;
  }
  {
    uint64_t dims[2] = {192, 128};
    uint64_t str[1] = {192 * 2};
    uint32_t box[2] = {64, 128};
    if ((rc = make_tmap_bf16(&tm_w1, p.w1p, 2, dims, str, box))) return rc;
  }
  {
    uint64_t dims[2] = {64, 64};
    uint64_t str[1] = {128};
    uint32_t box[2] = {64, 64};
    if ((rc = make_tmap_bf16(&tm_wout, p.woutp, 2, dims, str, box))) return rc;
  }
  const int smem_bytes = 3 * kFTile + 8192 + 2 * kFStage + 2 * kFTile + 8192 + 192 * 4 + (int)sizeof(UsfganFrBarriers) + 1024;
  int dev = 0, num_sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(usfgan_block_fr_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(usfgan_block_fr_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return fail((int)e, "usfgan_block_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  UsfganFrArgs a;
  a.xb_in = (const __nv_bfloat16*)p.xb_in;
  a.xb_out = (__nv_bfloat16*)p.xb_out;
  a.bias1 = p.bias1;
  a.bout = p.bout;
  a.idx_past = p.idx_past;
  a.idx_future = p.idx_future;
  a.aux_u = (const __nv_bfloat16*)p.aux_u;
  a.aux_q = (const __nv_bfloat16*)p.aux_q;
  a.q_batch_stride = p.q_batch_stride;
  a.q_ld = p.q_ld; a.q_fpad = p.q_fpad; a.hop = p.hop; a.reach = p.reach;
  a.B = p.B; a.T = p.T;
  a.dilation = p.adaptive ? 0 : p.dilation;
  a.adaptive = p.adaptive;
  a.tiles_per_row = tiles_per_row;
  a.total_tiles = p.B * tiles_per_row;
  a.out_scale = p.out_scale;
  a.out_relu = p.out_relu;
  const int grid = a.total_tiles < num_sms ? a.total_tiles : num_sms;
  const bool window = !p.adaptive && p.dilation >= 1 && p.dilation <= 8;
  if (window)
    usfgan_block_fr_kernel<true><<<grid, kFThreads, smem_bytes, as_stream(stream)>>>(tm_x, tm_w1, tm_wout, tm_xout, tm_x8, tm_xw, a);
  else
    usfgan_block_fr_kernel<false><<<grid, kFThreads, smem_bytes, as_stream(stream)>>>(tm_x, tm_w1, tm_wout, tm_xout, tm_x8, tm_xw, a);
  return check_launch("usfgan_block_bf16 (frame-rate aux)");
}

}  // namespace svsk
