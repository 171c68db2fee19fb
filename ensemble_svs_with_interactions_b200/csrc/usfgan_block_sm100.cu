// Fused uSFGAN / QPPWG residual block on sm_100a — replaces FixedBlock.forward and AdaptiveBlock.forward (+ pd_indexing)
// nnsvs/usfgan/layers/residual_block.py:123-157, 198-234 and nnsvs/usfgan/utils/index.py:12-54 with ONE launch per block.
//
//   D1[t][128] = [x(tap0) ; x(t) ; x(tap2) ; aux(t)] . W1p^T        K = 3*64 + A (A = 80 / 65 aux channels)
//   z = tanh(D1[:, :64] + b) * sigmoid(D1[:, 64:] + b)              (tanh on the FIRST half, unlike DiffNet)
//   D2[t][64]  = z . Wout^T ;   x'(t) = (D2 + bout + x(t)) * sqrt(1/2)
//   (conv1x1_skip is dead work in the reference, residual_block.py:333-336, and is not evaluated)
//   taps: FixedBlock  -> t -/+ dilation with REFLECT padding;  AdaptiveBlock -> idx_past[b,t] / idx_future[b,t]
//         (svsk_pd_index; -1 = zero).
//
// Persistent kernel, one CTA per SM looping over 128-sample tiles (time = MMA M).  The block's weights (88 KB bf16) are
// loaded into shared memory ONCE per CTA and stay resident; only activations stream:
//   warp 0      TMA producer: centre tap + aux k-blocks, and both side taps of interior fixed-block tiles
//   warp 1      GEMM1 issuer (tcgen05.mma cta_group::1, M=128, N=128) + TMEM owner
//   warp 14     GEMM2 issuer (N=64): tcgen05.mma issue blocks the issuing thread, so the second GEMM's waits and
//               commits get their own thread instead of sitting in the first GEMM's serial instruction stream
//   warps 2-5   gather producers (thread = row): side taps of adaptive blocks / boundary tiles via cp.async 16-byte
//               copies into the swizzled tile, completion signalled with cp.async.mbarrier.arrive.noinc
//   warps 6-13  epilogue (thread = sample, two warps per TMEM lane quarter alternating 16-column chunks):
//               gate -> G (bf16, swizzled smem) ; residual -> same buffer -> TMA store
// TMEM holds two D1 (2x128 columns) and two D2 (2x64) accumulators, so the MMAs of tile n+1 overlap the epilogue of
// tile n.  The residual x(t) is prefetched by its epilogue thread (one 128-byte row per thread) at the top of the tile.
#include <cuda_bf16.h>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"
#include "tma_util.cuh"

namespace svsk {

constexpr int kUTile = 128 * 128;  // 128 rows x 64 bf16
constexpr int kUMaxStages = 6;
constexpr int kUThreads = 480;  // producer, GEMM1 issuer, 4 gather, 8 epilogue, GEMM2 issuer warps

struct UsfganArgs {
  const __nv_bfloat16* xb_in;
  const float* bias1;
  const float* bout;
  const int32_t* idx_past;
  const int32_t* idx_future;
  int B, T, A, dilation, adaptive, nstages, akb, last_ksteps, tiles_per_row, total_tiles;
  float out_scale;
  int out_relu;
};

struct __align__(8) UsfganBarriers {
  uint64_t full_t[kUMaxStages];  // slot filled by TMA (1 arrival + tx bytes)
  uint64_t full_g[kUMaxStages];  // slot filled by the 128 gather threads
  uint64_t empty[kUMaxStages];
  uint64_t d1_full[2], g_full[2], d2_full[2];
  uint64_t w_full;
  uint32_t tmem_base;
};

__device__ __forceinline__ void cp_async_16(void* dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ptx::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(ptx::smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool tile_needs_gather(int t0, int T, int d, int adaptive) {
  if (adaptive) return true;
  const int last = min(t0 + 127, T - 1);
  return (t0 - d < 0) || (last + d >= T);  // a reflected tap: rows are not a shifted copy any more
}

__global__ void __launch_bounds__(kUThreads, 1)
usfgan_block_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_aux,
                    const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_wout,
                    const __grid_constant__ CUtensorMap tm_xout, const UsfganArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int KB = 3 + a.akb;                      // k-blocks per tile
  uint8_t* w1_s = smem;                          // KB tiles of [128 rows][64]
  uint8_t* wout_s = w1_s + KB * kUTile;          // [64 rows][64] = 8 KB
  uint8_t* ring = wout_s + 8192;
  uint8_t* gbuf = ring + a.nstages * kUTile;     // 3 x 16 KB, rotating: G, then the output tile, of tile n % 3
  float* bias_s = reinterpret_cast<float*>(gbuf + 3 * kUTile);  // [128] gate biases, [64] output biases
  UsfganBarriers* bars = reinterpret_cast<UsfganBarriers*>(bias_s + 192);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = a.T;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_x);
    ptx::prefetch_tmap(&tm_aux);
    ptx::prefetch_tmap(&tm_w1);
    ptx::prefetch_tmap(&tm_wout);
    ptx::prefetch_tmap(&tm_xout);
    for (int i = 0; i < a.nstages; ++i) {
      ptx::mbar_init(&bars->full_t[i], 1);
      ptx::mbar_init(&bars->full_g[i], 128);
      ptx::mbar_init(&bars->empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->d1_full[i], 1);
      ptx::mbar_init(&bars->g_full[i], 256);
      ptx::mbar_init(&bars->d2_full[i], 1);
    }
    ptx::mbar_init(&bars->w_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 192; i += kUThreads) bias_s[i] = i < 128 ? a.bias1[i] : a.bout[i - 128];
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      ptx::mbar_arrive_expect_tx(&bars->w_full, KB * kUTile + 8192);
      for (int kb = 0; kb < KB; ++kb) ptx::tma_load_2d(w1_s + kb * kUTile, &tm_w1, &bars->w_full, kb * 64, 0);
      ptx::tma_load_2d(wout_s, &tm_wout, &bars->w_full, 0, 0);
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
        const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
        const bool gather = tile_needs_gather(t0, T, a.dilation, a.adaptive);
        for (int kb = 0; kb < KB; ++kb) {
          ptx::mbar_wait(&bars->empty[s], ph ^ 1);
          uint8_t* slot = ring + s * kUTile;
          if (kb == 1) {
            ptx::mbar_arrive_expect_tx(&bars->full_t[s], kUTile);
            ptx::tma_load_3d(slot, &tm_x, &bars->full_t[s], 0, t0, b);
          } else if (kb >= 3) {
            ptx::mbar_arrive_expect_tx(&bars->full_t[s], kUTile);
            ptx::tma_load_3d(slot, &tm_aux, &bars->full_t[s], (kb - 3) * 64, t0, b);
          } else if (!gather) {
            ptx::mbar_arrive_expect_tx(&bars->full_t[s], kUTile);
            ptx::tma_load_3d(slot, &tm_x, &bars->full_t[s], 0, t0 + (kb - 1) * a.dilation, b);
          }
          if (++s == a.nstages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc1 = ptx::umma_idesc_bf16_f32(128, 128);
      ptx::mbar_wait(&bars->w_full, 0);
      ptx::tc_fence_after();
      const uint32_t ring_lo = ptx::umma_desc_lo(ptx::smem_u32(ring)), w1_lo = ptx::umma_desc_lo(ptx::smem_u32(w1_s));
      int s = 0;
      uint32_t ph = 0, pht = 0, phg = 0;  // per-slot phase bits of full_t / full_g (each toggles only when used)
      int n_issued = 0;  // tiles whose GEMM1 has been issued
      for (int tile = blockIdx.x;; tile += gridDim.x) {
        const bool have = tile < a.total_tiles;
        if (have) {
          const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
          const bool gather = tile_needs_gather(t0, T, a.dilation, a.adaptive);
          const int p = n_issued & 1;
          // D1[p] is free once the epilogue has gated tile n_issued - 2 out of it (GEMM2 has its own issuing thread, so
          // this thread has to observe g_full itself)
          if (n_issued >= 2) ptx::mbar_wait(&bars->g_full[p], ((n_issued - 2) >> 1) & 1);
          // the first k-block's barrier is probed here, every later one while the previous k-block's MMAs are issued
          bool ready = false;
          for (int kb = 0; kb < KB; ++kb) {
            const bool from_gather = gather && (kb == 0 || kb == 2);
            uint64_t* fb = from_gather ? &bars->full_g[s] : &bars->full_t[s];
            const uint32_t par = from_gather ? ((phg >> s) & 1) : ((pht >> s) & 1);
            if (!ready) ptx::mbar_wait(fb, par);
            if (from_gather) { phg ^= 1u << s; ptx::fence_proxy_async_smem(); } else { pht ^= 1u << s; }
            ptx::tc_fence_after();
            // probe the next k-block of this tile (the next tile's first k-block is waited for normally).  The probe is
            // issued before this k-block's MMAs and its result consumed after them (ptx::umma_bf16_x4_probe): a test whose
            // result is needed at once stalls this thread ~130 cycles per k-block (tools/ubench_umma.py).
            const int s_next = (s + 1 == a.nstages) ? 0 : s + 1;
            const bool ng = gather && (kb + 1 == 0 || kb + 1 == 2);
            uint64_t* nbar = ng ? &bars->full_g[s_next] : &bars->full_t[s_next];
            const uint32_t npar = ng ? ((phg >> s_next) & 1) : ((pht >> s_next) & 1);
            const uint32_t a_lo = ring_lo + s * (kUTile >> 4), b_lo = w1_lo + kb * (kUTile >> 4);
            const int ks = (kb == KB - 1) ? a.last_ksteps : 4;
            const bool r = ptx::umma_bf16_x4_probe(tmem + p * 128, a_lo, b_lo, idesc1, kb != 0, ks, nbar, npar);
            ready = r && (kb + 1 < KB);
            ptx::umma_commit(&bars->empty[s]);
            if (++s == a.nstages) { s = 0; ph ^= 1; }
          }
          ptx::umma_commit(&bars->d1_full[p]);
        }
        if (!have) break;
        ++n_issued;
      }
      (void)ph;
    }
  } else if (warp < 6) {
    // ------------------------------------------------------------------ gather producers (thread = row of the tile)
    const int r = threadIdx.x - 64;
    int s = 0;
    uint32_t ph = 0;
    // This row's two tap indices are requested one tile ahead, so that their (L2) latency is off the slot's chain.
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
    for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
      const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
      const bool gather = tile_needs_gather(t0, T, a.dilation, a.adaptive);
      const int t = t0 + r;
      const int ip = ip_next, ifu = ifu_next;
      load_idx(tile + gridDim.x, ip_next, ifu_next);
      for (int kb = 0; kb < KB; ++kb) {
        // Wait on EVERY slot, also the ones the TMA producer fills: parity waits only tell two consecutive phases apart,
        // so this warp group must never run more than one ring wrap ahead of the MMA issuer.
        ptx::mbar_wait_warp(&bars->empty[s], ph ^ 1);
        if (gather && (kb == 0 || kb == 2)) {
          int src = -1;
          if (t < T) {
            if (a.adaptive) {
              src = kb == 0 ? ip : ifu;
            } else {
              src = t + (kb - 1) * a.dilation;
              if (src < 0) src = -src;
              if (src >= T) src = 2 * (T - 1) - src;
            }
          }
          const bool ok = src >= 0 && src < T;
          const uint8_t* g = reinterpret_cast<const uint8_t*>(a.xb_in + ((size_t)b * T + (ok ? src : 0)) * 64);
          uint8_t* slot = ring + s * kUTile;
#pragma unroll
          for (int c = 0; c < 8; ++c)
            cp_async_16(slot + ptx::sw128_offset((uint32_t)r, (uint32_t)c), g + c * 16, ok ? 16u : 0u);
          cp_async_arrive_noinc(&bars->full_g[s]);
        }
        if (++s == a.nstages) { s = 0; ph ^= 1; }
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else if (warp == 14) {
    // ------------------------------------------------------------------ GEMM2 issuer: D2 = G . Wout^T per tile
    if (lane == 0) {
      const uint32_t idesc2 = ptx::umma_idesc_bf16_f32(128, 64);
      ptx::mbar_wait(&bars->w_full, 0);
      ptx::tc_fence_after();
      const uint32_t wo_lo = ptx::umma_desc_lo(ptx::smem_u32(wout_s)), g_lo = ptx::umma_desc_lo(ptx::smem_u32(gbuf));
      int m = 0;
      for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++m) {
        const int p = m & 1;
        ptx::mbar_wait(&bars->g_full[p], (m >> 1) & 1);
        ptx::tc_fence_after();
        const uint32_t gl = g_lo + (m % 3) * (kUTile >> 4);
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) ptx::umma_bf16_lo(tmem + 256 + p * 64, gl + 2 * k4, wo_lo + 2 * k4, idesc2, k4 != 0);
        ptx::umma_commit(&bars->d2_full[p]);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (thread = one sample, half the columns)
    const int q = warp & 3;
    const int sub = (warp - 6) >> 2;  // 0: 16-column chunks 0 and 2, 1: chunks 1 and 3
    const int row = q * 32 + lane;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    const bool qlead = (sub == 0 && lane == 0);  // issues the TMA stores of this lane quarter's 32 rows
    // Software-pipelined: iteration `it` gates tile it (so GEMM2(it) can be queued) and THEN finishes tile it-1, whose
    // GEMM2 ran behind GEMM1(it) in the in-order tensor pipe while this warp group was gating.
    const int my_tiles = a.total_tiles > (int)blockIdx.x ? (a.total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    uint4 xr_prev[2][2], xr_cur[2][2];
#pragma unroll
    for (int i = 0; i < 2; ++i) xr_prev[i][0] = xr_prev[i][1] = xr_cur[i][0] = xr_cur[i][1] = make_uint4(0, 0, 0, 0);
    for (int it = 0; it <= my_tiles; ++it) {
      if (it < my_tiles) {
        const int tile = blockIdx.x + it * gridDim.x;
        const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
        const int t = t0 + row, p = it & 1;
        // residual row of tile `it`, prefetched now and consumed one iteration later
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = 16 * (2 * i + sub);
          if (t < T) {
            const uint4* src = reinterpret_cast<const uint4*>(a.xb_in + ((size_t)b * T + t) * 64 + c0);
            xr_cur[i][0] = __ldg(src);
            xr_cur[i][1] = __ldg(src + 1);
          } else {
            xr_cur[i][0] = xr_cur[i][1] = make_uint4(0, 0, 0, 0);
          }
        }
        uint8_t* gb = gbuf + (it % 3) * kUTile;
        if (it >= 3) {  // buffer it%3 held the output tile of tile it-3: this quarter's TMA store must have read its rows
          if (qlead) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          ptx::named_bar_sync(4 + q, 64);
        }
        ptx::mbar_wait_warp(&bars->d1_full[p], (it >> 1) & 1);
        ptx::tc_fence_after();
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = 16 * (2 * i + sub);
          uint32_t ra[16], rb[16];
          ptx::tmem_ld16(tmem + tlane + p * 128 + c0, ra);
          ptx::tmem_ld16(tmem + tlane + p * 128 + 64 + c0, rb);
          ptx::tmem_ld_wait();
          uint32_t o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float z0 = ptx::tanh_approx(__uint_as_float(ra[2 * e]) + bias_s[c0 + 2 * e]) *
                             ptx::sigmoid_approx(__uint_as_float(rb[2 * e]) + bias_s[64 + c0 + 2 * e]);
            const float z1 = ptx::tanh_approx(__uint_as_float(ra[2 * e + 1]) + bias_s[c0 + 2 * e + 1]) *
                             ptx::sigmoid_approx(__uint_as_float(rb[2 * e + 1]) + bias_s[64 + c0 + 2 * e + 1]);
            o[e] = ptx::pack_bf16(z0, z1);
          }
          ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3)), o[0], o[1], o[2], o[3]);
          ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3) + 1), o[4], o[5], o[6], o[7]);
        }
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();
        ptx::mbar_arrive(&bars->g_full[p]);
      }
      if (it >= 1) {
        const int m = it - 1, p = m & 1;
        const int tile = blockIdx.x + m * gridDim.x;
        const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
        uint8_t* gb = gbuf + (m % 3) * kUTile;
        ptx::mbar_wait_warp(&bars->d2_full[p], (m >> 1) & 1);
        ptx::tc_fence_after();
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = 16 * (2 * i + sub);
          uint32_t rd[16];
          ptx::tmem_ld16(tmem + tlane + 256 + p * 64 + c0, rd);
          ptx::tmem_ld_wait();
          const uint32_t xw[8] = {xr_prev[i][0].x, xr_prev[i][0].y, xr_prev[i][0].z, xr_prev[i][0].w,
                                  xr_prev[i][1].x, xr_prev[i][1].y, xr_prev[i][1].z, xr_prev[i][1].w};
          uint32_t o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float lo = (__uint_as_float(rd[2 * e]) + bias_s[128 + c0 + 2 * e] + ptx::bf16_lo(xw[e])) * a.out_scale;
            float hi = (__uint_as_float(rd[2 * e + 1]) + bias_s[128 + c0 + 2 * e + 1] + ptx::bf16_hi(xw[e])) * a.out_scale;
            if (a.out_relu) { lo = fmaxf(lo, 0.f); hi = fmaxf(hi, 0.f); }
            o[e] = ptx::pack_bf16(lo, hi);
          }
          ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3)), o[0], o[1], o[2], o[3]);
          ptx::st_shared_v4(gb + ptx::sw128_offset((uint32_t)row, (uint32_t)(c0 >> 3) + 1), o[4], o[5], o[6], o[7]);
        }
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();
        // each TMEM lane quarter (two warps, 32 rows of the tile) stores its own rows: a 64-thread barrier and four
        // TMA issuers instead of a CTA-wide barrier and one
        ptx::named_bar_sync(4 + q, 64);
        if (qlead) {
          ptx::tma_store_3d(&tm_xout, gb + q * 4096, 0, t0 + q * 32, b);
          ptx::bulk_commit_group();
        }
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) { xr_prev[i][0] = xr_cur[i][0]; xr_prev[i][1] = xr_cur[i][1]; }
    }
    if (qlead) ptx::bulk_wait_read_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem, 512);
}

__global__ void usfgan_pack_kernel(const float* __restrict__ w_taps, const float* __restrict__ w_aux,
                                   const float* __restrict__ w_out, __nv_bfloat16* __restrict__ w1p,
                                   __nv_bfloat16* __restrict__ woutp, int C, int A, int G, int Ap) {
  const int K1 = 3 * C + Ap;
  const int r = blockIdx.x;
  if (r < G) {
    for (int k = threadIdx.x; k < K1; k += blockDim.x) {
      float v = 0.f;
      if (k < 3 * C) { int j = k / C, ci = k - j * C; v = w_taps[((size_t)r * C + ci) * 3 + j]; }
      else if (k - 3 * C < A) v = w_aux[(size_t)r * A + (k - 3 * C)];
      w1p[(size_t)r * K1 + k] = __float2bfloat16_rn(v);
    }
  }
  if (r < C)
    for (int k = threadIdx.x; k < G / 2; k += blockDim.x) woutp[(size_t)r * (G / 2) + k] = __float2bfloat16_rn(w_out[(size_t)r * (G / 2) + k]);
}

int usfgan_block_fr_launch(const svsk_usfgan_block_params& p, void* stream);  // usfgan_block_fr_sm100.cu

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_usfgan_pack_block(const float* w_taps, const float* w_aux, const float* w_out, void* w1p,
                                      void* woutp, int C, int A, int G, void* stream) {
  SVSK_REQUIRE(w_taps && (w_aux || A == 0) && w_out && w1p && woutp, SVSK_E_ARG, "usfgan_pack_block: null");
  SVSK_REQUIRE(C == 64 && G == 128 && A >= 0 && A <= 320, SVSK_E_ARG,
               "usfgan_pack_block: needs residual 64 / gate 128 / aux <= 320 (C=%d G=%d A=%d)", C, G, A);
  const int Ap = (A + 63) / 64 * 64;
  usfgan_pack_kernel<<<G, 128, 0, as_stream(stream)>>>(w_taps, w_aux, w_out, (__nv_bfloat16*)w1p, (__nv_bfloat16*)woutp,
                                                       C, A, G, Ap);
  return check_launch("usfgan_pack_block");
}

extern "C" int svsk_usfgan_block_bf16(const svsk_usfgan_block_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "usfgan_block_bf16: null params");
  const svsk_usfgan_block_params& p = *pp;
  const bool fr = p.aux_u != nullptr || p.aux_q != nullptr;
  SVSK_REQUIRE(p.xb_in && p.xb_out && (p.aux || fr) && p.w1p && p.woutp && p.bias1 && p.bout, SVSK_E_ARG,
               "usfgan_block_bf16: null tensor");
  SVSK_REQUIRE(p.xb_in != p.xb_out, SVSK_E_ARG, "usfgan_block_bf16: xb_in and xb_out must differ (taps read neighbours)");
  SVSK_REQUIRE(p.B > 0 && p.T > 0, SVSK_E_ARG, "usfgan_block_bf16: bad shape B=%d T=%d", p.B, p.T);
  SVSK_REQUIRE(fr || (p.A >= 1 && p.A <= 320 && p.A % 8 == 0), SVSK_E_ARG,
               "usfgan_block_bf16: bad aux width A=%d (aux row pitch must be a multiple of 16 bytes)", p.A);
  if (p.adaptive) SVSK_REQUIRE(p.idx_past && p.idx_future, SVSK_E_ARG, "usfgan_block_bf16: adaptive needs tap indices");
  else SVSK_REQUIRE(p.dilation >= 1 && p.dilation < p.T, SVSK_E_ARG,
                    "usfgan_block_bf16: reflect padding needs T > dilation (T=%d, dilation=%d)", p.T, p.dilation);
  SVSK_REQUIRE((long long)p.B * ((p.T + 127) / 128) < (1ll << 31), SVSK_E_ARG, "usfgan_block_bf16: too many tiles");
  int rc = require_sm100();
  if (rc) return rc;
  if (fr) return usfgan_block_fr_launch(p, stream);

  const int akb = (p.A + 63) / 64, KB = 3 + akb;
  const int K1p = 3 * 64 + akb * 64;
  const int fixed = KB * kUTile + 8192 + 3 * kUTile + 192 * 4 + (int)sizeof(UsfganBarriers) + 1024;
  int nstages = (232448 - fixed) / kUTile;
  if (nstages > kUMaxStages) nstages = kUMaxStages;
  SVSK_REQUIRE(nstages >= 3, SVSK_E_ARG, "usfgan_block_bf16: not enough shared memory (aux too wide)");
  const int smem_bytes = fixed + nstages * kUTile;

  CUtensorMap tm_x, tm_aux, tm_w1, tm_wout, tm_xout;
  {
    uint64_t dims[3] = {64, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {128, (uint64_t)p.T * 128};
    uint32_t box[3] = {64, 128, 1};
    uint32_t box_q[3] = {64, 32, 1};  // stores go out per TMEM lane quarter: 32 rows
    if ((rc = make_tmap_bf16(&tm_x, p.xb_in, 3, dims, str, box))) return rc;
    if ((rc = make_tmap_bf16(&tm_xout, p.xb_out, 3, dims, str, box_q))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)p.A, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.A * 2, (uint64_t)p.T * p.A * 2};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_aux, p.aux, 3, dims, str, box))) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)K1p, 128};
    uint64_t str[1] = {(uint64_t)K1p * 2};
    uint32_t box[2] = {64, 128};
    if ((rc = make_tmap_bf16(&tm_w1, p.w1p, 2, dims, str, box))) return rc;
  }
  {
    uint64_t dims[2] = {64, 64};
    uint64_t str[1] = {128};
    uint32_t box[2] = {64, 64};
    if ((rc = make_tmap_bf16(&tm_wout, p.woutp, 2, dims, str, box))) return rc;
  }
  int dev = 0, num_sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(usfgan_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return fail((int)e, "usfgan_block_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  UsfganArgs a;
  a.xb_in = (const __nv_bfloat16*)p.xb_in;
  a.bias1 = p.bias1;
  a.bout = p.bout;
  a.idx_past = p.idx_past;
  a.idx_future = p.idx_future;
  a.B = p.B; a.T = p.T; a.A = p.A;
  a.dilation = p.adaptive ? 0 : p.dilation;
  a.adaptive = p.adaptive;
  a.nstages = nstages;
  a.akb = akb;
  a.last_ksteps = (p.A - (akb - 1) * 64 + 15) / 16;
  a.tiles_per_row = (p.T + 127) / 128;
  a.total_tiles = p.B * a.tiles_per_row;
  a.out_scale = p.out_scale;
  a.out_relu = p.out_relu;
  const int grid = a.total_tiles < num_sms ? a.total_tiles : num_sms;
  usfgan_block_kernel<<<grid, kUThreads, smem_bytes, as_stream(stream)>>>(tm_x, tm_aux, tm_w1, tm_wout, tm_xout, a);
  return check_launch("usfgan_block_bf16");
}
