// General NTC bf16 Conv1d on tcgen05 — the "everything that is not a gated block" kernel of the vocoder:
// PeriodicityEstimator's three k=5 replicate-padded convs (nnsvs/usfgan/layers/residual_block.py:339-399) and the 1x1
// convs of conv_last (nnsvs/usfgan/models/generator.py:461-466).
//   y[b][t][co] = act( bias[co] + sum_j sum_ci w[co][ci][j] * x[b][src_j(t)][ci] ),  src_j(t) = t + (j - origin)*dilation
// Persistent CTAs over 128-sample tiles (time = MMA M, Cout = N <= 256).  The packed weights stay resident in shared
// memory; the input streams through a TMA ring (zero padding = TMA OOB fill).  When the taps span at most 32 rows
// ((ksize - 1) * dilation: the estimator's k = 5 convs) a ring entry is a WINDOW of 128 + span rows per 64 input channels
// and the taps are row offsets of the MMA's A descriptor, as in the DiffNet kernels: one load and one barrier round per
// channel block instead of one per tap (the three estimator convs went 2.4 -> 1.x ms at config 3); wider taps stream one
// shifted 128-row tile per tap.  Replicate / reflect padding only differs from a shifted copy on tiles that touch a
// sequence end: those tiles are filled row by row by four gather warps (cp.async).  Two TMEM accumulators let the epilogue
// (8 warps: bias, ReLU / sigmoid, bf16, swizzled smem, one TMA store per lane quarter) of tile n overlap the MMAs of n+1.
#include <cuda_bf16.h>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"
#include "tma_util.cuh"

namespace svsk {

constexpr int kCTile = 128 * 128;
constexpr int kCMaxStages = 6;
constexpr int kCThreads = 448;  // producer, MMA, 4 gather, 8 epilogue warps
constexpr int kCMaxSpan = 32;    // window mode: the taps of a tile span at most this many rows

struct ConvArgs {
  const __nv_bfloat16* x;
  const float* bias;
  int B, T, Cin, Cout, ksize, dilation, origin, pad_mode, act;
  int cb, kb_total, last_ksteps, nstages, tiles_per_row, total_tiles, out_chunks;
  int window;       // 1: a ring entry is a window of win_rows rows of one channel block, taps = row offsets
  int win_rows;     // 128 + span rounded up to 8 rows
  int stage_bytes;  // bytes of a ring entry
  int entries;      // ring entries per tile: cb (window) or kb_total
};

struct __align__(8) ConvBarriers {
  uint64_t full_t[kCMaxStages];
  uint64_t full_g[kCMaxStages];
  uint64_t empty[kCMaxStages];
  uint64_t d_full[2], d_empty[2];
  uint64_t w_full;
  uint32_t tmem_base;
};

__device__ __forceinline__ void cv_cp_async_16(void* dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ptx::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cv_cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(ptx::smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool conv_tile_needs_gather(int t0, int T, const ConvArgs& a) {
  if (a.pad_mode == SVSK_PAD_ZEROS) return false;
  const int lo = -a.origin * a.dilation, hi = (a.ksize - 1 - a.origin) * a.dilation;
  const int last = min(t0 + 127, T - 1);
  return (t0 + lo < 0) || (last + hi >= T);
}

__global__ void __launch_bounds__(kCThreads, 1)
conv1d_bf16_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                   const __grid_constant__ CUtensorMap tm_y, const ConvArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int wtile = a.Cout * 128;                      // one weight k-block: Cout rows x 64 bf16
  uint8_t* w_s = smem;
  uint8_t* ring = w_s + ((a.kb_total * wtile + 1023) & ~1023);
  uint8_t* obuf = ring + a.nstages * a.stage_bytes;    // 2 x out_chunks x 16 KB output staging
  float* bias_s = reinterpret_cast<float*>(obuf + 2 * a.out_chunks * kCTile);
  ConvBarriers* bars = reinterpret_cast<ConvBarriers*>(bias_s + 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = a.T, KB = a.kb_total;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_x);
    ptx::prefetch_tmap(&tm_w);
    ptx::prefetch_tmap(&tm_y);
    for (int i = 0; i < a.nstages; ++i) {
      ptx::mbar_init(&bars->full_t[i], 1);
      ptx::mbar_init(&bars->full_g[i], 128);
      ptx::mbar_init(&bars->empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->d_full[i], 1);
      ptx::mbar_init(&bars->d_empty[i], 256);
    }
    ptx::mbar_init(&bars->w_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 256; i += kCThreads) bias_s[i] = (i < a.Cout && a.bias) ? a.bias[i] : 0.f;
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp == 0) {
    if (lane == 0) {
      ptx::mbar_arrive_expect_tx(&bars->w_full, KB * wtile);
      for (int kb = 0; kb < KB; ++kb) ptx::tma_load_2d(w_s + kb * wtile, &tm_w, &bars->w_full, kb * 64, 0);
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
        const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
        const bool gather = conv_tile_needs_gather(t0, T, a);
        for (int e = 0; e < a.entries; ++e) {
          ptx::mbar_wait(&bars->empty[s], ph ^ 1);
          if (!gather) {
            ptx::mbar_arrive_expect_tx(&bars->full_t[s], a.stage_bytes);
            if (a.window) {
              ptx::tma_load_3d(ring + s * a.stage_bytes, &tm_x, &bars->full_t[s], e * 64, t0 - a.origin * a.dilation, b);
            } else {
              const int j = e / a.cb, cb = e - j * a.cb;
              ptx::tma_load_3d(ring + s * a.stage_bytes, &tm_x, &bars->full_t[s], cb * 64, t0 + (j - a.origin) * a.dilation, b);
            }
          }
          if (++s == a.nstages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = ptx::umma_idesc_bf16_f32(128, a.Cout);
      ptx::mbar_wait(&bars->w_full, 0);
      ptx::tc_fence_after();
      const uint32_t wa = ptx::smem_u32(w_s);
      int s = 0, n = 0;
      uint32_t pht = 0, phg = 0;
      for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++n) {
        const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
        const bool gather = conv_tile_needs_gather(t0, T, a);
        const int p = n & 1;
        ptx::mbar_wait(&bars->d_empty[p], ((n >> 1) & 1) ^ 1);  // epilogue of tile n-2 has drained this accumulator
        ptx::tc_fence_after();
        for (int e = 0; e < a.entries; ++e) {
          if (gather) {
            ptx::mbar_wait(&bars->full_g[s], (phg >> s) & 1);
            phg ^= 1u << s;
            ptx::fence_proxy_async_smem();
          } else {
            ptx::mbar_wait(&bars->full_t[s], (pht >> s) & 1);
            pht ^= 1u << s;
          }
          ptx::tc_fence_after();
          const uint32_t a0 = ptx::smem_u32(ring + s * a.stage_bytes);
          if (a.window) {  // entry = channel block e: every tap is the same window read at a row offset
            const int ks = (e == a.cb - 1) ? a.last_ksteps : 4;
            for (int j = 0; j < a.ksize; ++j)
              for (int k4 = 0; k4 < ks; ++k4)
                ptx::umma_bf16(tmem + p * 256, ptx::umma_desc_k_sw128(a0 + j * a.dilation * 128 + k4 * 32),
                               ptx::umma_desc_k_sw128(wa + (j * a.cb + e) * wtile + k4 * 32), idesc, (e | j | k4) != 0);
          } else {
            const int cb = e % a.cb;
            const int ks = (cb == a.cb - 1) ? a.last_ksteps : 4;
            for (int k4 = 0; k4 < ks; ++k4)
              ptx::umma_bf16(tmem + p * 256, ptx::umma_desc_k_sw128(a0 + k4 * 32),
                             ptx::umma_desc_k_sw128(wa + e * wtile + k4 * 32), idesc, (e | k4) != 0);
          }
          ptx::umma_commit(&bars->empty[s]);
          if (++s == a.nstages) s = 0;
        }
        ptx::umma_commit(&bars->d_full[p]);
      }
    }
  } else if (warp < 6) {
    const int r = threadIdx.x - 64;
    int s = 0;
    uint32_t ph = 0;
    const int row_chunks = a.Cin / 8;  // 16-byte chunks in one input row
    for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
      const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
      const bool gather = conv_tile_needs_gather(t0, T, a);
      const int t = t0 + r;
      for (int e = 0; e < a.entries; ++e) {
        ptx::mbar_wait(&bars->empty[s], ph ^ 1);  // every slot: stay within one ring wrap of the MMA issuer
        if (gather) {
          const int j = a.window ? 0 : e / a.cb, cb = a.window ? e : e - j * a.cb;
          uint8_t* slot = ring + s * a.stage_bytes;
          // window mode: rows r and r + 128 of the window (row i <-> sample t0 - origin * dilation + i); else row r of tap j
          for (int wr = r; wr < (a.window ? a.win_rows : 128); wr += 128) {
            int src = -1;
            if (a.window ? (t0 + wr - a.origin * a.dilation < T + (a.ksize - 1 - a.origin) * a.dilation) : (t < T)) {
              src = a.window ? t0 - a.origin * a.dilation + wr : t + (j - a.origin) * a.dilation;
              if (a.pad_mode == SVSK_PAD_REFLECT) {
                if (src < 0) src = -src;
                if (src >= T) src = 2 * (T - 1) - src;
              } else {
                src = src < 0 ? 0 : (src >= T ? T - 1 : src);
              }
            }
            const bool ok = src >= 0 && src < T;
            const uint8_t* g = reinterpret_cast<const uint8_t*>(a.x + ((size_t)b * T + (ok ? src : 0)) * a.Cin) + cb * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const bool have = ok && (cb * 8 + c) < row_chunks;
              cv_cp_async_16(slot + ptx::sw128_offset((uint32_t)wr, (uint32_t)c), have ? g + c * 16 : g, have ? 16u : 0u);
            }
          }
          cv_cp_async_arrive_noinc(&bars->full_g[s]);
        }
        if (++s == a.nstages) { s = 0; ph ^= 1; }
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else {
    const int q = warp & 3;
    const int sub = (warp - 6) >> 2;  // the two warps of a TMEM lane quarter alternate 16-column chunks
    const int row = q * 32 + lane;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    const bool qlead = (sub == 0 && lane == 0);  // issues the quarter's TMA stores
    int n = 0;
    for (int tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++n) {
      const int b = tile / a.tiles_per_row, t0 = (tile - b * a.tiles_per_row) * 128;
      const int p = n & 1;
      uint8_t* ob = obuf + p * a.out_chunks * kCTile;
      if (n >= 2) {  // this quarter's 32 rows of the buffer: its TMA store of tile n-2 must have read them
        if (qlead) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        ptx::named_bar_sync(1 + q, 64);
      }
      ptx::mbar_wait(&bars->d_full[p], (n >> 1) & 1);
      ptx::tc_fence_after();
      for (int c0 = 16 * sub; c0 < a.Cout; c0 += 32) {
        uint32_t rd[16];
        ptx::tmem_ld16(tmem + tlane + p * 256 + c0, rd);
        ptx::tmem_ld_wait();
        uint32_t o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float v0 = __uint_as_float(rd[2 * e]) + bias_s[c0 + 2 * e];
          float v1 = __uint_as_float(rd[2 * e + 1]) + bias_s[c0 + 2 * e + 1];
          if (a.act == SVSK_ACT_RELU) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
          else if (a.act == SVSK_ACT_SIGMOID) { v0 = ptx::sigmoid_approx(v0); v1 = ptx::sigmoid_approx(v1); }
          o[e] = ptx::pack_bf16(v0, v1);
        }
        uint8_t* oc = ob + (c0 >> 6) * kCTile;
        const uint32_t ch16 = (uint32_t)((c0 & 63) >> 3);
        ptx::st_shared_v4(oc + ptx::sw128_offset((uint32_t)row, ch16), o[0], o[1], o[2], o[3]);
        ptx::st_shared_v4(oc + ptx::sw128_offset((uint32_t)row, ch16 + 1), o[4], o[5], o[6], o[7]);
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(&bars->d_empty[p]);
      ptx::fence_proxy_async_smem();
      ptx::named_bar_sync(1 + q, 64);
      if (qlead) {  // one store per TMEM lane quarter (32 rows): no CTA-wide barrier, four issuers
        for (int oc = 0; oc < a.out_chunks; ++oc)
          ptx::tma_store_3d(&tm_y, ob + oc * kCTile + q * 4096, oc * 64, t0 + q * 32, b);
        ptx::bulk_commit_group();
      }
    }
    if (qlead) ptx::bulk_wait_read_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem, 512);
}

__global__ void conv1d_pack_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wp, int Cout, int Cin, int ks,
                                   int Cinp) {
  const int co = blockIdx.x;
  const int K = ks * Cinp;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const int j = k / Cinp, ci = k - j * Cinp;
    wp[(size_t)co * K + k] = __float2bfloat16_rn(ci < Cin ? w[((size_t)co * Cin + ci) * ks + j] : 0.f);
  }
}

// s = a*h + (1-a)*n on NTC bf16 (generator.py:505-507); fp32 math
__global__ void periodic_mix_bf16_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ h,
                                         const __nv_bfloat16* __restrict__ n, __nv_bfloat16* __restrict__ s, size_t cnt8) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cnt8) return;
  const uint4 av = reinterpret_cast<const uint4*>(a)[i], hv = reinterpret_cast<const uint4*>(h)[i],
              nv = reinterpret_cast<const uint4*>(n)[i];
  const uint32_t aw[4] = {av.x, av.y, av.z, av.w}, hw[4] = {hv.x, hv.y, hv.z, hv.w}, nw[4] = {nv.x, nv.y, nv.z, nv.w};
  uint32_t o[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float a0 = ptx::bf16_lo(aw[e]), a1 = ptx::bf16_hi(aw[e]);
    o[e] = ptx::pack_bf16(a0 * ptx::bf16_lo(hw[e]) + (1.f - a0) * ptx::bf16_lo(nw[e]),
                          a1 * ptx::bf16_hi(hw[e]) + (1.f - a1) * ptx::bf16_hi(nw[e]));
  }
  reinterpret_cast<uint4*>(s)[i] = make_uint4(o[0], o[1], o[2], o[3]);
}

// y[n] = bias + sum_c w[c] * x[n][c]   (the final 64 -> 1 projection of conv_last); one thread per row
__global__ void dot_rows_bf16_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w, float bias,
                                     float* __restrict__ y, size_t rows, int C) {
  size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const uint4* xr = reinterpret_cast<const uint4*>(x + r * C);
  float acc = bias;
  for (int c8 = 0; c8 < C / 8; ++c8) {
    const uint4 v = xr[c8];
    const uint32_t vw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) acc += ptx::bf16_lo(vw[e]) * w[c8 * 8 + 2 * e] + ptx::bf16_hi(vw[e]) * w[c8 * 8 + 2 * e + 1];
  }
  y[r] = acc;
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_conv1d_pack_bf16(const float* w, void* wp, int Cout, int Cin, int ksize, void* stream) {
  SVSK_REQUIRE(w && wp && Cout > 0 && Cin > 0 && ksize >= 1 && ksize <= 8, SVSK_E_ARG, "conv1d_pack_bf16: bad args");
  const int Cinp = (Cin + 63) / 64 * 64;
  conv1d_pack_kernel<<<Cout, 128, 0, as_stream(stream)>>>(w, (__nv_bfloat16*)wp, Cout, Cin, ksize, Cinp);
  return check_launch("conv1d_pack_bf16");
}

extern "C" int svsk_conv1d_bf16(const svsk_conv1d_bf16_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "conv1d_bf16: null params");
  const svsk_conv1d_bf16_params& p = *pp;
  SVSK_REQUIRE(p.x && p.wp && p.y, SVSK_E_ARG, "conv1d_bf16: null tensor");
  SVSK_REQUIRE(p.x != p.y, SVSK_E_ARG, "conv1d_bf16: in-place is not supported");
  SVSK_REQUIRE(p.B > 0 && p.T > 0 && p.Cin >= 8 && p.Cin % 8 == 0, SVSK_E_ARG, "conv1d_bf16: Cin=%d must be a multiple of 8", p.Cin);
  SVSK_REQUIRE(p.Cout >= 16 && p.Cout <= 256 && p.Cout % 16 == 0, SVSK_E_ARG, "conv1d_bf16: Cout=%d (16..256, %%16)", p.Cout);
  SVSK_REQUIRE(p.ksize >= 1 && p.ksize <= 8 && p.dilation >= 1 && p.tap_origin >= 0 && p.tap_origin < p.ksize, SVSK_E_ARG,
               "conv1d_bf16: bad taps");
  SVSK_REQUIRE(p.pad_mode == SVSK_PAD_ZEROS || p.pad_mode == SVSK_PAD_REFLECT || p.pad_mode == SVSK_PAD_REPLICATE,
               SVSK_E_ARG, "conv1d_bf16: pad_mode %d", p.pad_mode);
  if (p.pad_mode == SVSK_PAD_REFLECT) {
    const int reach = (p.tap_origin > p.ksize - 1 - p.tap_origin ? p.tap_origin : p.ksize - 1 - p.tap_origin) * p.dilation;
    SVSK_REQUIRE(reach < p.T, SVSK_E_ARG, "conv1d_bf16: reflect padding needs T > %d", reach);
  }
  int rc = require_sm100();
  if (rc) return rc;

  const int cb = (p.Cin + 63) / 64, KB = p.ksize * cb, Cinp = cb * 64;
  const int wtile = p.Cout * 128;
  const int out_chunks = (p.Cout + 63) / 64;
  const int wbytes = (KB * wtile + 1023) & ~1023;
  const int fixed = wbytes + 2 * out_chunks * kCTile + 256 * 4 + (int)sizeof(ConvBarriers) + 1024;
  // window mode: all taps of a tile out of one (128 + span)-row load per channel block
  const int span = (p.ksize - 1) * p.dilation;
  const int window = (p.ksize > 1 && span <= kCMaxSpan) ? 1 : 0;
  const int win_rows = window ? (128 + span + 7) / 8 * 8 : 128;
  const int stage_bytes = win_rows * 128;
  int nstages = (232448 - fixed) / stage_bytes;
  if (nstages > kCMaxStages) nstages = kCMaxStages;
  SVSK_REQUIRE(nstages >= 3, SVSK_E_ARG, "conv1d_bf16: weights (%d KB) do not fit shared memory", wbytes / 1024);
  const int smem_bytes = fixed + nstages * stage_bytes;

  CUtensorMap tm_x, tm_w, tm_y;
  {
    uint64_t dims[3] = {(uint64_t)p.Cin, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.Cin * 2, (uint64_t)p.T * p.Cin * 2};
    uint32_t box[3] = {64, (uint32_t)win_rows, 1};
    if ((rc = make_tmap_bf16(&tm_x, p.x, 3, dims, str, box))) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)p.ksize * Cinp, (uint64_t)p.Cout};
    uint64_t str[1] = {(uint64_t)p.ksize * Cinp * 2};
    uint32_t box[2] = {64, (uint32_t)p.Cout};
    if ((rc = make_tmap_bf16(&tm_w, p.wp, 2, dims, str, box))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)p.Cout, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.Cout * 2, (uint64_t)p.T * p.Cout * 2};
    uint32_t box[3] = {64, 32, 1};  // stores go out per epilogue warp: 32 rows
    if ((rc = make_tmap_bf16(&tm_y, p.y, 3, dims, str, box))) return rc;
  }
  int dev = 0, num_sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv1d_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return fail((int)e, "conv1d_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  ConvArgs a;
  a.x = (const __nv_bfloat16*)p.x;
  a.bias = p.bias;
  a.B = p.B; a.T = p.T; a.Cin = p.Cin; a.Cout = p.Cout;
  a.ksize = p.ksize; a.dilation = p.dilation; a.origin = p.tap_origin; a.pad_mode = p.pad_mode; a.act = p.act;
  a.cb = cb;
  a.kb_total = KB;
  a.last_ksteps = (p.Cin - (cb - 1) * 64 + 15) / 16;
  a.nstages = nstages;
  a.tiles_per_row = (p.T + 127) / 128;
  SVSK_REQUIRE((long long)p.B * a.tiles_per_row < (1ll << 31), SVSK_E_ARG, "conv1d_bf16: too many tiles");
  a.total_tiles = p.B * a.tiles_per_row;
  a.out_chunks = out_chunks;
  a.window = window;
  a.win_rows = win_rows;
  a.stage_bytes = stage_bytes;
  a.entries = window ? cb : KB;
  const int grid = a.total_tiles < num_sms ? a.total_tiles : num_sms;
  conv1d_bf16_kernel<<<grid, kCThreads, smem_bytes, as_stream(stream)>>>(tm_x, tm_w, tm_y, a);
  return check_launch("conv1d_bf16");
}

extern "C" int svsk_periodic_mix_bf16(const void* a, const void* h, const void* n, void* s, size_t cnt, void* stream) {
  SVSK_REQUIRE(a && h && n && s, SVSK_E_ARG, "periodic_mix_bf16: null");
  SVSK_REQUIRE(cnt % 8 == 0, SVSK_E_ARG, "periodic_mix_bf16: element count must be a multiple of 8");
  if (cnt == 0) return 0;
  const size_t cnt8 = cnt / 8;
  periodic_mix_bf16_kernel<<<(unsigned)((cnt8 + 255) / 256), 256, 0, as_stream(stream)>>>(
      (const __nv_bfloat16*)a, (const __nv_bfloat16*)h, (const __nv_bfloat16*)n, (__nv_bfloat16*)s, cnt8);
  return check_launch("periodic_mix_bf16");
}

extern "C" int svsk_dot_rows_bf16(const void* x, const float* w, float bias, float* y, size_t rows, int C, void* stream) {
  SVSK_REQUIRE(x && w && y && C >= 8 && C % 8 == 0, SVSK_E_ARG, "dot_rows_bf16: bad args");
  if (rows == 0) return 0;
  dot_rows_bf16_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, as_stream(stream)>>>((const __nv_bfloat16*)x, w, bias, y,
                                                                                       rows, C);
  return check_launch("dot_rows_bf16");
}
