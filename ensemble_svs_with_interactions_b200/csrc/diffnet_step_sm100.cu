// Everything between two residual-stack launches of a DDPM sampling step, in ONE launch per 128-frame tile:
//   tail   h   = relu(skip_projection(skip_sum / sqrt(L)))             nnsvs/diffsinger/denoiser.py:120-122
//          eps = output_projection(h)                                   denoiser.py:123
//   update x   <- posterior mean (clipped x0) + [t > 0] * sigma_t * z   nnsvs/diffsinger/diffusion.py:164-204
//   head   xb  = relu(input_projection(x))  (the next denoiser call)    denoiser.py:109-112
// Before: cast -> GEMM -> GEMM -> update -> cast -> GEMM as six launches (~50 of the 455 us of a step at BASELINE
// config 2, almost all of it launch latency of dependent tiny kernels).  Three chained tcgen05 GEMMs here, M = 128
// frames per CTA, operands staged once in shared memory, accumulators in TMEM:
//   GEMM-a  D_a[128][C]  = A[128][C] . Wskip[C][C]^T     A = bf16(skip32 * scale), converted by the CTA's threads
//   GEMM-b  D_b[128][Mp] = H[128][C] . Wout[Mp][C]^T     H = bf16(relu(D_a + b_skip)) written over A
//   GEMM-c  D_c[128][C]  = X[128][Mp] . Win[C][Mp]^T     X = bf16(updated x) written over H; D_c reuses D_a's columns
// The weight region holds Wskip first (C/64 tiles of C rows), then Wout (C/64 tiles of Mp rows) and Win (ceil(Mp/64)
// tiles of C rows), TMA-loaded as soon as GEMM-a has completed.
#include <cuda_bf16.h>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"
#include "tma_util.cuh"

namespace svsk {

constexpr int kStepThreads = 256;
constexpr int kStepTile = 128 * 128;  // 128 rows x 64 bf16

struct DiffnetStepArgs {
  const float* skip32;
  float* x32s;
  const float* z;
  float* eps_out;
  const float *b_skip, *b_out, *b_in;
  const long long* t;
  const float *sra, *srm1, *c1, *c2, *plv;
  float skip_scale;
  int B, T, C, Mp, clip, head;
};

struct __align__(8) DiffnetStepBarriers {
  uint64_t w_full[2];    // 0: Wskip landed, 1: Wout + Win landed
  uint64_t mma_done[3];  // GEMM-a, -b, -c complete
  uint32_t tmem_base;
};

// kC = C (128 or 256) is compile-time: the staging loops divide by C / 8 per element, and constants in the single-thread
// roles' loops are worth several per cent on this library's kernels (DESIGN §4 item 17).
template <int kC>
__global__ void __launch_bounds__(kStepThreads, 1)
diffnet_step_kernel(const __grid_constant__ CUtensorMap tm_wskip, const __grid_constant__ CUtensorMap tm_wout,
                    const __grid_constant__ CUtensorMap tm_win, const __grid_constant__ CUtensorMap tm_xout,
                    const DiffnetStepArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int C = kC;
  const int Mp = a.Mp, T = a.T;
  constexpr int CB = C / 64;
  const int MB = (Mp + 63) / 64;
  uint8_t* ah = smem;                       // CB tiles: A, then H, then X (2 tiles), then the output tile
  uint8_t* ws = ah + CB * kStepTile;        // CB tiles of C rows (Wskip); later Wout | Win
  constexpr int ws_tile = C * 128;          // bytes of one Wskip / Win tile
  uint8_t* wout_s = ws;                     // CB tiles at a 16 KB pitch (Mp <= 128 rows each)
  uint8_t* win_s = ws + CB * kStepTile;     // MB tiles of C rows
  const int ws_bytes = max(CB * ws_tile, CB * kStepTile + MB * ws_tile);
  DiffnetStepBarriers* bars = reinterpret_cast<DiffnetStepBarriers*>(ws + ws_bytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y, t0 = blockIdx.x * 128;

  if (threadIdx.x == 0) {
    ptx::prefetch_tmap(&tm_wskip);
    ptx::prefetch_tmap(&tm_wout);
    ptx::prefetch_tmap(&tm_win);
    ptx::prefetch_tmap(&tm_xout);
    ptx::mbar_init(&bars->w_full[0], 1);
    ptx::mbar_init(&bars->w_full[1], 1);
    for (int i = 0; i < 3; ++i) ptx::mbar_init(&bars->mma_done[i], 1);
    ptx::fence_mbar_init();
    ptx::mbar_arrive_expect_tx(&bars->w_full[0], CB * ws_tile);
    for (int kb = 0; kb < CB; ++kb) ptx::tma_load_2d(ws + kb * ws_tile, &tm_wskip, &bars->w_full[0], kb * 64, 0);
  }
  if (warp == 1) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }

  // ---- A = bf16(skip32 * scale): 16 bytes (8 channels) per thread and step, rows past the end of the track = 0.
  //      Eight steps' loads are in flight together (the loop is bound by the latency of its 128 KB of fp32 reads).
  {
    const int chunks = C / 8;  // 16-byte bf16 chunks per row
    const int total = 128 * chunks;
    const float s = a.skip_scale;
    for (int i0 = threadIdx.x; i0 < total; i0 += 8 * kStepThreads) {
      float4 v[8][2];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * kStepThreads;
        const int r = i / chunks, ch = i - r * chunks;
        v[u][0] = v[u][1] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total && t0 + r < T) {
          const float4* src = reinterpret_cast<const float4*>(a.skip32 + ((size_t)b * T + t0 + r) * C + ch * 8);
          v[u][0] = __ldg(src);
          v[u][1] = __ldg(src + 1);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * kStepThreads;
        if (i < total) {
          const int r = i / chunks, ch = i - r * chunks;
          ptx::st_shared_v4(ah + (ch >> 3) * kStepTile + ptx::sw128_offset((uint32_t)r, (uint32_t)(ch & 7)),
                            ptx::pack_bf16(v[u][0].x * s, v[u][0].y * s), ptx::pack_bf16(v[u][0].z * s, v[u][0].w * s),
                            ptx::pack_bf16(v[u][1].x * s, v[u][1].y * s), ptx::pack_bf16(v[u][1].z * s, v[u][1].w * s));
        }
      }
    }
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const uint32_t tm_a = tmem, tm_b = tmem + 256;  // D_a / D_c: columns [0, C) ; D_b: columns [256, 256 + Mp)

  // ---- GEMM-a
  if (threadIdx.x == 0) {
    ptx::mbar_wait(&bars->w_full[0], 0);
    ptx::tc_fence_after();
    const uint32_t idesc = ptx::umma_idesc_bf16_f32(128, (uint32_t)C);
    const uint32_t a_lo = ptx::umma_desc_lo(ptx::smem_u32(ah)), w_lo = ptx::umma_desc_lo(ptx::smem_u32(ws));
    for (int kb = 0; kb < CB; ++kb)
      for (int k4 = 0; k4 < 4; ++k4)
        ptx::umma_bf16_lo(tm_a, a_lo + kb * (kStepTile >> 4) + 2 * k4, w_lo + kb * (ws_tile >> 4) + 2 * k4, idesc, (kb | k4) != 0);
    ptx::umma_commit(&bars->mma_done[0]);
  }
  ptx::mbar_wait(&bars->mma_done[0], 0);
  ptx::tc_fence_after();
  if (threadIdx.x == 0) {  // Wskip is dead: bring in the other two weight matrices while H is being written
    ptx::mbar_arrive_expect_tx(&bars->w_full[1], CB * Mp * 128 + (a.head ? MB * ws_tile : 0));
    for (int kb = 0; kb < CB; ++kb) ptx::tma_load_2d(wout_s + kb * kStepTile, &tm_wout, &bars->w_full[1], kb * 64, 0);
    if (a.head)
      for (int kb = 0; kb < MB; ++kb) ptx::tma_load_2d(win_s + kb * ws_tile, &tm_win, &bars->w_full[1], kb * 64, 0);
  }

  const int q = warp & 3, half = warp >> 2;  // TMEM lane quarter ; the two warps of a quarter alternate 16-column chunks
  const int row = q * 32 + lane, tt = t0 + row;
  const bool in_seq = tt < T;
  const uint32_t tlane = (uint32_t)(q * 32) << 16;

  // ---- H = bf16(relu(D_a + b_skip)) over A
  for (int c0 = 16 * half; c0 < C; c0 += 32) {
    uint32_t r[16];
    ptx::tmem_ld16(tm_a + tlane + c0, r);
    ptx::tmem_ld_wait();
    uint32_t o[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float v0 = fmaxf(__uint_as_float(r[2 * e]) + __ldg(a.b_skip + c0 + 2 * e), 0.f);
      const float v1 = fmaxf(__uint_as_float(r[2 * e + 1]) + __ldg(a.b_skip + c0 + 2 * e + 1), 0.f);
      o[e] = ptx::pack_bf16(v0, v1);
    }
    uint8_t* tile = ah + (c0 >> 6) * kStepTile;
    const uint32_t ch = (uint32_t)((c0 & 63) >> 3);
    ptx::st_shared_v4(tile + ptx::sw128_offset((uint32_t)row, ch), o[0], o[1], o[2], o[3]);
    ptx::st_shared_v4(tile + ptx::sw128_offset((uint32_t)row, ch + 1), o[4], o[5], o[6], o[7]);
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();

  // ---- GEMM-b
  if (threadIdx.x == 0) {
    ptx::mbar_wait(&bars->w_full[1], 0);
    ptx::tc_fence_after();
    const uint32_t idesc = ptx::umma_idesc_bf16_f32(128, (uint32_t)Mp);
    const uint32_t h_lo = ptx::umma_desc_lo(ptx::smem_u32(ah)), w_lo = ptx::umma_desc_lo(ptx::smem_u32(wout_s));
    for (int kb = 0; kb < CB; ++kb)
      for (int k4 = 0; k4 < 4; ++k4)
        ptx::umma_bf16_lo(tm_b, h_lo + kb * (kStepTile >> 4) + 2 * k4, w_lo + kb * (kStepTile >> 4) + 2 * k4, idesc, (kb | k4) != 0);
    ptx::umma_commit(&bars->mma_done[1]);
  }
  // x and z of this thread's first three 16-channel chunks are requested while GEMM-b runs (z streams from HBM)
  float4 xr[3][4], zr[3][4];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int c0 = 16 * half + 32 * k;
#pragma unroll
    for (int e = 0; e < 4; ++e) xr[k][e] = zr[k][e] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (in_seq && c0 < Mp) {
      const size_t base = ((size_t)b * T + tt) * Mp + c0;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        xr[k][e] = *reinterpret_cast<const float4*>(a.x32s + base + 4 * e);
        zr[k][e] = __ldg(reinterpret_cast<const float4*>(a.z + base + 4 * e));
      }
    }
  }
  ptx::mbar_wait(&bars->mma_done[1], 0);
  ptx::tc_fence_after();

  // ---- eps = D_b + b_out ; DDPM update of x in place ; X = bf16(x) over H
  {
    const long long tb = a.t[b];
    const float ca = a.sra[tb], cb = a.srm1[tb], c1 = a.c1[tb], c2 = a.c2[tb];
    const float sigma = tb == 0 ? 0.f : expf(0.5f * a.plv[tb]);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c0 = 16 * half + 32 * k;
      if (c0 < Mp) {
        uint32_t r[16];
        ptx::tmem_ld16(tm_b + tlane + c0, r);
        ptx::tmem_ld_wait();
        uint32_t o[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (in_seq) {
          const size_t base = ((size_t)b * T + tt) * Mp + c0;
          float xn[16];
#pragma unroll
          for (int e = 0; e < 16; e += 4) {
            float4 xv, zv;
            if (k < 3) { xv = xr[k < 3 ? k : 0][e >> 2]; zv = zr[k < 3 ? k : 0][e >> 2]; }
            else {
              xv = *reinterpret_cast<const float4*>(a.x32s + base + e);
              zv = __ldg(reinterpret_cast<const float4*>(a.z + base + e));
            }
            const float4 bo = __ldg(reinterpret_cast<const float4*>(a.b_out + c0 + e));
            const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, zs[4] = {zv.x, zv.y, zv.z, zv.w}, bs[4] = {bo.x, bo.y, bo.z, bo.w};
            float ep[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              ep[u] = __uint_as_float(r[e + u]) + bs[u];
              float x0 = ca * xs[u] - cb * ep[u];
              if (a.clip) x0 = fminf(fmaxf(x0, -1.f), 1.f);
              const float mean = c1 * x0 + c2 * xs[u];
              xn[e + u] = mean + sigma * zs[u];
            }
            *reinterpret_cast<float4*>(a.x32s + base + e) = make_float4(xn[e], xn[e + 1], xn[e + 2], xn[e + 3]);
            if (a.eps_out) *reinterpret_cast<float4*>(a.eps_out + base + e) = make_float4(ep[0], ep[1], ep[2], ep[3]);
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = ptx::pack_bf16(xn[2 * e], xn[2 * e + 1]);
        }
        if (a.head) {
          uint8_t* tile = ah + (c0 >> 6) * kStepTile;
          const uint32_t ch = (uint32_t)((c0 & 63) >> 3);
          ptx::st_shared_v4(tile + ptx::sw128_offset((uint32_t)row, ch), o[0], o[1], o[2], o[3]);
          ptx::st_shared_v4(tile + ptx::sw128_offset((uint32_t)row, ch + 1), o[4], o[5], o[6], o[7]);
        }
      }
    }
  }
  if (a.head) {  // uniform over the grid: the last sampling step has no next denoiser call
    ptx::fence_proxy_async_smem();
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();

    // ---- GEMM-c (K = Mp: whole 16-column steps only, the weight tile's columns past Mp are TMA zero fill)
    if (threadIdx.x == 0) {
      const uint32_t idesc = ptx::umma_idesc_bf16_f32(128, (uint32_t)C);
      const uint32_t x_lo = ptx::umma_desc_lo(ptx::smem_u32(ah)), w_lo = ptx::umma_desc_lo(ptx::smem_u32(win_s));
      const int ksteps = Mp / 16;
      for (int ks = 0; ks < ksteps; ++ks) {
        const int kb = ks >> 2, k4 = ks & 3;
        ptx::umma_bf16_lo(tm_a, x_lo + kb * (kStepTile >> 4) + 2 * k4, w_lo + kb * (ws_tile >> 4) + 2 * k4, idesc, ks != 0);
      }
      ptx::umma_commit(&bars->mma_done[2]);
    }
    ptx::mbar_wait(&bars->mma_done[2], 0);
    ptx::tc_fence_after();

    // ---- xb = bf16(relu(D_c + b_in)) over X, then one TMA store per 64-channel tile (rows past the end are clipped)
    for (int c0 = 16 * half; c0 < C; c0 += 32) {
      uint32_t r[16];
      ptx::tmem_ld16(tm_a + tlane + c0, r);
      ptx::tmem_ld_wait();
      uint32_t o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float v0 = fmaxf(__uint_as_float(r[2 * e]) + __ldg(a.b_in + c0 + 2 * e), 0.f);
        const float v1 = fmaxf(__uint_as_float(r[2 * e + 1]) + __ldg(a.b_in + c0 + 2 * e + 1), 0.f);
        o[e] = ptx::pack_bf16(v0, v1);
      }
      uint8_t* tile = ah + (c0 >> 6) * kStepTile;
      const uint32_t ch = (uint32_t)((c0 & 63) >> 3);
      ptx::st_shared_v4(tile + ptx::sw128_offset((uint32_t)row, ch), o[0], o[1], o[2], o[3]);
      ptx::st_shared_v4(tile + ptx::sw128_offset((uint32_t)row, ch + 1), o[4], o[5], o[6], o[7]);
    }
    ptx::fence_proxy_async_smem();
    ptx::tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int cb = 0; cb < CB; ++cb) ptx::tma_store_3d(&tm_xout, ah + cb * kStepTile, cb * 64, t0, b);
      ptx::bulk_commit_group();
      ptx::bulk_wait_read_all();
    }
  } else {
    ptx::tc_fence_before();
    __syncthreads();
  }
  if (warp == 1) ptx::tmem_dealloc(tmem, 512);
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_diffnet_step_bf16(const svsk_diffnet_step_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "diffnet_step_bf16: null params");
  const svsk_diffnet_step_params& p = *pp;
  SVSK_REQUIRE(p.skip32 && p.x32s && p.z && p.w_skip && p.w_out && p.b_skip && p.b_out && p.t && p.sqrt_recip_alphas_cumprod &&
                   p.sqrt_recipm1_alphas_cumprod && p.posterior_mean_coef1 && p.posterior_mean_coef2 &&
                   p.posterior_log_variance_clipped,
               SVSK_E_ARG, "diffnet_step_bf16: null tensor");
  SVSK_REQUIRE(p.xb_out == nullptr || (p.w_in && p.b_in), SVSK_E_ARG, "diffnet_step_bf16: xb_out needs w_in / b_in");
  SVSK_REQUIRE(p.C == 128 || p.C == 256, SVSK_E_ARG, "diffnet_step_bf16: C=%d (need 128 or 256)", p.C);
  SVSK_REQUIRE(p.Mp >= 16 && p.Mp <= 128 && p.Mp % 16 == 0, SVSK_E_ARG, "diffnet_step_bf16: Mp=%d (need a multiple of 16, 16..128)", p.Mp);
  SVSK_REQUIRE(p.B > 0 && p.B <= 65535 && p.T > 0, SVSK_E_ARG, "diffnet_step_bf16: bad B/T");
  SVSK_REQUIRE(((uintptr_t)p.skip32 % 16) == 0 && ((uintptr_t)p.x32s % 16) == 0 && ((uintptr_t)p.z % 16) == 0 &&
                   ((uintptr_t)p.b_out % 16) == 0 && (p.eps_out == nullptr || ((uintptr_t)p.eps_out % 16) == 0),
               SVSK_E_ALIGN, "diffnet_step_bf16: skip32 / x32s / z / eps_out / b_out must be 16-byte aligned");
  int rc = require_sm100();
  if (rc) return rc;

  const int CB = p.C / 64, MB = (p.Mp + 63) / 64, ws_tile = p.C * 128;
  const int ws_bytes = CB * ws_tile > CB * kStepTile + MB * ws_tile ? CB * ws_tile : CB * kStepTile + MB * ws_tile;
  const int smem_bytes = CB * kStepTile + ws_bytes + (int)sizeof(DiffnetStepBarriers) + 1024;
  CUtensorMap tm_wskip, tm_wout, tm_win, tm_xout;
  {
    uint64_t dims[2] = {(uint64_t)p.C, (uint64_t)p.C};
    uint64_t str[1] = {(uint64_t)p.C * 2};
    uint32_t box[2] = {64, (uint32_t)p.C};
    if ((rc = make_tmap_bf16(&tm_wskip, p.w_skip, 2, dims, str, box))) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)p.C, (uint64_t)p.Mp};
    uint64_t str[1] = {(uint64_t)p.C * 2};
    uint32_t box[2] = {64, (uint32_t)p.Mp};
    if ((rc = make_tmap_bf16(&tm_wout, p.w_out, 2, dims, str, box))) return rc;
  }
  if (p.xb_out) {
    uint64_t dims[2] = {(uint64_t)p.Mp, (uint64_t)p.C};
    uint64_t str[1] = {(uint64_t)p.Mp * 2};
    uint32_t box[2] = {64, (uint32_t)p.C};
    if ((rc = make_tmap_bf16(&tm_win, p.w_in, 2, dims, str, box))) return rc;
    uint64_t dims3[3] = {(uint64_t)p.C, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str3[2] = {(uint64_t)p.C * 2, (uint64_t)p.T * p.C * 2};
    uint32_t box3[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_xout, p.xb_out, 3, dims3, str3, box3))) return rc;
  } else {
    tm_win = tm_wout;   // never dereferenced
    tm_xout = tm_wout;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(diffnet_step_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(diffnet_step_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return fail((int)e, "diffnet_step_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  DiffnetStepArgs a;
  a.skip32 = p.skip32; a.x32s = p.x32s; a.z = p.z; a.eps_out = p.eps_out;
  a.b_skip = p.b_skip; a.b_out = p.b_out; a.b_in = p.b_in;
  a.t = (const long long*)p.t;
  a.sra = p.sqrt_recip_alphas_cumprod; a.srm1 = p.sqrt_recipm1_alphas_cumprod;
  a.c1 = p.posterior_mean_coef1; a.c2 = p.posterior_mean_coef2; a.plv = p.posterior_log_variance_clipped;
  a.skip_scale = p.skip_scale;
  a.B = p.B; a.T = p.T; a.C = p.C; a.Mp = p.Mp; a.clip = p.clip_denoised; a.head = p.xb_out ? 1 : 0;
  if (p.C == 128)
    diffnet_step_kernel<128><<<dim3(ceil_div(p.T, 128), p.B), kStepThreads, smem_bytes, as_stream(stream)>>>(tm_wskip, tm_wout, tm_win,
                                                                                                              tm_xout, a);
  else
    diffnet_step_kernel<256><<<dim3(ceil_div(p.T, 128), p.B), kStepThreads, smem_bytes, as_stream(stream)>>>(tm_wskip, tm_wout, tm_win,
                                                                                                              tm_xout, a);
  return check_launch("diffnet_step_bf16");
}
