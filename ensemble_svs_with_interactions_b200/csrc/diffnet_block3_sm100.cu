// Fused DiffNet residual block, CTA-pair version with a RESIDENT activation window: replaces ResidualBlock.forward
// (nnsvs/diffsinger/denoiser.py:54-66) with one launch per layer.  Same maths, orientation and epilogues as
// diffnet_block2_sm100.cu (time = MMA M, 256 frames per CTA pair, output channels = N, N-block-outer GEMM1); what
// changed is how the A operand reaches the tensor cores.
//
// Measured on v2 (profiles/r01n_timeline_v2_accounting.log): the MMA thread spends half of GEMM1 waiting for ring
// stages, the producer is always out of free slots — every CTA streams 1.25 MB through a 4 x 32 KB ring, 40 B/cycle/SM
// on 96 SMs = 62 % of the L2 slice throughput, and 0.5 MB of that is the activations, read once per tap and once more
// for the second 256-channel block.
//
// v3: the three conv taps are the SAME rows of x at row offsets -d / 0 / +d.  A K-major SWIZZLE_128B operand descriptor
// may start at any 128-byte row (the swizzle is a function of the shared-memory address, probed by
// tools/ubench_rowshift.py), so ONE window tile of 128 + 2*8 rows per 64-channel block serves all taps and both output
// blocks, stays resident for the whole kernel, and is also the "old x" the residual epilogue updates in place.  The
// conditioner tiles are loaded once into the buffer that later holds G (G is first written after the first output block
// is complete, long after the conditioner k-blocks, which run FIRST and feed both output blocks).  The ring therefore
// carries nothing but 16 KB weight tiles, one per k-block, all of them parameters: the first ring fill is in flight
// before griddepcontrol.wait returns.  0.78 MB per CTA instead of 1.28 MB.
//
// Ring entry order (producer, MMA issuer and the peer's forwarder all walk it):
//   A: for hb < H/64, block j:  W1[block j][k = 3C + 64 hb]   (A operand = conditioner tile hb)
//   B: for block j:     W1[block j][k-block kb], kb < 3C/64   (A operand = window tile kb % CB at row 8 + (kb/CB - 1) d)
//   C: for block j:     Wout[block j][kb], kb < C/64          (A operand = G tile kb)
// Warps: 0 = TMA producer (both CTAs), 1 = MMA issuer (leader CTA) / forwarder (peer) + TMEM alloc, 2..9 = epilogue.
#include <cuda_bf16.h>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"
#include "tma_util.cuh"

namespace svsk {

constexpr int k3Tile = 128 * 128;            // 128 rows x 64 bf16
constexpr int k3Halo = 8;                    // window rows either side of the tile: dilation <= 8
constexpr int k3WinRows = 128 + 2 * k3Halo;
constexpr int k3WinBytes = k3WinRows * 128;  // 18 KB, a multiple of the 1024-byte swizzle atom
constexpr int k3MaxEntries = 8;
constexpr int k3SmemLimit = 232448;
constexpr int k3TmemCols = 512;
constexpr int k3Threads = 320;

struct Diffnet3Args {
  float* skip32;
  const float* stepbias;
  const float* bout;
  int B, T, C, H, dilation, sb_stride, init_skip, write_x, nentries;
};

struct __align__(8) Diffnet3Barriers {
  uint64_t full[k3MaxEntries];  // ring entry landed: own TMA bytes, and on the leader also the peer's (forwarded) arrival
  uint64_t empty[k3MaxEntries];
  uint64_t xw_full;             // window tiles landed (leader: in both CTAs)
  uint64_t cd_full[8];          // conditioner tile hb landed (leader: in both CTAs)
  uint64_t d1_full[2];
  uint64_t d2_full[2];
  uint64_t g_ready;
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(k3Threads, 1)
diffnet_block3_kernel(const __grid_constant__ CUtensorMap tm_xw, const __grid_constant__ CUtensorMap tm_cond,
                      const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_wout,
                      const __grid_constant__ CUtensorMap tm_xout, const __grid_constant__ CUtensorMap tm_skip,
                      const Diffnet3Args a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const int C = a.C, H = a.H, T = a.T;
  const int CB = C / 64, HB = H / 64;
  const int KB2 = CB;
  const int NB = (2 * C) / 256;  // 256-column output blocks of either GEMM
  const int twoC = 2 * C;
  uint8_t* xw_smem = smem;                                // CB window tiles
  uint8_t* g_smem = xw_smem + CB * k3WinBytes;            // max(HB, KB2) tiles: conditioner tiles, then G (A operand of GEMM2)
  uint8_t* ring = g_smem + max(HB, KB2) * k3Tile;         // nentries x 16 KB
  float* sb_full = reinterpret_cast<float*>(ring + a.nentries * k3Tile);
  float* sb_l = sb_full + twoC;
  float* sb_r = sb_l + twoC;
  float* bo_s = sb_r + twoC;
  Diffnet3Barriers* bars = reinterpret_cast<Diffnet3Barriers*>(bo_s + twoC);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int b = blockIdx.y;
  const int t_cta0 = (blockIdx.x >> 1) * 256 + (int)rank * 128;  // first frame of this CTA's 128 TMEM lanes
  const int w_row0 = (int)rank * 128;                             // this CTA's half of a 256-row weight block

  const int n_a = HB * NB;                       // phase-A ring entries
  const int n_total = n_a + NB * 3 * CB + NB * KB2;
  int pre_issued = 0;                            // producer: entries issued before the CTA-wide sync

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_xw);
    ptx::prefetch_tmap(&tm_cond);
    ptx::prefetch_tmap(&tm_w1);
    ptx::prefetch_tmap(&tm_wout);
    ptx::prefetch_tmap(&tm_xout);
    ptx::prefetch_tmap(&tm_skip);
    for (int i = 0; i < a.nentries; ++i) {
      ptx::mbar_init(&bars->full[i], rank == 0 ? 2 : 1);  // own producer's arrive.expect_tx (+ the peer's remote arrive)
      ptx::mbar_init(&bars->empty[i], 1);                 // one multicast tcgen05.commit
    }
    ptx::mbar_init(&bars->xw_full, rank == 0 ? 2 : 1);
    for (int i = 0; i < HB; ++i) ptx::mbar_init(&bars->cd_full[i], rank == 0 ? 2 : 1);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->d1_full[i], 1);
      ptx::mbar_init(&bars->d2_full[i], 1);
    }
    ptx::mbar_init(&bars->g_ready, 2 * 256);  // every epilogue thread of both CTAs
    ptx::fence_mbar_init();
    // The ring only ever holds weight tiles (parameters): the first fill is issued before waiting for the previous
    // kernel (contract in svsk.h: packed weights are not written by the kernel launched immediately before this one).
    pre_issued = min(a.nentries, n_total);
    for (int e = 0; e < pre_issued; ++e) {
      ptx::mbar_arrive_expect_tx(&bars->full[e], k3Tile);
      int kcol, wrow;
      const CUtensorMap* tm = &tm_w1;
      if (e < n_a) { kcol = 3 * CB + e / NB; wrow = e % NB; }
      else if (e < n_a + NB * 3 * CB) { const int i = e - n_a; kcol = i % (3 * CB); wrow = i / (3 * CB); }
      else { const int i = e - n_a - NB * 3 * CB; kcol = i % KB2; wrow = i / KB2; tm = &tm_wout; }
      ptx::tma_load_2d(ring + e * k3Tile, tm, &bars->full[e], kcol * 64, wrow * 256 + w_row0);
    }
    // Programmatic dependent launch: activations (conditioner tiles, then x = the previous layer's output) from here.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    for (int hb = 0; hb < HB; ++hb) {
      ptx::mbar_arrive_expect_tx(&bars->cd_full[hb], k3Tile);
      ptx::tma_load_3d(g_smem + hb * k3Tile, &tm_cond, &bars->cd_full[hb], hb * 64, t_cta0, b);
    }
    ptx::mbar_arrive_expect_tx(&bars->xw_full, CB * k3WinBytes);
    for (int cb = 0; cb < CB; ++cb)
      ptx::tma_load_3d(xw_smem + cb * k3WinBytes, &tm_xw, &bars->xw_full, cb * 64, t_cta0 - k3Halo, b);
  }
  if (warp == 1) {
    ptx::tmem_alloc2(&bars->tmem_base, k3TmemCols);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t tmem = bars->tmem_base;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    if (lane == 0) {
      int s = pre_issued % a.nentries;
      uint32_t ph = (pre_issued == a.nentries) ? 1u : 0u;
      for (int e = pre_issued; e < n_total; ++e) {
        ptx::mbar_wait(&bars->empty[s], ph ^ 1);
        uint8_t* dst = ring + s * k3Tile;
        ptx::mbar_arrive_expect_tx(&bars->full[s], k3Tile);
        if (e < n_a) {
          ptx::tma_load_2d(dst, &tm_w1, &bars->full[s], (3 * CB + e / NB) * 64, (e % NB) * 256 + w_row0);
        } else if (e < n_a + NB * 3 * CB) {
          const int i = e - n_a, j = i / (3 * CB), kb = i - j * 3 * CB;
          ptx::tma_load_2d(dst, &tm_w1, &bars->full[s], kb * 64, j * 256 + w_row0);
        } else {
          const int i = e - n_a - NB * 3 * CB, j = i / KB2, kb = i - j * KB2;
          ptx::tma_load_2d(dst, &tm_wout, &bars->full[s], kb * 64, j * 256 + w_row0);
        }
        if (++s == a.nentries) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer: one thread of the leader CTA
    if (rank == 0 && lane == 0) {
      const uint32_t idesc = ptx::umma_idesc_bf16_f32(256, 256);
      const uint32_t ring_lo = ptx::umma_desc_lo(ptx::smem_u32(ring)), g_lo = ptx::umma_desc_lo(ptx::smem_u32(g_smem));
      const uint32_t xw_lo = ptx::umma_desc_lo(ptx::smem_u32(xw_smem));
      int s = 0;
      uint32_t ph = 0;
      bool ready = false;  // the barrier of ring entry (s, ph) was already seen complete by the previous group's probe
      // An mbarrier wait whose result is needed at once stalls this thread ~160 cycles even on a long-completed phase
      // (tools/ubench_umma.py): every MMA group therefore probes the NEXT entry's barrier while its MMAs are issued.
#define SVSK_WAIT_ENTRY()                       \
  do {                                          \
    if (!ready) ptx::mbar_wait(&bars->full[s], ph); \
    ready = false;                              \
    ptx::tc_fence_after();                      \
  } while (0)
#define SVSK_NEXT_ENTRY() do { if (++s == a.nentries) { s = 0; ph ^= 1; } } while (0)
#define SVSK_ISSUE4(dcol, alo, blo, acc0)                                                                          \
  do {                                                                                                             \
    const int sn = (s + 1 == a.nentries) ? 0 : s + 1;                                                              \
    ready = ptx::umma2_bf16_x4_probe(tmem + (dcol), alo, blo, idesc, acc0, 4, &bars->full[sn], sn ? ph : ph ^ 1); \
  } while (0)
      // ---- phase A: conditioner k-blocks out of the (future) G buffer, both output blocks per tile
      for (int hb = 0; hb < HB; ++hb) {
        ptx::mbar_wait(&bars->cd_full[hb], 0);
        const uint32_t a_lo = g_lo + hb * (k3Tile >> 4);
        for (int j = 0; j < NB; ++j) {
          SVSK_WAIT_ENTRY();
          SVSK_ISSUE4(j * 256, a_lo, ring_lo + s * (k3Tile >> 4), hb != 0);
          ptx::umma_commit2_mc(&bars->empty[s], 3);
          SVSK_NEXT_ENTRY();
        }
      }
      // ---- phase B: the three taps out of the resident window
      ptx::mbar_wait(&bars->xw_full, 0);
      ptx::tc_fence_after();
      for (int j = 0; j < NB; ++j) {
        for (int jt = 0; jt < 3; ++jt) {
          const uint32_t row_lo = xw_lo + (uint32_t)(k3Halo + (jt - 1) * a.dilation) * (128u >> 4);
          for (int cb = 0; cb < CB; ++cb) {
            SVSK_WAIT_ENTRY();
            SVSK_ISSUE4(j * 256, row_lo + cb * (k3WinBytes >> 4), ring_lo + s * (k3Tile >> 4), 1);
            ptx::umma_commit2_mc(&bars->empty[s], 3);
            SVSK_NEXT_ENTRY();
          }
        }
        ptx::umma_commit2_mc(&bars->d1_full[j], 3);
      }
      // ---- phase C: GEMM2
      ptx::mbar_wait(&bars->g_ready, 0);
      ptx::tc_fence_after();
      for (int j = 0; j < NB; ++j) {
        for (int kb = 0; kb < KB2; ++kb) {
          SVSK_WAIT_ENTRY();
          SVSK_ISSUE4(j * 256, g_lo + kb * (k3Tile >> 4), ring_lo + s * (k3Tile >> 4), kb != 0);
          ptx::umma_commit2_mc(&bars->empty[s], 3);
          SVSK_NEXT_ENTRY();
        }
        ptx::umma_commit2_mc(&bars->d2_full[j], 3);
      }
#undef SVSK_WAIT_ENTRY
#undef SVSK_NEXT_ENTRY
#undef SVSK_ISSUE4
    } else if (rank == 1 && lane == 0) {
      // peer CTA: second arrival on the leader's barriers ("my ring entry / window has landed"), in the leader's order
      int s = 0;
      uint32_t ph = 0;
      for (int e = 0; e < n_total; ++e) {
        if (e < n_a && e % NB == 0) {
          ptx::mbar_wait(&bars->cd_full[e / NB], 0);
          ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->cd_full[e / NB]), 0));
        }
        if (e == n_a) {
          ptx::mbar_wait(&bars->xw_full, 0);
          ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->xw_full), 0));
        }
        ptx::mbar_wait(&bars->full[s], ph);
        ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->full[s]), 0));
        if (++s == a.nentries) { s = 0; ph ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (thread = one frame)
    const int q = warp & 3;           // TMEM lane quarter this warp may read
    const int sub = (warp - 2) >> 2;  // the two warps of a quarter alternate 16-column chunks
    const int row = q * 32 + lane;
    const int t = t_cta0 + row;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    const bool has_l = (t - a.dilation) >= 0, has_r = (t + a.dilation) < T;
    const bool warp_edge = __any_sync(0xffffffffu, !has_l || !has_r);  // warp-uniform: the bias correction is a branch

    // per-column biases -> smem (off the path to the first MMA): sb_full = centre + left + right tap terms, what an
    // interior frame gets.  The step-bias rows may come from the preceding kernel: wait for it first.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    {
      const float* sb = a.stepbias + (size_t)b * a.sb_stride;
      for (int i = threadIdx.x - 64; i < twoC; i += 256) {
        const float l = sb[i], c = sb[twoC + i], r = sb[2 * twoC + i];
        sb_full[i] = c + l + r;
        sb_l[i] = l;
        sb_r[i] = r;
        bo_s[i] = a.bout[i];
      }
      ptx::named_bar_sync(1, 256);
    }

    // ---- epilogue 1: gating -> G
    for (int j = 0; j < NB; ++j) {
      ptx::mbar_wait(&bars->d1_full[j], 0);
      ptx::tc_fence_after();
      uint32_t rgb[2][16], rfb[2][16];
      ptx::tmem_ld16(tmem + tlane + j * 256 + 16 * sub, rgb[0]);
      ptx::tmem_ld16(tmem + tlane + j * 256 + 128 + 16 * sub, rfb[0]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int c0 = 16 * (2 * i + sub);
        ptx::tmem_ld_wait();
        if (i + 1 < 4) {  // next chunk's TMEM loads fly while this chunk is gated
          ptx::tmem_ld16(tmem + tlane + j * 256 + c0 + 32, rgb[(i + 1) & 1]);
          ptx::tmem_ld16(tmem + tlane + j * 256 + 128 + c0 + 32, rfb[(i + 1) & 1]);
        }
        const uint32_t* rg = rgb[i & 1];
        const uint32_t* rf = rfb[i & 1];
        const int pg = j * 256 + c0, pf = pg + 128;
        uint64_t gv[8], fv[8];  // column pairs (FADD2 / FMUL2 / FFMA2), see diffnet_stack_sm100.cu
#pragma unroll
        for (int e = 0; e < 16; e += 4) {
          const float4 bg = ptx::ld_shared_v4f(sb_full + pg + e);
          const float4 bf = ptx::ld_shared_v4f(sb_full + pf + e);
          gv[e >> 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rg[e]), __uint_as_float(rg[e + 1])), ptx::f2_pack(bg.x, bg.y));
          gv[(e >> 1) + 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rg[e + 2]), __uint_as_float(rg[e + 3])), ptx::f2_pack(bg.z, bg.w));
          fv[e >> 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rf[e]), __uint_as_float(rf[e + 1])), ptx::f2_pack(bf.x, bf.y));
          fv[(e >> 1) + 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rf[e + 2]), __uint_as_float(rf[e + 3])), ptx::f2_pack(bf.z, bf.w));
        }
        if (warp_edge) {  // a branch around the rare case, not 128 predicated-off instructions per chunk (see diffnet_stack_sm100.cu)
          if (!has_l) {
#pragma unroll
            for (int u = 0; u < 16; u += 2) {
              gv[u >> 1] = ptx::f2_add(gv[u >> 1], ptx::f2_pack(-sb_l[pg + u], -sb_l[pg + u + 1]));
              fv[u >> 1] = ptx::f2_add(fv[u >> 1], ptx::f2_pack(-sb_l[pf + u], -sb_l[pf + u + 1]));
            }
          }
          if (!has_r) {
#pragma unroll
            for (int u = 0; u < 16; u += 2) {
              gv[u >> 1] = ptx::f2_add(gv[u >> 1], ptx::f2_pack(-sb_r[pg + u], -sb_r[pg + u + 1]));
              fv[u >> 1] = ptx::f2_add(fv[u >> 1], ptx::f2_pack(-sb_r[pf + u], -sb_r[pf + u + 1]));
            }
          }
        }
        float z[16];
#pragma unroll
        for (int u = 0; u < 16; u += 2) ptx::f2_unpack(ptx::f2_gate(gv[u >> 1], fv[u >> 1]), z[u], z[u + 1]);
        const int kc0 = j * 128 + c0;  // first gated channel of the chunk = K index of GEMM2
        uint8_t* gk = g_smem + (kc0 >> 6) * k3Tile;
        const uint32_t ch16 = (uint32_t)((kc0 & 63) >> 3);
        ptx::st_shared_v4(gk + ptx::sw128_offset((uint32_t)row, ch16), ptx::pack_bf16(z[0], z[1]),
                          ptx::pack_bf16(z[2], z[3]), ptx::pack_bf16(z[4], z[5]), ptx::pack_bf16(z[6], z[7]));
        ptx::st_shared_v4(gk + ptx::sw128_offset((uint32_t)row, ch16 + 1), ptx::pack_bf16(z[8], z[9]),
                          ptx::pack_bf16(z[10], z[11]), ptx::pack_bf16(z[12], z[13]), ptx::pack_bf16(z[14], z[15]));
      }
    }
    ptx::tc_fence_before();
    ptx::fence_proxy_async_smem();  // G (generic-proxy stores) -> visible to the tensor cores' async proxy
    if (rank == 0) ptx::mbar_arrive(&bars->g_ready);
    else ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->g_ready), 0));

    // ---- epilogue 2: residual -> in place over the window's centre rows -> TMA store ; skip -> fp32 slabs -> TMA
    //      reduce-add (or plain store on the first layer)
    const bool elected = (warp == 2 && lane == 0);
    const float s2 = 0.70710678118654752f;
    int skip_slab = 0;  // running index of 32-column skip slabs of this CTA
    for (int j = 0; j < NB; ++j) {
      ptx::mbar_wait(&bars->d2_full[j], 0);
      ptx::tc_fence_after();
      const int res_cols = min(max(C - j * 256, 0), 256);  // residual columns in this 256-column block
      if (res_cols > 0 && a.write_x) {
        ptx::mbar_wait(&bars->xw_full, 0);  // (long since complete) makes the TMA-written window visible to this thread
#pragma unroll 1
        for (int i = 0; i < res_cols / 32; ++i) {
          const int c0 = 16 * (2 * i + sub);
          const int oc0 = j * 256 + c0;  // output channel = residual channel
          uint32_t r[16];
          ptx::tmem_ld16(tmem + tlane + j * 256 + c0, r);
          ptx::tmem_ld_wait();
          uint8_t* xt = xw_smem + (oc0 >> 6) * k3WinBytes + k3Halo * 128;  // centre rows of the window tile
          const uint32_t ch16 = (uint32_t)((oc0 & 63) >> 3);
          uint8_t* p0 = xt + ptx::sw128_offset((uint32_t)row, ch16);
          uint8_t* p1 = xt + ptx::sw128_offset((uint32_t)row, ch16 + 1);
          const uint4 xa = ptx::ld_shared_v4(p0), xb = ptx::ld_shared_v4(p1);
          const uint32_t xo[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
          uint32_t o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float lo = (ptx::bf16_lo(xo[e]) + __uint_as_float(r[2 * e]) + bo_s[oc0 + 2 * e]) * s2;
            const float hi = (ptx::bf16_hi(xo[e]) + __uint_as_float(r[2 * e + 1]) + bo_s[oc0 + 2 * e + 1]) * s2;
            o[e] = ptx::pack_bf16(lo, hi);
          }
          ptx::st_shared_v4(p0, o[0], o[1], o[2], o[3]);
          ptx::st_shared_v4(p1, o[4], o[5], o[6], o[7]);
        }
        ptx::fence_proxy_async_smem();
        ptx::named_bar_sync(1, 256);
        if (elected) {
          for (int cb = j * 4; cb < j * 4 + res_cols / 64; ++cb)
            ptx::tma_store_3d(&tm_xout, xw_smem + cb * k3WinBytes + k3Halo * 128, cb * 64, t_cta0, b);
          ptx::bulk_commit_group();
        }
      }
      // skip part: columns [res_cols, 256) of this block, 32 at a time (one 128-byte fp32 row per frame)
      if (res_cols < 256) {
        if (j != NB - 1) __trap();  // skip columns only live in the last block: all MMAs are done, ring + G are free
#pragma unroll 1
        for (int i = res_cols / 32; i < 8; i += 2, skip_slab += 2) {
          uint32_t r0[16], r1[16];
          ptx::tmem_ld16(tmem + tlane + j * 256 + 16 * (2 * i + sub), r0);
          ptx::tmem_ld16(tmem + tlane + j * 256 + 16 * (2 * i + 2 + sub), r1);
          ptx::tmem_ld_wait();
          uint8_t* slab[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {  // slab buffers: the ring entries first, then 16 KB pieces of G
            const int n = skip_slab + u;
            slab[u] = (n < a.nentries) ? ring + n * k3Tile : g_smem + (n - a.nentries) * k3Tile;
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const uint32_t* r = u ? r1 : r0;
            const int oc0 = j * 256 + 16 * (2 * (i + u) + sub);
#pragma unroll
            for (int e = 0; e < 16; e += 4) {
              const float4 bo = ptx::ld_shared_v4f(bo_s + oc0 + e);
              ptx::st_shared_v4f(slab[u] + ptx::sw128_offset((uint32_t)row, (uint32_t)(sub * 4 + (e >> 2))),
                                 __uint_as_float(r[e]) + bo.x, __uint_as_float(r[e + 1]) + bo.y,
                                 __uint_as_float(r[e + 2]) + bo.z, __uint_as_float(r[e + 3]) + bo.w);
            }
          }
          ptx::fence_proxy_async_smem();
          ptx::named_bar_sync(1, 256);
          if (elected) {
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int ch0 = j * 256 + 32 * (i + u) - C;  // first skip channel of the slab
              if (a.init_skip) ptx::tma_store_3d(&tm_skip, slab[u], ch0, t_cta0, b);
              else ptx::tma_reduce_add_3d(&tm_skip, slab[u], ch0, t_cta0, b);
            }
            ptx::bulk_commit_group();
          }
        }
      }
    }
    if (elected) ptx::bulk_wait_read_all();  // smem may be released; global visibility comes with grid completion
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();  // the peer's smem / TMEM are in use by the leader's MMAs until here
  if (warp == 1) ptx::tmem_dealloc2(tmem, k3TmemCols);
}

}  // namespace svsk

using namespace svsk;

extern "C" int svsk_diffnet_block3_bf16(const svsk_diffnet_block_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "diffnet_block3_bf16: null params");
  const svsk_diffnet_block_params& p = *pp;
  SVSK_REQUIRE(p.xb_in && p.xb_out && p.skip32 && p.cond && p.w1p && p.woutp && p.stepbias && p.bout, SVSK_E_ARG,
               "diffnet_block3_bf16: null tensor");
  SVSK_REQUIRE(p.xb_in != p.xb_out, SVSK_E_ARG, "diffnet_block3_bf16: xb_in and xb_out must differ (halo reads)");
  SVSK_REQUIRE(p.C == 128 || p.C == 256, SVSK_E_ARG, "diffnet_block3_bf16: C=%d (need 128 or 256)", p.C);
  SVSK_REQUIRE(p.H > 0 && p.H % 64 == 0, SVSK_E_ARG, "diffnet_block3_bf16: H=%d (need a multiple of 64)", p.H);
  SVSK_REQUIRE(p.B > 0 && p.B <= 65535 && p.T > 0, SVSK_E_ARG, "diffnet_block3_bf16: bad B/T");
  SVSK_REQUIRE(p.dilation >= 1 && p.dilation <= k3Halo, SVSK_E_ARG,
               "diffnet_block3_bf16: dilation %d outside the resident window (1..%d); use svsk_diffnet_block2_bf16",
               p.dilation, k3Halo);
  SVSK_REQUIRE(p.stepbias_batch_stride == 0 || p.stepbias_batch_stride >= 6 * p.C, SVSK_E_ARG,
               "diffnet_block3_bf16: stepbias stride %d", p.stepbias_batch_stride);
  SVSK_REQUIRE(((uintptr_t)p.skip32 % 16) == 0 && ((uintptr_t)p.xb_out % 16) == 0, SVSK_E_ALIGN,
               "diffnet_block3_bf16: skip32 / xb_out must be 16-byte aligned");
  int rc = require_sm100();
  if (rc) return rc;

  const int CB = p.C / 64, HB = p.H / 64;
  SVSK_REQUIRE(HB <= 8, SVSK_E_ARG, "diffnet_block3_bf16: H=%d (at most 512)", p.H);
  const int gc_tiles = HB > CB ? HB : CB;  // conditioner tiles first, G afterwards
  const int fixed = CB * k3WinBytes + gc_tiles * k3Tile + 4 * 2 * p.C * (int)sizeof(float) + (int)sizeof(Diffnet3Barriers) + 1024;
  int nentries = (k3SmemLimit - fixed) / k3Tile;
  if (nentries > k3MaxEntries) nentries = k3MaxEntries;
  // skip slabs are staged in the ring entries and in G: 32 fp32 columns each
  SVSK_REQUIRE(nentries >= 3 && nentries + CB >= p.C / 32, SVSK_E_ARG, "diffnet_block3_bf16: not enough shared memory");
  const int smem_bytes = nentries * k3Tile + fixed;

  CUtensorMap tm_xw, tm_cond, tm_w1, tm_wout, tm_xout, tm_skip;
  {
    uint64_t dims[3] = {(uint64_t)p.C, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.C * 2, (uint64_t)p.T * p.C * 2};
    uint32_t boxw[3] = {64, (uint32_t)k3WinRows, 1};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_xw, p.xb_in, 3, dims, str, boxw))) return rc;
    if ((rc = make_tmap_bf16(&tm_xout, p.xb_out, 3, dims, str, box))) return rc;
    uint64_t str4[2] = {(uint64_t)p.C * 4, (uint64_t)p.T * p.C * 4};
    uint32_t box4[3] = {32, 128, 1};
    if ((rc = make_tmap_f32(&tm_skip, p.skip32, 3, dims, str4, box4))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)p.H, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.H * 2, (uint64_t)p.T * p.H * 2};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_cond, p.cond, 3, dims, str, box))) return rc;
  }
  {
    const uint64_t K1 = 3 * (uint64_t)p.C + p.H;
    uint64_t dims[2] = {K1, (uint64_t)2 * p.C};
    uint64_t str[1] = {K1 * 2};
    uint32_t box[2] = {64, 128};
    if ((rc = make_tmap_bf16(&tm_w1, p.w1p, 2, dims, str, box))) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)p.C, (uint64_t)2 * p.C};
    uint64_t str[1] = {(uint64_t)p.C * 2};
    uint32_t box[2] = {64, 128};
    if ((rc = make_tmap_bf16(&tm_wout, p.woutp, 2, dims, str, box))) return rc;
  }

  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(diffnet_block3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, k3SmemLimit);
    if (e != cudaSuccess) return fail((int)e, "diffnet_block3_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  Diffnet3Args a;
  a.skip32 = p.skip32;
  a.stepbias = p.stepbias;
  a.bout = p.bout;
  a.B = p.B; a.T = p.T; a.C = p.C; a.H = p.H;
  a.dilation = p.dilation;
  a.sb_stride = p.stepbias_batch_stride;
  a.init_skip = p.init_skip;
  a.write_x = p.write_x;
  a.nentries = nentries;

  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * ceil_div(p.T, 256), p.B);
  cfg.blockDim = dim3(k3Threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = as_stream(stream);
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaError_t e = cudaLaunchKernelEx(&cfg, diffnet_block3_kernel, tm_xw, tm_cond, tm_w1, tm_wout, tm_xout, tm_skip, a);
  if (e != cudaSuccess) return fail((int)e, "diffnet_block3_bf16: launch: %s", cudaGetErrorString(e));
  return check_launch("diffnet_block3_bf16");
}
