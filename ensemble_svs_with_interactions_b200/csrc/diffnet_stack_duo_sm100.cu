// The DiffNet residual stack at C = 128 (the multi-track recipe's bap denoiser: 10 blocks x 128 channels) with TWO
// 256-frame tiles per CTA pair — the variant svsk_diffnet_stack_bf16 runs for C = 128, H <= 128.  Same arithmetic, operand
// layouts, tap descriptors and epilogues as diffnet_stack_sm100.cu (nnsvs/diffsinger/denoiser.py:54-66, 114-118).
//
// Why: at C = 128 a layer of one tile is a serial chain — GEMM1 (4.1 k cycles of MMAs) -> gating (4.7 k) -> GEMM2 (1 k)
// -> residual epilogue (2.1 k) -> neighbour exchange -> next layer's GEMM1 — of 16.4 k cycles (halo rows through
// distributed shared memory) or 21 k (through global memory: tracks beyond 2048 frames, what the pipeline's 6 x 6000
// batches run) for 5.3 k cycles of tensor-pipe work (profiles/r02j_stack_c128_timeline.log): 0.29 of the tensor roofline.
// The chain cannot be shortened much (the gate needs the whole accumulator row, the next layer needs the residual), but
// at C = 128 a tile only needs half of TMEM and 68 KB of shared memory, so a CTA pair can carry two INDEPENDENT chains:
// slot u = 0, 1 holds its own activation window, G buffer, 256 TMEM columns, barriers, four epilogue warps and
// activation-producer warp; one thread issues the MMAs of both slots in the fixed order GEMM1(0) GEMM1(1) GEMM2(0) GEMM2(1)
// per layer, so one slot's gating / residual epilogue / halo round trip runs under the other slot's MMAs.  The weight ring
// is shared (each slot streams its own copy of a layer's tiles, in the order the MMA thread consumes them).  A 6 x 6000
// batch is 144 virtual pairs = 72 CTA pairs: ONE launch instead of two.
//
// Halo rows always travel through global memory + per-tile layer counters here (any track length); the two slots of a
// pair are virtual pairs half a track apart.  All CTAs must be co-resident (cooperative launch), as in the C = 256
// kernel's global-memory mode.
//
// Warps: 0 = weight producer, 1 = MMA issuer (leader CTA) / forwarder (peer) + TMEM owner, then 4 kDW epilogue warps per
// slot (thread = one frame, kDW warps per TMEM lane quarter alternating 16-column chunks), the last two = activation
// producer of slot 0 / 1.
#include <cuda_bf16.h>
#include <cstdlib>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"
#include "tma_util.cuh"

namespace svsk {

constexpr int kDTile = 128 * 128;            // 128 rows x 64 bf16
constexpr int kDHalo = 8;
constexpr int kDWinRows = 128 + 2 * kDHalo;
constexpr int kDWinBytes = kDWinRows * 128;  // 18 KB per 64 channels
constexpr int kDHaloBytes = kDHalo * 128;
constexpr int kDC = 128, kDCB = 2, kDKB2 = 2, kDTwoC = 256;
constexpr int kDGTiles = 2;                  // G buffer of a slot: conditioner tiles, then G, then skip staging
constexpr int kDSlotBytes = kDCB * kDWinBytes + kDGTiles * kDTile;  // 68 KB
constexpr int kDMaxEntries = 6;
constexpr int kDW = 2;                       // epilogue warps per TMEM lane quarter and slot (they alternate 16-column chunks)
constexpr int kDEpi = 128 * kDW;             // epilogue threads per slot
constexpr int kDThreads = 64 + 2 * kDEpi + 64;
constexpr int kDSmemLimit = 232448;
constexpr int kDMaxLayers = 64;

struct DuoArgs {
  const float* stepbias;  // [batch][layer][6C] (strides below)
  const float* bout;      // [layer][2C]
  int* flags;             // [B * tiles_per_track] layers published per 128-frame tile; zero at launch
  int B, T, H, L, sb_batch_stride, sb_layer_stride, init_skip, nentries, tiles_per_track;
  int dilation[kDMaxLayers];
};

struct __align__(8) DuoSlotBarriers {
  uint64_t cd_full[2];   // conditioner tile hb of this layer landed (leader: in both CTAs)
  uint64_t xw_full;      // layer 0: whole window landed; later layers: halo rows landed (leader: in both CTAs)
  uint64_t xc_ready;     // leader: centre rows updated in place by every epilogue thread of both CTAs
  uint64_t xe_ready;     // this CTA's centre rows updated (-> activation producer publishes the edge rows)
  uint64_t d1_full, d2_full;
  uint64_t d2_drained;   // leader: every epilogue thread of both CTAs has read the accumulator out of TMEM
  uint64_t g_ready;      // leader: gating written to G by every epilogue thread of both CTAs
  uint64_t gc_free;      // this CTA's G buffer is free again (skip slabs read by the TMA unit)
};
struct __align__(8) DuoBarriers {
  uint64_t full[kDMaxEntries];
  uint64_t empty[kDMaxEntries];
  DuoSlotBarriers s[2];
  uint32_t tmem_base;
};

// weight tile i of a slot's GEMM1 (i < 3 CB + HB): centre taps first, then the side taps, then the conditioner k-blocks
__device__ __forceinline__ int duo_gemm1_kcol(int i) {
  if (i < kDCB) return kDCB + i;
  i -= kDCB;
  if (i < 2 * kDCB) return (i / kDCB) * 2 * kDCB + i % kDCB;
  return 3 * kDCB + (i - 2 * kDCB);
}

__device__ __forceinline__ int duo_ld_relaxed_gpu(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void duo_st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void duo_fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// kHB = H / 64 (1 or 2) is compile-time: the single-thread roles pay for every run-time loop bound and branch
// (diffnet_stack_sm100.cu, DESIGN §4 item 17).
template <int kHB>
__global__ void __launch_bounds__(kDThreads, 1)
diffnet_stack_duo_kernel(const __grid_constant__ CUtensorMap tm_xw0, const __grid_constant__ CUtensorMap tm_e0,
                         const __grid_constant__ CUtensorMap tm_e1, const __grid_constant__ CUtensorMap tm_cond,
                         const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_wout,
                         const __grid_constant__ CUtensorMap tm_skip, const DuoArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const int T = a.T, L = a.L;
  constexpr int HB = kHB;
  uint8_t* ring = smem + 2 * kDSlotBytes;
  float* bias_base = reinterpret_cast<float*>(ring + a.nentries * kDTile);  // per slot: sb_full | sb_l | sb_r | bo_s
  DuoBarriers* bars = reinterpret_cast<DuoBarriers*>(bias_base + 2 * 4 * kDTwoC);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank() & 1u;  // rank in the CTA pair (tcgen05 cta_group::2): 0 = leader
  const uint16_t pair_mask = 3u;
  const int b = blockIdx.y;
  const int pair = blockIdx.x >> 1;
  const int w_row0 = (int)rank * 128;  // this CTA's half of the 256-row weight block
  const int n_g1 = 3 * kDCB + HB;      // ring entries of one slot's GEMM1
  // Slot u works on the virtual pair vp = pair + u * (pairs per track): frames [vp * 256, vp * 256 + 256), this CTA its
  // half.  NOT 2 * pair + u: with adjacent slots, slot 0 waits every layer for the edge rows of slot 1 of its own pair,
  // whose MMAs are issued after its own — a circular coupling that made the layer period the sum of both slots' chains
  // (26.5 k cycles, profiles/r02n_stack_duo_timeline.log).  This way slot 0's neighbours are the slots 0 of the
  // neighbouring pairs (the same phase of the same schedule) and the two families only meet once per track.
  const int npairs = (int)(gridDim.x >> 1);
  const int vp0 = pair, vp1 = pair + npairs;
  const bool live1 = vp1 * 256 < T;  // (slot 0 is always live: the grid has ceil(n256 / 2) pairs per track)
  const int n_slots = live1 ? 2 : 1;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_xw0);
    ptx::prefetch_tmap(&tm_e0);
    ptx::prefetch_tmap(&tm_e1);
    ptx::prefetch_tmap(&tm_cond);
    ptx::prefetch_tmap(&tm_w1);
    ptx::prefetch_tmap(&tm_wout);
    ptx::prefetch_tmap(&tm_skip);
    const uint32_t two = rank == 0 ? 2u : 1u;           // leader barriers also count the peer's forwarded arrival
    const uint32_t all = rank == 0 ? 2u * kDEpi : 1u;   // leader barriers every epilogue thread of the slot (both CTAs) arrives on
    for (int i = 0; i < a.nentries; ++i) {
      ptx::mbar_init(&bars->full[i], two);
      ptx::mbar_init(&bars->empty[i], 1);
    }
    for (int u = 0; u < 2; ++u) {
      DuoSlotBarriers* sb = &bars->s[u];
      ptx::mbar_init(&sb->cd_full[0], two);
      ptx::mbar_init(&sb->cd_full[1], two);
      ptx::mbar_init(&sb->xw_full, two);
      ptx::mbar_init(&sb->xc_ready, all);
      ptx::mbar_init(&sb->xe_ready, kDEpi);
      ptx::mbar_init(&sb->d1_full, 1);
      ptx::mbar_init(&sb->d2_full, 1);
      ptx::mbar_init(&sb->d2_drained, all);
      ptx::mbar_init(&sb->g_ready, all);
      ptx::mbar_init(&sb->gc_free, 4 * kDW);  // one arrival per epilogue warp
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc2(&bars->tmem_base, 512);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp == 0) {
    // ------------------------------------------------------------------ weight producer (both CTAs)
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int l = 0; l < L; ++l) {
        for (int phase = 0; phase < 2; ++phase) {
          const int n_e = phase == 0 ? n_g1 : kDKB2;
          for (int u = 0; u < n_slots; ++u) {
            for (int i = 0; i < n_e; ++i) {
              ptx::mbar_wait(&bars->empty[s], ph ^ 1);
              ptx::mbar_arrive_expect_tx(&bars->full[s], kDTile);
              if (phase == 0) ptx::tma_load_3d(ring + s * kDTile, &tm_w1, &bars->full[s], duo_gemm1_kcol(i) * 64, w_row0, l);
              else ptx::tma_load_3d(ring + s * kDTile, &tm_wout, &bars->full[s], i * 64, w_row0, l);
              if (++s == a.nentries) { s = 0; ph ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp >= 2 + 8 * kDW) {
    // ------------------------------------------------------------------ activation producer of slot u (both CTAs)
    const int u = warp - (2 + 8 * kDW);
    if (lane == 0 && u < n_slots) {
      DuoSlotBarriers* sb = &bars->s[u];
      uint8_t* xw_smem = smem + u * kDSlotBytes;
      uint8_t* g_smem = xw_smem + kDCB * kDWinBytes;
      const int t_cta0 = (u ? vp1 : vp0) * 256 + (int)rank * 128;
      const int tile_idx = b * a.tiles_per_track + (t_cta0 >> 7);
      // (the peer's half of the last virtual pair may lie wholly past the end of the track: its stores are clipped, its
      // counter exists — tiles_per_track counts both halves — and nobody waits for it)
      const bool has_left = t_cta0 > 0, has_right = t_cta0 + 128 < T;
      // layer 0: conditioner tiles and the whole window of the stack's input
      for (int hb = 0; hb < HB; ++hb) {
        ptx::mbar_arrive_expect_tx(&sb->cd_full[hb], kDTile);
        ptx::tma_load_3d(g_smem + hb * kDTile, &tm_cond, &sb->cd_full[hb], hb * 64, t_cta0, b);
      }
      ptx::mbar_arrive_expect_tx(&sb->xw_full, kDCB * kDWinBytes);
      for (int cb = 0; cb < kDCB; ++cb)
        ptx::tma_load_3d(xw_smem + cb * kDWinBytes, &tm_xw0, &sb->xw_full, cb * 64, t_cta0 - kDHalo, b);
      for (int l = 1; l < L; ++l) {
        const uint32_t pp = (uint32_t)(l - 1) & 1u;
        const CUtensorMap* tm_e = pp ? &tm_e1 : &tm_e0;
        // publish the first / last 8 rows of layer l-1's output (the epilogue has written them in place)
        ptx::mbar_wait(&sb->xe_ready, pp);
        for (int cb = 0; cb < kDCB; ++cb) {
          uint8_t* centre = xw_smem + cb * kDWinBytes + kDHalo * 128;
          ptx::tma_store_3d(tm_e, centre, cb * 64, t_cta0, b);
          ptx::tma_store_3d(tm_e, centre + (128 - kDHalo) * 128, cb * 64, t_cta0 + 128 - kDHalo, b);
        }
        ptx::bulk_commit_group();
        ptx::bulk_wait_all();  // the stores are complete (not merely read out of shared memory)
        duo_fence_proxy_async_global();
        duo_st_release_gpu(a.flags + tile_idx, l);
        // halo rows of layer l's input: the neighbours' edge rows of layer l-1's output
        for (uint32_t spin = 0;; ++spin) {  // both flags per round trip, relaxed; one acquire fence at the end
          const int fl = has_left ? duo_ld_relaxed_gpu(a.flags + tile_idx - 1) : l;
          const int fr = has_right ? duo_ld_relaxed_gpu(a.flags + tile_idx + 1) : l;
          if (fl >= l && fr >= l) break;
          if (spin > (1u << 21)) __trap();
        }
        asm volatile("fence.acq_rel.gpu;" ::: "memory");
        duo_fence_proxy_async_global();
        // (Measured and not kept: fetching the 4 KB of halo rows with ld.global.cg by the whole warp + st.shared instead of
        // TMA, which saves the second fence — 141.8 vs 135.4 us per launch: an L2 round trip under this load is ~2 k cycles
        // whoever issues it.)
        ptx::mbar_arrive_expect_tx(&sb->xw_full, 2 * kDCB * kDHaloBytes);
        for (int cb = 0; cb < kDCB; ++cb) {
          uint8_t* tile = xw_smem + cb * kDWinBytes;
          ptx::tma_load_3d(tile, tm_e, &sb->xw_full, cb * 64, t_cta0 - kDHalo, b);
          ptx::tma_load_3d(tile + (kDHalo + 128) * 128, tm_e, &sb->xw_full, cb * 64, t_cta0 + 128, b);
        }
        // conditioner tiles of layer l, once the G buffer is free again
        ptx::mbar_wait(&sb->gc_free, pp);
        for (int hb = 0; hb < HB; ++hb) {
          ptx::mbar_arrive_expect_tx(&sb->cd_full[hb], kDTile);
          ptx::tma_load_3d(g_smem + hb * kDTile, &tm_cond, &sb->cd_full[hb], hb * 64, t_cta0, b);
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0 && lane == 0) {
      // ---------------------------------------------------------------- MMA issuer: one thread of the leader CTA
      const uint32_t idesc = ptx::umma_idesc_bf16_f32(256, 256);
      const uint32_t ring_lo = ptx::umma_desc_lo(ptx::smem_u32(ring));
      int s = 0;
      uint32_t ph = 0;
      bool ready = false;  // the barrier of ring entry (s, ph) was already seen complete by the previous group's probe
      // (an mbarrier wait whose result is needed at once stalls this thread ~160 cycles even on a long-completed phase:
      // every MMA group probes the NEXT entry's barrier while its MMAs are issued, tools/ubench_umma.py)
#define DUO_WAIT_ENTRY()                        \
  do {                                          \
    if (!ready) ptx::mbar_wait(&bars->full[s], ph); \
    ready = false;                              \
    ptx::tc_fence_after();                      \
  } while (0)
#define DUO_ISSUE4(tb, alo, acc0)                                                                                       \
  do {                                                                                                                  \
    const int sn = (s + 1 == a.nentries) ? 0 : s + 1;                                                                   \
    ready = ptx::umma2_bf16_x4_probe(tmem + (tb), alo, ring_lo + s * (kDTile >> 4), idesc, acc0, 4, &bars->full[sn],   \
                                     sn ? ph : ph ^ 1);                                                                 \
    ptx::umma_commit2_mc(&bars->empty[s], pair_mask);                                                                   \
    if (++s == a.nentries) { s = 0; ph ^= 1; }                                                                          \
  } while (0)
      for (int l = 0; l < L; ++l) {
        const uint32_t pl = (uint32_t)l & 1u, pp = pl ^ 1u;
        const int d = a.dilation[l];
        for (int u = 0; u < n_slots; ++u) {  // ---- GEMM1 of slot u
          DuoSlotBarriers* sb = &bars->s[u];
          const uint32_t xw_lo = ptx::umma_desc_lo(ptx::smem_u32(smem + u * kDSlotBytes));
          const uint32_t g_lo = ptx::umma_desc_lo(ptx::smem_u32(smem + u * kDSlotBytes + kDCB * kDWinBytes));
          const uint32_t tb = (uint32_t)u * 256u;
          if (l == 0) {
            ptx::mbar_wait(&sb->xw_full, 0);
          } else {
            ptx::mbar_wait(&sb->xc_ready, pp);    // centre rows rewritten in place by the previous layer's epilogue
            ptx::mbar_wait(&sb->d2_drained, pp);  // ... and the accumulator read out (residual and skip halves)
          }
          ptx::tc_fence_after();
          for (int cb = 0; cb < kDCB; ++cb) {
            DUO_WAIT_ENTRY();
            DUO_ISSUE4(tb, xw_lo + cb * (kDWinBytes >> 4) + kDHalo * 8, cb != 0);
          }
          if (l != 0) {  // halo rows of this layer
            ptx::mbar_wait(&sb->xw_full, pl);
            ptx::tc_fence_after();
          }
          for (int jt = 0; jt < 3; jt += 2) {
            const uint32_t row_lo = xw_lo + (uint32_t)(kDHalo + (jt - 1) * d) * 8u;
            for (int cb = 0; cb < kDCB; ++cb) {
              DUO_WAIT_ENTRY();
              DUO_ISSUE4(tb, row_lo + cb * (kDWinBytes >> 4), 1);
            }
          }
          for (int hb = 0; hb < HB; ++hb) {
            ptx::mbar_wait(&sb->cd_full[hb], pl);
            ptx::tc_fence_after();
            DUO_WAIT_ENTRY();
            DUO_ISSUE4(tb, g_lo + hb * (kDTile >> 4), 1);
          }
          ptx::umma_commit2_mc(&sb->d1_full, pair_mask);
        }
        for (int u = 0; u < n_slots; ++u) {  // ---- GEMM2 of slot u
          DuoSlotBarriers* sb = &bars->s[u];
          const uint32_t g_lo = ptx::umma_desc_lo(ptx::smem_u32(smem + u * kDSlotBytes + kDCB * kDWinBytes));
          const uint32_t tb = (uint32_t)u * 256u;
          ptx::mbar_wait(&sb->g_ready, pl);
          ptx::tc_fence_after();
          for (int kb = 0; kb < kDKB2; ++kb) {
            DUO_WAIT_ENTRY();
            DUO_ISSUE4(tb, g_lo + kb * (kDTile >> 4), kb != 0);
          }
          ptx::umma_commit2_mc(&sb->d2_full, pair_mask);
        }
      }
#undef DUO_WAIT_ENTRY
#undef DUO_ISSUE4
    } else if (rank == 1 && lane == 0) {
      // peer CTA: second arrival on the leader's barriers ("mine has landed too"), in the order the leader waits
      int s = 0;
      uint32_t ph = 0;
      const uint32_t leader_full0 = ptx::mapa(ptx::smem_u32(&bars->full[0]), 0);
      auto forward_entries = [&](int n) {
        for (int k = 0; k < n; ++k) {
          ptx::mbar_wait(&bars->full[s], ph);
          ptx::mbar_arrive_cluster(leader_full0 + (uint32_t)s * 8u);
          if (++s == a.nentries) { s = 0; ph ^= 1; }
        }
      };
      for (int l = 0; l < L; ++l) {
        const uint32_t pl = (uint32_t)l & 1u;
        for (int u = 0; u < n_slots; ++u) {
          DuoSlotBarriers* sb = &bars->s[u];
          auto forward_xw = [&]() {
            ptx::mbar_wait(&sb->xw_full, pl);
            ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&sb->xw_full), 0));
          };
          if (l == 0) forward_xw();
          forward_entries(kDCB);
          if (l != 0) forward_xw();
          forward_entries(2 * kDCB);
          for (int hb = 0; hb < HB; ++hb) {
            ptx::mbar_wait(&sb->cd_full[hb], pl);
            ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&sb->cd_full[hb]), 0));
            forward_entries(1);
          }
        }
        forward_entries(n_slots * kDKB2);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps of slot u (thread = one frame)
    const int u = (warp - 2) / (4 * kDW);
    const int sub = ((warp - 2) >> 2) % kDW;  // which of the quarter's kDW warps
    if (u < n_slots) {
      DuoSlotBarriers* sb = &bars->s[u];
      uint8_t* xw_smem = smem + u * kDSlotBytes;
      uint8_t* g_smem = xw_smem + kDCB * kDWinBytes;
      float* sb_full = bias_base + u * 4 * kDTwoC;
      float* sb_l = sb_full + kDTwoC;
      float* sb_r = sb_l + kDTwoC;
      float* bo_s = sb_r + kDTwoC;
      const int q = warp & 3;  // TMEM lane quarter this warp may read
      const int row = q * 32 + lane;
      const int et = (int)threadIdx.x - 64 - u * kDEpi;  // 0..127 within the slot's epilogue threads
      const int t_cta0 = (u ? vp1 : vp0) * 256 + (int)rank * 128;
      const int t = t_cta0 + row;
      const bool in_seq = t < T;
      const uint32_t tcol = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)u * 256u;
      const uint32_t xc_leader = ptx::mapa(ptx::smem_u32(&sb->xc_ready), 0);
      const uint32_t gr_leader = ptx::mapa(ptx::smem_u32(&sb->g_ready), 0);
      const uint32_t dr_leader = ptx::mapa(ptx::smem_u32(&sb->d2_drained), 0);
      const float s2 = 0.70710678118654752f;

      for (int l = 0; l < L; ++l) {
        const uint32_t pl = (uint32_t)l & 1u;
        const int d = a.dilation[l];
        const bool has_l = (t - d) >= 0, has_r = (t + d) < T;
        const bool warp_edge = __any_sync(0xffffffffu, !has_l || !has_r);  // warp-uniform: the bias correction is a branch
        const bool last = (l == L - 1);
        // per-column biases of this layer -> smem: sb_full = centre + left + right tap terms (an interior frame's sum)
        {
          const float* sbp = a.stepbias + (size_t)b * a.sb_batch_stride + (size_t)l * a.sb_layer_stride;
          const float* bo = a.bout + (size_t)l * kDTwoC;
          for (int i = et; i < kDTwoC; i += kDEpi) {
            const float lft = sbp[i], c = sbp[kDTwoC + i], r = sbp[2 * kDTwoC + i];
            sb_full[i] = c + lft + r;
            sb_l[i] = lft;
            sb_r[i] = r;
            bo_s[i] = bo[i];
          }
          ptx::named_bar_sync(1 + u, kDEpi);
        }

        // ---- epilogue 1: gating -> G  (accumulator columns [0,128) gate, [128,256) filter)
        ptx::mbar_wait(&sb->d1_full, pl);
        ptx::tc_fence_after();
        {
          uint32_t rgb[2][16], rfb[2][16];
          ptx::tmem_ld16(tcol + 16 * sub, rgb[0]);
          ptx::tmem_ld16(tcol + 128 + 16 * sub, rfb[0]);
#pragma unroll
          for (int i = 0; i < 8 / kDW; ++i) {
            const int c0 = 16 * (kDW * i + sub);
            ptx::tmem_ld_wait();
            if (i + 1 < 8 / kDW) {  // next chunk's TMEM loads fly while this chunk is gated
              ptx::tmem_ld16(tcol + c0 + 16 * kDW, rgb[(i + 1) & 1]);
              ptx::tmem_ld16(tcol + 128 + c0 + 16 * kDW, rfb[(i + 1) & 1]);
            }
            const uint32_t* rg = rgb[i & 1];
            const uint32_t* rf = rfb[i & 1];
            const int pg = c0, pf = c0 + 128;
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
            uint8_t* gk = g_smem + (c0 >> 6) * kDTile;  // gated channel c0.. = K index of GEMM2
            const uint32_t ch16 = (uint32_t)((c0 & 63) >> 3);
            ptx::st_shared_v4(gk + ptx::sw128_offset((uint32_t)row, ch16), ptx::pack_bf16(z[0], z[1]),
                              ptx::pack_bf16(z[2], z[3]), ptx::pack_bf16(z[4], z[5]), ptx::pack_bf16(z[6], z[7]));
            ptx::st_shared_v4(gk + ptx::sw128_offset((uint32_t)row, ch16 + 1), ptx::pack_bf16(z[8], z[9]),
                              ptx::pack_bf16(z[10], z[11]), ptx::pack_bf16(z[12], z[13]), ptx::pack_bf16(z[14], z[15]));
          }
        }
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();  // G (generic-proxy stores) -> visible to the tensor cores' async proxy
        ptx::mbar_arrive_cluster(gr_leader);

        // ---- epilogue 2: residual (columns [0,128)) -> in place over the window's centre rows (the next layer's centre
        //      tap); skip (columns [128,256)) -> fp32 slabs in the G buffer -> TMA reduce-add (plain store on layer 0)
        ptx::mbar_wait(&sb->d2_full, pl);
        ptx::tc_fence_after();
        if (!last) {
          if (l == 0) ptx::mbar_wait(&sb->xw_full, 0);  // (long complete) makes the TMA-written window visible here
          uint32_t rr[2][16];
          ptx::tmem_ld16(tcol + 16 * sub, rr[0]);
#pragma unroll
          for (int i = 0; i < 8 / kDW; ++i) {
            const int c0 = 16 * (kDW * i + sub);
            ptx::tmem_ld_wait();
            if (i + 1 < 8 / kDW) ptx::tmem_ld16(tcol + c0 + 16 * kDW, rr[(i + 1) & 1]);
            const uint32_t* r = rr[i & 1];
            uint8_t* xt = xw_smem + (c0 >> 6) * kDWinBytes + kDHalo * 128;  // centre rows of the window tile
            const uint32_t ch16 = (uint32_t)((c0 & 63) >> 3);
            uint8_t* p0 = xt + ptx::sw128_offset((uint32_t)row, ch16);
            uint8_t* p1 = xt + ptx::sw128_offset((uint32_t)row, ch16 + 1);
            const uint4 xa = ptx::ld_shared_v4(p0), xb = ptx::ld_shared_v4(p1);
            const uint32_t xo[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
            uint32_t o[8];
#pragma unroll
            for (int e = 0; e < 8; e += 2) {
              const float4 bo = ptx::ld_shared_v4f(bo_s + c0 + 2 * e);
              const float v0 = (ptx::bf16_lo(xo[e]) + __uint_as_float(r[2 * e]) + bo.x) * s2;
              const float v1 = (ptx::bf16_hi(xo[e]) + __uint_as_float(r[2 * e + 1]) + bo.y) * s2;
              const float v2 = (ptx::bf16_lo(xo[e + 1]) + __uint_as_float(r[2 * e + 2]) + bo.z) * s2;
              const float v3 = (ptx::bf16_hi(xo[e + 1]) + __uint_as_float(r[2 * e + 3]) + bo.w) * s2;
              o[e] = in_seq ? ptx::pack_bf16(v0, v1) : 0u;  // rows past the end stay zero: they are the conv's zero padding
              o[e + 1] = in_seq ? ptx::pack_bf16(v2, v3) : 0u;
            }
            ptx::st_shared_v4(p0, o[0], o[1], o[2], o[3]);
            ptx::st_shared_v4(p1, o[4], o[5], o[6], o[7]);
          }
          ptx::fence_proxy_async_smem();
          ptx::mbar_arrive_cluster(xc_leader);  // the next layer's centre tap is waiting for this
          ptx::mbar_arrive(&sb->xe_ready);
        }
        // skip: 4 slabs of 32 columns (one 128-byte fp32 row per frame); the kDW warps of a lane quarter alternate slabs,
        // each stages its 32 rows of a slab in its own 4 KB piece of a G tile and issues its own TMA reduce-add
        {
          constexpr int kSlots = kDGTiles / kDW > 0 ? kDGTiles / kDW : 1;  // staging tiles per warp
          static_assert(kDW * kSlots <= kDGTiles, "skip staging needs one G tile per concurrently staging warp");
          int n_staged = 0;
#pragma unroll 1
          for (int k = sub; k < 4; k += kDW, ++n_staged) {
            const int c0 = kDC + 32 * k;
            uint32_t r0[16], r1[16];
            ptx::tmem_ld16(tcol + c0, r0);
            ptx::tmem_ld16(tcol + c0 + 16, r1);
            if (n_staged >= kSlots) {  // the staging tile is used again: its previous TMA must have read it
              if (lane == 0) {
                if (kSlots == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
              }
              __syncwarp();
            }
            uint8_t* slab = g_smem + (sub * kSlots + n_staged % kSlots) * kDTile;
            ptx::tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
              const uint32_t* r = e < 16 ? r0 : r1;
              const float4 bo = ptx::ld_shared_v4f(bo_s + c0 + e);
              ptx::st_shared_v4f(slab + ptx::sw128_offset((uint32_t)row, (uint32_t)(e >> 2)),
                                 __uint_as_float(r[e & 15]) + bo.x, __uint_as_float(r[(e & 15) + 1]) + bo.y,
                                 __uint_as_float(r[(e & 15) + 2]) + bo.z, __uint_as_float(r[(e & 15) + 3]) + bo.w);
            }
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              const int ch0 = c0 - kDC;  // first skip channel of the slab
              if (l == 0 && a.init_skip) ptx::tma_store_3d(&tm_skip, slab + q * 4096, ch0, t_cta0 + q * 32, b);
              else ptx::tma_reduce_add_3d(&tm_skip, slab + q * 4096, ch0, t_cta0 + q * 32, b);
              ptx::bulk_commit_group();
            }
          }
          if (lane == 0) {
            ptx::bulk_wait_read_all();  // this warp's slabs are read: the G buffer may take the next conditioner tiles
            ptx::mbar_arrive(&sb->gc_free);
          }
        }
        ptx::tc_fence_before();
        ptx::mbar_arrive_cluster(dr_leader);
        // the bias arrays are rewritten at the top of the next layer: every epilogue thread of the slot must be done with them
        ptx::named_bar_sync(1 + u, kDEpi);
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();  // the peer's smem / TMEM are in use by the leader's MMAs until here
  if (warp == 1) ptx::tmem_dealloc2(tmem, 512);
}

static int duo_smem(int H, int* nentries_out) {
  (void)H;
  const int fixed = 2 * kDSlotBytes + 2 * 4 * kDTwoC * (int)sizeof(float) + (int)sizeof(DuoBarriers) + 1024;
  int nentries = (kDSmemLimit - fixed) / kDTile;
  if (nentries > kDMaxEntries) nentries = kDMaxEntries;
  *nentries_out = nentries;
  return fixed + nentries * kDTile;
}

using DuoKernelFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap,
                             DuoArgs);
static DuoKernelFn duo_kernel_variant(int hb) {
  return hb == 1 ? diffnet_stack_duo_kernel<1> : diffnet_stack_duo_kernel<2>;
}

bool diffnet_stack_duo_applies(int C, int H) {
  return C == kDC && H > 0 && H % 64 == 0 && H <= 128 && !getenv("SVSK_STACK_NO_DUO");
}

static int duo_prepare(int* nentries, int* smem_bytes) {
  *smem_bytes = duo_smem(0, nentries);
  SVSK_REQUIRE(*nentries >= 3, SVSK_E_ARG, "diffnet_stack_bf16: not enough shared memory");
  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaSuccess;
    for (int hb = 1; hb <= 2 && e == cudaSuccess; ++hb)
      e = cudaFuncSetAttribute(duo_kernel_variant(hb), cudaFuncAttributeMaxDynamicSharedMemorySize, kDSmemLimit);
    if (e != cudaSuccess) return fail((int)e, "diffnet_stack_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  return 0;
}

static void duo_launch_config(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* attr, int B, int T, int smem_bytes, void* stream) {
  *cfg = cudaLaunchConfig_t{};
  const int n256 = ceil_div(T, 256);
  cfg->gridDim = dim3(2 * ceil_div(n256, 2), B);
  cfg->blockDim = dim3(kDThreads);
  cfg->dynamicSmemBytes = smem_bytes;
  cfg->stream = as_stream(stream);
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  // cooperative: the grid starts only when ALL its CTAs can be resident at once — the neighbour hand-shakes need it.
  // A track that is a single CTA pair has no neighbour: plain launch.
  attr[1].id = cudaLaunchAttributeCooperative;
  attr[1].val.cooperative = 1;
  cfg->attrs = attr;
  cfg->numAttrs = n256 <= 2 ? 1 : 2;
}

// 1 / 0: all CTA pairs of B tracks x T frames fit the device at once / do not
int diffnet_stack_duo_fits(int B, int T) {
  int nentries = 0, smem_bytes = 0;
  if (duo_prepare(&nentries, &smem_bytes)) return 0;
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  duo_launch_config(&cfg, attr, B, T, smem_bytes, nullptr);
  int max_clusters = 0;
  if (cudaOccupancyMaxActiveClusters(&max_clusters, duo_kernel_variant(2), &cfg) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return (int)(cfg.gridDim.x / 2) * B <= max_clusters ? 1 : 0;
}

// Called by svsk_diffnet_stack_bf16 (diffnet_stack_sm100.cu) after the common argument checks.
int diffnet_stack_duo_launch(const svsk_diffnet_stack_params& p, void* stream) {
  int rc, nentries = 0, smem_bytes = 0;
  if ((rc = duo_prepare(&nentries, &smem_bytes))) return rc;
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  duo_launch_config(&cfg, attr, p.B, p.T, smem_bytes, stream);
  int max_clusters = 0;
  cudaError_t oe = cudaOccupancyMaxActiveClusters(&max_clusters, duo_kernel_variant(2), &cfg);
  if (oe != cudaSuccess) return fail((int)oe, "diffnet_stack_bf16: cudaOccupancyMaxActiveClusters: %s", cudaGetErrorString(oe));
  const int n_clusters = (int)(cfg.gridDim.x / 2) * p.B;
  SVSK_REQUIRE(n_clusters <= max_clusters, SVSK_E_ARG,
               "diffnet_stack_bf16: %d CTA pairs do not fit the device at once (%d); run the layers with "
               "svsk_diffnet_block3_bf16", n_clusters, max_clusters);

  CUtensorMap tm_xw0, tm_e0, tm_e1, tm_cond, tm_w1, tm_wout, tm_skip;
  {
    uint64_t dims[3] = {(uint64_t)p.C, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.C * 2, (uint64_t)p.T * p.C * 2};
    uint32_t boxw[3] = {64, (uint32_t)kDWinRows, 1};
    uint32_t boxe[3] = {64, (uint32_t)kDHalo, 1};
    if ((rc = make_tmap_bf16(&tm_xw0, p.xb_in, 3, dims, str, boxw))) return rc;
    if ((rc = make_tmap_bf16(&tm_e0, p.edge0, 3, dims, str, boxe))) return rc;
    if ((rc = make_tmap_bf16(&tm_e1, p.edge1, 3, dims, str, boxe))) return rc;
    uint64_t str4[2] = {(uint64_t)p.C * 4, (uint64_t)p.T * p.C * 4};
    uint32_t box4[3] = {32, 32, 1};  // one warp's 32 rows of a 32-column skip slab
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
    uint64_t dims[3] = {K1, (uint64_t)2 * p.C, (uint64_t)p.L};
    uint64_t str[2] = {K1 * 2, K1 * 2 * 2 * p.C};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_w1, p.w1p, 3, dims, str, box))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)p.C, (uint64_t)2 * p.C, (uint64_t)p.L};
    uint64_t str[2] = {(uint64_t)p.C * 2, (uint64_t)p.C * 2 * 2 * p.C};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_wout, p.woutp, 3, dims, str, box))) return rc;
  }

  DuoArgs a;
  a.stepbias = p.stepbias;
  a.bout = p.bout;
  a.flags = p.flags;
  a.B = p.B; a.T = p.T; a.H = p.H; a.L = p.L;
  a.sb_batch_stride = p.stepbias_batch_stride;
  a.sb_layer_stride = p.stepbias_layer_stride;
  a.init_skip = p.init_skip;
  a.nentries = nentries;
  a.tiles_per_track = 2 * ceil_div(p.T, 256);
  for (int l = 0; l < kDMaxLayers; ++l) a.dilation[l] = l < p.L ? p.dilation[l] : 1;

  cudaError_t e = cudaMemsetAsync(p.flags, 0, sizeof(int) * (size_t)p.B * a.tiles_per_track, as_stream(stream));
  if (e != cudaSuccess) return fail((int)e, "diffnet_stack_bf16: flag reset: %s", cudaGetErrorString(e));
  e = cudaLaunchKernelEx(&cfg, duo_kernel_variant(p.H / 64), tm_xw0, tm_e0, tm_e1, tm_cond, tm_w1, tm_wout, tm_skip, a);
  if (e != cudaSuccess) return fail((int)e, "diffnet_stack_bf16: launch: %s", cudaGetErrorString(e));
  return check_launch("diffnet_stack_bf16 (two tiles per CTA pair)");
}

}  // namespace svsk
