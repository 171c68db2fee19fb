// The whole DiffNet residual stack in ONE launch: replaces the loop over ResidualBlock.forward in DiffNet.forward
// (nnsvs/diffsinger/denoiser.py:114-118; block maths denoiser.py:54-66) for all L layers of one denoiser call.
//
// Why: the per-layer kernel (diffnet_block3_sm100.cu) computes for 20.5 k tensor-pipe cycles out of a 50 k-cycle
// launch period (profiles/r01w_timeline_v3.log): 6 k cycles pass before the first MMA (barrier/TMEM set-up, cluster
// sync, first loads), 5 k between a CTA's exit and its successor's start, the skip epilogue (6.7 k) runs with the
// tensor pipe idle.  At the reference workload (6 tracks x 2000 frames) there is exactly one 128-frame tile per SM, so
// every CTA can simply KEEP its tile for all layers:
//   * set-up once per call instead of once per layer;
//   * the centre rows of the activation window are updated in place by the residual epilogue and are already the next
//     layer's centre tap: only the 8 halo rows either side come from the neighbouring tiles, through global memory
//     Two transports: when a whole track fits one thread-block cluster (<= 16 tiles = 2048 frames, the reference
//     workload) the epilogue threads of the edge rows write them straight into the neighbouring CTAs' windows through
//     distributed shared memory (~1 k cycles door to door); otherwise they are TMA-stored to a scratch tensor, a
//     per-tile layer counter is released, and the neighbour TMA-loads them (~8 k cycles: every hop is an L2 round trip
//     of ~2.5 k cycles under the weight stream's load, profiles/r01x_bench_stack_timeline.log);
//   * the next layer's weights stream in while the skip epilogue of this layer drains TMEM: GEMM1 of layer l+1 starts
//     on the first 256 TMEM columns as soon as the residual half has been read out.
// Everything else (operand layouts, row-offset tap descriptors, gating, TMA epilogues) is the per-layer kernel's.
//
// In that one-cluster-per-track mode the weight tiles, identical for every tile of the track, are TMA-multicast: each
// CTA pair fetches 1/n_pairs of every tile for all CTAs of its parity, so L2 serves each weight byte once per track
// instead of once per tile, and a ring slot is refilled when ALL pairs have released it (cluster-wide empty barrier).
//
// Per layer, ring entries (16 KB weight tiles) in this order — producer, MMA issuer and the peer's forwarder agree:
//   0: centre tap, block 0        (A = window rows 8..135, needs only this CTA pair's own previous epilogue)
//   1: side taps, block 0         (A = window at rows 8 -/+ d, needs the neighbours' edge rows of the previous layer)
//   2: conditioner, blocks 0..NB-1 (A = conditioner tiles in the G buffer, which the previous skip epilogue released)
//   3: all taps, blocks 1..NB-1
//   4: output projection, blocks 0..NB-1 (A = G)
// Hoisted conditioner projection (kUseP, svsk_diffnet_stack_params::pcond_*): inside a sampling run cond is the same
// for all K denoiser calls, so conditioner_projection(cond) of every layer is computed once per run and this kernel skips
// entry group 2 (K = 3C instead of 3C + H: 20 % of the MMAs at C = H = 256, and the wait for the conditioner tiles).  The
// projection comes back in the gating epilogue: its gate half is TMA-loaded (bf16, the G tiles' own layout) into the very
// bytes of the G buffer that the thread overwrites with its gate output — the slot and the moment the conditioner tiles
// used to take — and its filter half is read from global memory two chunks ahead into 16 registers (a [chunk][frame][16]
// layout: a warp reads 1 KB contiguous; the lines are prefetched into L2 one layer ahead by the activation producer).
// Warps: 0 = weight producer (both CTAs), 1 = MMA issuer (leader) / forwarder (peer) + TMEM owner, 2..9 = epilogue
// (kSW = 2 per TMEM lane quarter), 10 = activation producer (conditioner tiles, window / halo rows, edge-row publication).
// All CTAs must be co-resident (neighbours wait for each other): the host entry checks the grid against
// cudaOccupancyMaxActiveClusters and refuses otherwise (callers fall back to one svsk_diffnet_block3_bf16 per layer).
#include <cuda_bf16.h>
#include <cstdlib>

#include "sm100_ptx.cuh"
#include "svsk_common.cuh"
#include "tma_util.cuh"

// How the three single-thread roles wait for a ring entry (compile-time: a run-time switch in these loops costs more than
// either flavour gains, DESIGN §4 item 17): suspending try_wait (ptx::mbar_wait) or polling test_wait (ptx::mbar_wait_spin).
// Measured with -DSVSK_STACK_{PRODUCER,ISSUER,FORWARDER}_WAIT=ptx::mbar_wait_spin builds on one box (gpurun_out/s39_ab.log,
// 6 x 2000 frames, hoisted projection): 346.1 / 347.4 / 347.0 us, all three 346.6 us, against 345.2-347.1 us suspending —
// no difference, so the suspending waits stay (they leave the issue slots to the epilogue warps).
#ifndef SVSK_STACK_PRODUCER_WAIT
#define SVSK_STACK_PRODUCER_WAIT ptx::mbar_wait
#endif
#ifndef SVSK_STACK_ISSUER_WAIT
#define SVSK_STACK_ISSUER_WAIT ptx::mbar_wait
#endif
#ifndef SVSK_STACK_FORWARDER_WAIT
#define SVSK_STACK_FORWARDER_WAIT ptx::mbar_wait
#endif

namespace svsk {

constexpr int kSTile = 128 * 128;            // 128 rows x 64 bf16
constexpr int kSHalo = 8;                    // window rows either side of the tile: dilation <= 8
constexpr int kSWinRows = 128 + 2 * kSHalo;
constexpr int kSWinBytes = kSWinRows * 128;  // 18 KB, a multiple of the 1024-byte swizzle atom
constexpr int kSHaloBytes = kSHalo * 128;    // 1 KB per window tile and side
constexpr int kSMaxEntries = 8;
constexpr int kSSmemLimit = 232448;
constexpr int kSTmemCols = 512;
// Epilogue warps per TMEM lane quarter (they alternate 16-column chunks).  2 and 4 measure the same (403 vs 395 us per
// 20-layer launch): the epilogues are bound by the TMEM read port (64 B/cycle/SM: 128 KB per gating block, per residual
// half and per skip half = 2 k cycles each), not by warp-level latency hiding; 4 costs 96-register threads.
constexpr int kSW = 2;
constexpr int kSEpi = 128 * kSW;             // epilogue threads per CTA
constexpr int kSActWarp = 2 + 4 * kSW;       // the activation producer's warp
constexpr int kSThreads = 32 * (kSActWarp + 1);
constexpr int kSMaxLayers = 64;

struct DiffnetStackArgs {
  const float* stepbias;  // [batch][layer][6C] (strides below)
  const float* bout;      // [layer][2C]
  int* flags;             // [B * tiles_per_track] layers published per tile; zero at launch
  int dsmem_halo;         // 1: one cluster per track, halo rows through distributed shared memory; 0: through global memory
  int B, T, C, H, L, sb_batch_stride, sb_layer_stride, init_skip, nentries, tiles_per_track;
  // C = 128 (one 256-column output block): the accumulator alternates between the two halves of TMEM from layer to
  // layer, so that a layer's GEMM1 does not wait for the previous layer's skip columns to be read out (they share the
  // block with the residual columns: ~5 k of a 19.4 k-cycle layer, profiles/r02j_stack_c128_timeline.log), and the
  // conditioner tiles — the same for every layer — stay in their own shared-memory tiles instead of being reloaded into
  // the G buffer once the skip epilogue has released it (3.8 k cycles into the layer).
  int cond_resident;
  // Measured in round 2 and removed (it was a run-time switch inside the single-thread roles' loops, see the template
  // parameters of the kernel): the conditioner k-blocks issued BEFORE block 0's side taps in global-memory halo mode, on the
  // idea that the halo rows land ~9.5 k cycles after the previous residual epilogue there and the conditioner MMAs need
  // none — 446.1 vs 434.5 us per launch at 3 x 6000 frames, slower: the conditioner tiles (G buffer released by the previous
  // skip epilogue, then a 64 KB load) arrive no earlier than the halo rows, and the side taps then queue behind them.
  // Hoisted conditioner projection (see the header comment): filter half, [tile][L][NB][8][128][16] bf16 from this launch's
  // first track on; the gate half comes through tm_cond (then a map of [B*L][T][C]).
  int use_p;
  const uint4* pfilt;
  // Measured and removed (gpurun_out/s24, s27; 6 x 2000 frames, hoisted projection, 371 us per launch): the peer CTA's
  // weight loads completing on the LEADER's ring barrier (cta_group::2 TMA with the peer bit of the barrier address
  // cleared, as CUTLASS's 2-SM kernels do) instead of a forwarding thread: 384 us; producer / forwarder polling
  // (mbarrier.test_wait) instead of suspending: 370 us; every pair loading its own weight tiles instead of the
  // cluster-wide multicast: 366 us with half the ring misses but 8x the L2 reads.  Their run-time switches cost the
  // single-thread roles more than any of them gained.
  int dilation[kSMaxLayers];
};

struct __align__(8) DiffnetStackBarriers {
  uint64_t full[kSMaxEntries];  // ring entry landed: own TMA bytes, and on the leader also the peer's (forwarded) arrival
  uint64_t empty[kSMaxEntries];
  uint64_t cd_full[8];          // conditioner tile hb of this layer landed (leader: in both CTAs); use_p: gate-half tile hb of the projection (each CTA its own)
  uint64_t xw_full;             // layer 0: whole window landed; later layers: halo rows landed (leader: in both CTAs)
  uint64_t xh_full;             // DSMEM mode: the neighbours' edge threads have written this CTA's halo rows (leader: both CTAs)
  uint64_t halo_free;           // DSMEM mode: the CTA pairs that read the halo rows this CTA writes have finished GEMM1
  uint64_t xc_ready;            // leader: centre rows updated in place by every epilogue thread of both CTAs
  uint64_t xe_ready;            // this CTA's centre rows updated (-> activation producer publishes the edge rows)
  uint64_t d1_full[2];
  uint64_t d2_full[2];
  uint64_t d2_drained[2];       // leader: every epilogue thread of both CTAs has read block j out of TMEM
  uint64_t g_ready[2];          // leader: gating block j written to G by every epilogue thread of both CTAs
  uint64_t gc_free;             // this CTA's G buffer is free again (skip slabs read by the TMA unit)
  uint32_t tmem_base;
};

// ring entry i of a layer -> which weight tile (see the order in the header comment)
__device__ __forceinline__ void stack_entry(int i, int CB, int HB, int NB, int KB2, int& kcol, int& blk, bool& wout) {
  wout = false;
  if (i < CB) { kcol = CB + i; blk = 0; return; }
  i -= CB;
  if (i < 2 * CB) { kcol = (i / CB) * 2 * CB + i % CB; blk = 0; return; }
  i -= 2 * CB;
  if (i < HB * NB) { kcol = 3 * CB + i / NB; blk = i % NB; return; }
  i -= HB * NB;
  if (i < (NB - 1) * 3 * CB) { blk = 1 + i / (3 * CB); kcol = i % (3 * CB); return; }
  i -= (NB - 1) * 3 * CB;
  wout = true;
  blk = i / KB2;
  kcol = i % KB2;
}

// one cluster per track: are the weight tiles multicast (see the kernel)?
__host__ __device__ constexpr bool stack_multicast(bool use_p, int C) { return !(use_p && C == 256); }

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ld_relaxed_gpu(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ uint4 ldg_stream_v4(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// kUseP: the conditioner projection is precomputed (DiffnetStackArgs::use_p) — a compile-time switch, so that the instantiation without it
// keeps the register allocation it had before the projection's prefetch registers existed (168 registers are the cap at
// 352 threads; a handful of spilled loop invariants cost the MMA-issuing thread 5 % of the launch).
// kDsmem (one cluster per track, halo rows through distributed shared memory) is compile-time for the same reason: the
// single-thread roles pay for every run-time branch in their loops.
template <bool kUseP, bool kDsmem, int kC>
__global__ void __launch_bounds__(kSThreads, 1)
diffnet_stack_kernel(const __grid_constant__ CUtensorMap tm_xw0, const __grid_constant__ CUtensorMap tm_e0,
                     const __grid_constant__ CUtensorMap tm_e1, const __grid_constant__ CUtensorMap tm_cond,
                     const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_wout,
                     const __grid_constant__ CUtensorMap tm_skip, const DiffnetStackArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  constexpr int C = kC;  // 128 or 256: loop bounds of the single-thread roles are compile-time constants
  const int H = a.H, T = a.T, L = a.L;
  constexpr int CB = C / 64;
  const int HB = kUseP ? 0 : H / 64;  // conditioner k-blocks of GEMM1 (none when the projection is precomputed)
  const int PB = kUseP ? CB : 0;      // ... then: gate-half tiles of the projection per layer, loaded where G will be written
  constexpr int KB2 = CB;
  constexpr int NB = (2 * C) / 256;  // 256-column output blocks of either GEMM
  constexpr int twoC = 2 * C;
  uint8_t* xw_smem = smem;                         // CB window tiles
  uint8_t* g_smem = xw_smem + CB * kSWinBytes;     // max(HB, KB2, 4) tiles: conditioner tiles, then G, then skip slabs
  uint8_t* cond_smem = (kC == 128 && a.cond_resident) ? g_smem + max(max(HB, KB2), 4) * kSTile : g_smem;   // HB resident tiles, or the G buffer
  uint8_t* ring = g_smem + (max(max(HB, KB2), 4) + ((kC == 128 && a.cond_resident) ? HB : 0)) * kSTile;  // nentries x 16 KB (the G buffer holds >= 4 skip slabs)
  float* sb_full = reinterpret_cast<float*>(ring + a.nentries * kSTile);
  float* sb_l = sb_full + twoC;
  float* sb_r = sb_l + twoC;
  float* bo_s = sb_r + twoC;
  DiffnetStackBarriers* bars = reinterpret_cast<DiffnetStackBarriers*>(bo_s + twoC);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = ptx::cluster_ctarank();   // rank in the cluster (a CTA pair, or a whole track in DSMEM mode)
  const uint32_t rank = crank & 1u;                // rank in the CTA pair (tcgen05 cta_group::2): 0 = leader
  const uint32_t lead = crank & ~1u;               // cluster rank of this pair's leader
  const uint32_t csize = ptx::cluster_nctarank();
  const uint16_t pair_mask = (uint16_t)(3u << lead);
  const bool nb_left = kDsmem && crank > 0, nb_right = kDsmem && crank + 1 < csize;  // DSMEM neighbours
  // weight multicast (one cluster per track): every pair fetches rows [pidx, pidx+1) * 128/n_pairs of each half-tile
  // Weight multicast inside a track's cluster (every pair fetches 1/n_pairs of a tile for all CTAs of its parity, so L2
  // serves each weight byte once per track) — except in the hoisted-projection variant at C = 256: once the single-thread
  // roles' overheads were gone (DESIGN §4 item 19) the cluster-wide coupling of the ring (a slot is refilled when ALL pairs
  // have released it) was that variant's largest stall, and per-pair loads measure 304.3 -> 290.3 us per launch at
  // 6 x 2000 frames on the same box (ring entries not yet landed when reached: 297 -> 193 of 800, gpurun_out/s50_ab.log).
  // The in-GEMM variant (326.7 vs 332.4 us) and C = 128 (85.9 vs 87.0 us) are still faster with the multicast
  // (gpurun_out/s51_ab.log).
  constexpr bool mc = kDsmem && stack_multicast(kUseP, kC);
  const int n_pairs = mc ? (int)(csize >> 1) : 1, pidx = mc ? (int)(crank >> 1) : 0;
  const int slice_rows = 128 / n_pairs;
  const uint16_t parity_mask = (uint16_t)((0x5555u << rank) & ((1u << csize) - 1u));  // CTAs with this CTA's pair rank
  const uint16_t empty_mask = mc ? (uint16_t)((1u << csize) - 1u) : pair_mask;        // whom a freed ring slot is told to
  const int b = blockIdx.y;
  const int t_cta0 = (blockIdx.x >> 1) * 256 + (int)rank * 128;  // first frame of this CTA's 128 TMEM lanes
  const int w_row0 = (int)rank * 128;                             // this CTA's half of a 256-row weight block
  const int n_layer = NB * (3 * CB + HB) + NB * KB2;              // ring entries per layer
  const int n_total = L * n_layer;
  int pre_issued = 0;  // weight producer: entries issued before the CTA-wide sync

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tm_xw0);
    ptx::prefetch_tmap(&tm_e0);
    ptx::prefetch_tmap(&tm_e1);
    ptx::prefetch_tmap(&tm_cond);
    ptx::prefetch_tmap(&tm_w1);
    ptx::prefetch_tmap(&tm_wout);
    ptx::prefetch_tmap(&tm_skip);
    const uint32_t two = rank == 0 ? 2u : 1u;        // leader barriers also count the peer's forwarded arrival
    const uint32_t all = rank == 0 ? 2u * kSEpi : 1u; // leader barriers every epilogue thread of the pair arrives on
    for (int i = 0; i < a.nentries; ++i) {
      ptx::mbar_init(&bars->full[i], two);
      ptx::mbar_init(&bars->empty[i], (uint32_t)n_pairs);  // one multicast tcgen05.commit per CTA pair sharing the weights
    }
    for (int i = 0; i < HB; ++i) ptx::mbar_init(&bars->cd_full[i], two);
    for (int i = 0; i < PB; ++i) ptx::mbar_init(&bars->cd_full[i], 1);  // read by this CTA's own epilogue threads
    ptx::mbar_init(&bars->xw_full, two);
    // halo rows: 8 * kSW arrivals per neighbour (8 rows x the kSW epilogue warps of a lane quarter) + the peer's forward
    ptx::mbar_init(&bars->xh_full, max(1u, 8u * kSW * ((nb_left ? 1u : 0u) + (nb_right ? 1u : 0u)) + (rank == 0 ? 1u : 0u)));
    // credits: this pair's GEMM1 + the GEMM1 of the pair on the other side of this CTA's outer edge
    ptx::mbar_init(&bars->halo_free, 1u + ((rank == 0 ? nb_left : nb_right) ? 1u : 0u));
    ptx::mbar_init(&bars->xc_ready, all);
    ptx::mbar_init(&bars->xe_ready, kSEpi);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->d1_full[i], 1);
      ptx::mbar_init(&bars->d2_full[i], 1);
      ptx::mbar_init(&bars->d2_drained[i], all);
    }
    ptx::mbar_init(&bars->g_ready[0], all);
    ptx::mbar_init(&bars->g_ready[1], all);
    ptx::mbar_init(&bars->gc_free, 4 * kSW);  // one arrival per epilogue warp
    ptx::fence_mbar_init();
    pre_issued = mc ? 0 : min(a.nentries, n_total);  // (multicast writes into CTAs that may not have set up their barriers yet)
    for (int e = 0; e < pre_issued; ++e) {
      int kcol, blk;
      bool wout;
      stack_entry(e, CB, HB, NB, KB2, kcol, blk, wout);
      ptx::mbar_arrive_expect_tx(&bars->full[e], kSTile);
      ptx::tma_load_3d(ring + e * kSTile, wout ? &tm_wout : &tm_w1, &bars->full[e], kcol * 64, blk * 256 + w_row0, 0);
    }
  }
  if (warp == 1) {
    ptx::tmem_alloc2(&bars->tmem_base, kSTmemCols);
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
      int s = pre_issued % a.nentries;
      uint32_t ph = (pre_issued == a.nentries) ? 1u : 0u;
      int l = pre_issued / n_layer, i = pre_issued - l * n_layer;
      for (int e = pre_issued; e < n_total; ++e) {
        // which tile: worked out BEFORE the wait (a few integer divisions by run-time values, ~100 instructions of one
        // thread) — after it they would sit on the refill path of a ring that is as deep as shared memory allows
        int kcol, blk;
        bool wout;
        stack_entry(i, CB, HB, NB, KB2, kcol, blk, wout);
        const CUtensorMap* tm = wout ? &tm_wout : &tm_w1;
        const int c0 = kcol * 64, c1 = blk * 256 + w_row0 + (mc ? pidx * slice_rows : 0);
        uint8_t* dst = ring + s * kSTile + (mc ? pidx * slice_rows * 128 : 0);
        SVSK_STACK_PRODUCER_WAIT(&bars->empty[s], ph ^ 1);
        ptx::mbar_arrive_expect_tx(&bars->full[s], kSTile);
        if (mc) ptx::tma_load_3d_mc(dst, tm, &bars->full[s], c0, c1, l, parity_mask);
        else ptx::tma_load_3d(dst, tm, &bars->full[s], c0, c1, l);
        if (++s == a.nentries) { s = 0; ph ^= 1; }
        if (++i == n_layer) { i = 0; ++l; }
      }
    }
  } else if (warp == kSActWarp) {
    // ------------------------------------------------------------------ activation producer (both CTAs)
    if (lane == 0) {
      const int tile_idx = b * a.tiles_per_track + (t_cta0 >> 7);
      const bool has_left = t_cta0 > 0, has_right = t_cta0 + 128 < T;
      // layer 0: conditioner tiles and the whole window of the stack's input
      for (int hb = 0; hb < HB; ++hb) {
        ptx::mbar_arrive_expect_tx(&bars->cd_full[hb], kSTile);
        ptx::tma_load_3d(cond_smem + hb * kSTile, &tm_cond, &bars->cd_full[hb], hb * 64, t_cta0, b);
      }
      // precomputed projection: gate-half tiles of layer l (frames past T: zero fill); filter half -> L2, one layer ahead
      const bool pf_ok = kUseP && (t_cta0 >> 7) < a.tiles_per_track;
      const uint32_t pf_layer_bytes = (uint32_t)NB * 32768u;
      const uint8_t* pf_tile = reinterpret_cast<const uint8_t*>(a.pfilt) + (size_t)tile_idx * L * pf_layer_bytes;
      auto load_pgate = [&](int l) {
        for (int hb = 0; hb < PB; ++hb) {
          ptx::mbar_arrive_expect_tx(&bars->cd_full[hb], kSTile);
          ptx::tma_load_3d(g_smem + hb * kSTile, &tm_cond, &bars->cd_full[hb], hb * 64, t_cta0, b * L + l);
        }
        if (pf_ok && l + 1 < L) prefetch_l2_bulk(pf_tile + (size_t)(l + 1) * pf_layer_bytes, pf_layer_bytes);
      };
      if (pf_ok) prefetch_l2_bulk(pf_tile, pf_layer_bytes);
      load_pgate(0);
      ptx::mbar_arrive_expect_tx(&bars->xw_full, CB * kSWinBytes);
      for (int cb = 0; cb < CB; ++cb)
        ptx::tma_load_3d(xw_smem + cb * kSWinBytes, &tm_xw0, &bars->xw_full, cb * 64, t_cta0 - kSHalo, b);
      for (int l = 1; l < L; ++l) {
        const uint32_t pp = (uint32_t)(l - 1) & 1u;
        const CUtensorMap* tm_e = pp ? &tm_e1 : &tm_e0;
        if (kDsmem) {  // the halo rows travel through distributed shared memory: only the conditioner tiles here
          if ((kC == 128 && a.cond_resident) && !kUseP) break;  // ... and not even those
          ptx::mbar_wait(&bars->gc_free, pp);
          for (int hb = 0; hb < HB; ++hb) {
            ptx::mbar_arrive_expect_tx(&bars->cd_full[hb], kSTile);
            ptx::tma_load_3d(g_smem + hb * kSTile, &tm_cond, &bars->cd_full[hb], hb * 64, t_cta0, b);
          }
          load_pgate(l);
          continue;
        }
        // publish the first / last 8 rows of layer l-1's output (the epilogue has written them in place)
        ptx::mbar_wait(&bars->xe_ready, pp);
        for (int cb = 0; cb < CB; ++cb) {
          uint8_t* centre = xw_smem + cb * kSWinBytes + kSHalo * 128;
          ptx::tma_store_3d(tm_e, centre, cb * 64, t_cta0, b);
          ptx::tma_store_3d(tm_e, centre + (128 - kSHalo) * 128, cb * 64, t_cta0 + 128 - kSHalo, b);
        }
        ptx::bulk_commit_group();
        ptx::bulk_wait_all();  // the stores are complete (not merely read out of shared memory)
        fence_proxy_async_global();
        st_release_gpu(a.flags + tile_idx, l);
        // halo rows of layer l's input: the neighbours' edge rows of layer l-1's output
        for (uint32_t spin = 0;; ++spin) {  // both flags per round trip, relaxed; one acquire fence at the end
          const int fl = has_left ? ld_relaxed_gpu(a.flags + tile_idx - 1) : l;
          const int fr = has_right ? ld_relaxed_gpu(a.flags + tile_idx + 1) : l;
          if (fl >= l && fr >= l) break;
          if (spin > (1u << 21)) __trap();
        }
        asm volatile("fence.acq_rel.gpu;" ::: "memory");
        fence_proxy_async_global();
        ptx::mbar_arrive_expect_tx(&bars->xw_full, 2 * CB * kSHaloBytes);
        for (int cb = 0; cb < CB; ++cb) {
          uint8_t* tile = xw_smem + cb * kSWinBytes;
          ptx::tma_load_3d(tile, tm_e, &bars->xw_full, cb * 64, t_cta0 - kSHalo, b);
          ptx::tma_load_3d(tile + (kSHalo + 128) * 128, tm_e, &bars->xw_full, cb * 64, t_cta0 + 128, b);
        }
        // conditioner tiles of layer l, once the G buffer is free again
        if ((kC == 128 && a.cond_resident) && !kUseP) continue;
        ptx::mbar_wait(&bars->gc_free, pp);
        for (int hb = 0; hb < HB; ++hb) {
          ptx::mbar_arrive_expect_tx(&bars->cd_full[hb], kSTile);
          ptx::tma_load_3d(g_smem + hb * kSTile, &tm_cond, &bars->cd_full[hb], hb * 64, t_cta0, b);
        }
        load_pgate(l);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer: one thread of the leader CTA
    if (rank == 0 && lane == 0) {
      const uint32_t idesc = ptx::umma_idesc_bf16_f32(256, 256);
      const uint32_t ring_lo = ptx::umma_desc_lo(ptx::smem_u32(ring)), g_lo = ptx::umma_desc_lo(ptx::smem_u32(g_smem));
      const uint32_t cond_lo = ptx::umma_desc_lo(ptx::smem_u32(cond_smem));
      const uint32_t xw_lo = ptx::umma_desc_lo(ptx::smem_u32(xw_smem));
      int s = 0;
      uint32_t ph = 0;
      // CTAs that write halo rows this pair's GEMM1 reads: the pair itself and the outer neighbour on either side
      const uint16_t halo_mask = (uint16_t)(pair_mask | (lead > 0 ? 1u << (lead - 1) : 0u) | (lead + 2 < csize ? 1u << (lead + 2) : 0u));
      bool ready = false;  // the barrier of ring entry (s, ph) was already seen complete by the previous group's probe
      // An mbarrier wait whose result is needed at once stalls this thread ~160 cycles even on a long-completed phase
      // (tools/ubench_umma.py): every MMA group therefore probes the NEXT entry's barrier while its MMAs are issued.
#define SVSK_WAIT_ENTRY()                                 \
  do {                                                    \
    if (!ready) SVSK_STACK_ISSUER_WAIT(&bars->full[s], ph); \
    ready = false;                                        \
    ptx::tc_fence_after();                                \
  } while (0)
#define SVSK_NEXT_ENTRY() do { if (++s == a.nentries) { s = 0; ph ^= 1; } } while (0)
#define SVSK_ISSUE4(dcol, alo, blo, acc0)                                                                          \
  do {                                                                                                             \
    const int sn = (s + 1 == a.nentries) ? 0 : s + 1;                                                              \
    ready = ptx::umma2_bf16_x4_probe(tmem + tb + (dcol), alo, blo, idesc, acc0, 4, &bars->full[sn], sn ? ph : ph ^ 1);  \
    ptx::umma_commit2_mc(&bars->empty[s], empty_mask);                                                                      \
    SVSK_NEXT_ENTRY();                                                                                             \
  } while (0)
      for (int l = 0; l < L; ++l) {
        const uint32_t pl = (uint32_t)l & 1u, pp = pl ^ 1u;
        const int d = a.dilation[l];
        const uint32_t tb = kC == 128 ? pl * 256u : 0u;  // TMEM column base of this layer's accumulator block(s)
        // ---- centre tap, block 0
        if (l == 0) {
          ptx::mbar_wait(&bars->xw_full, 0);
        } else {
          ptx::mbar_wait(&bars->xc_ready, pp);      // centre rows rewritten in place by the previous layer's epilogue
          // and the accumulator block read out: by the previous layer — or, alternating halves, by the one before it
          // (barrier pl completes once every two layers)
          if (kC != 128) ptx::mbar_wait(&bars->d2_drained[0], pp);
          else if (l >= 2) ptx::mbar_wait(&bars->d2_drained[pl], (uint32_t)((l - 2) >> 1) & 1u);
        }
        ptx::tc_fence_after();
        for (int cb = 0; cb < CB; ++cb) {
          SVSK_WAIT_ENTRY();
          SVSK_ISSUE4(0, xw_lo + cb * (kSWinBytes >> 4) + kSHalo * 8, ring_lo + s * (kSTile >> 4), cb != 0);
        }
        {
          {
            // ---- side taps, block 0
            if (l != 0) {  // halo rows of this layer
              if (kDsmem) ptx::mbar_wait(&bars->xh_full, pp);
              else ptx::mbar_wait(&bars->xw_full, pl);
              ptx::tc_fence_after();
            }
            for (int jt = 0; jt < 3; jt += 2) {
              const uint32_t row_lo = xw_lo + (uint32_t)(kSHalo + (jt - 1) * d) * 8u;
              for (int cb = 0; cb < CB; ++cb) {
                SVSK_WAIT_ENTRY();
                SVSK_ISSUE4(0, row_lo + cb * (kSWinBytes >> 4), ring_lo + s * (kSTile >> 4), 1);
              }
            }
          }
          {
            // ---- conditioner k-blocks out of the (future) G buffer, all output blocks per tile
            for (int hb = 0; hb < HB; ++hb) {
              if (l == 0 || !(kC == 128 && a.cond_resident)) ptx::mbar_wait(&bars->cd_full[hb], pl);
              if (hb == 0 && l != 0 && NB > 1) ptx::mbar_wait(&bars->d2_drained[1], pp);
              ptx::tc_fence_after();
              const uint32_t a_lo = cond_lo + hb * (kSTile >> 4);
              for (int j = 0; j < NB; ++j) {
                SVSK_WAIT_ENTRY();
                SVSK_ISSUE4(j * 256, a_lo, ring_lo + s * (kSTile >> 4), (j == 0 || hb != 0) ? 1 : 0);
              }
            }
          }
        }
        ptx::umma_commit2_mc(&bars->d1_full[0], pair_mask);
        // ---- all taps, blocks 1..
        for (int j = 1; j < NB; ++j) {
          if (HB == 0 && l != 0) {  // no conditioner k-blocks ahead of these: the block's first MMAs overwrite the accumulator
            ptx::mbar_wait(&bars->d2_drained[j], pp);
            ptx::tc_fence_after();
          }
          for (int jt = 0; jt < 3; ++jt) {
            const uint32_t row_lo = xw_lo + (uint32_t)(kSHalo + (jt - 1) * d) * 8u;
            for (int cb = 0; cb < CB; ++cb) {
              SVSK_WAIT_ENTRY();
              SVSK_ISSUE4(j * 256, row_lo + cb * (kSWinBytes >> 4), ring_lo + s * (kSTile >> 4), (HB == 0 && jt == 0 && cb == 0) ? 0 : 1);
            }
          }
          ptx::umma_commit2_mc(&bars->d1_full[j], pair_mask);
        }
        // GEMM1 of this layer has read the window for the last time: the neighbouring tiles may overwrite its halo rows
        if (kDsmem) ptx::umma_commit2_mc(&bars->halo_free, halo_mask);
        // ---- GEMM2: G tiles of gating block 0 first (its k-blocks of output block 0 run while block 1 is still gated)
        ptx::mbar_wait(&bars->g_ready[0], pl);
        ptx::tc_fence_after();
        for (int j = 0; j < NB; ++j) {
          for (int kb = 0; kb < KB2; ++kb) {
            if (NB > 1 && j == 0 && kb == KB2 / 2) {  // G tiles KB2/2.. come from gating block 1
              ptx::mbar_wait(&bars->g_ready[1], pl);
              ptx::tc_fence_after();
            }
            SVSK_WAIT_ENTRY();
            SVSK_ISSUE4(j * 256, g_lo + kb * (kSTile >> 4), ring_lo + s * (kSTile >> 4), kb != 0);
          }
          ptx::umma_commit2_mc(&bars->d2_full[j], pair_mask);
        }
      }
#undef SVSK_WAIT_ENTRY
#undef SVSK_NEXT_ENTRY
#undef SVSK_ISSUE4
    } else if (rank == 1 && lane == 0) {
      // peer CTA: second arrival on the leader's barriers ("mine has landed too"), in the order the leader waits
      int s = 0;
      uint32_t ph = 0;
      const uint32_t leader_full0 = ptx::mapa(ptx::smem_u32(&bars->full[0]), lead);
      for (int l = 0; l < L; ++l) {
        const uint32_t pl = (uint32_t)l & 1u;
        int i = 0;
        auto forward_entries = [&](int n) {
          for (int k = 0; k < n; ++k, ++i) {
            SVSK_STACK_FORWARDER_WAIT(&bars->full[s], ph);
            ptx::mbar_arrive_cluster(leader_full0 + (uint32_t)s * 8u);
            if (++s == a.nentries) { s = 0; ph ^= 1; }
          }
        };
        auto forward_xw = [&]() {
          if (kDsmem && l != 0) {
            ptx::mbar_wait(&bars->xh_full, pl ^ 1u);
            ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->xh_full), lead));
            return;
          }
          ptx::mbar_wait(&bars->xw_full, pl);
          ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->xw_full), lead));
        };
        if (l == 0) forward_xw();
        forward_entries(CB);
        {
          {
            if (l != 0) forward_xw();
            forward_entries(2 * CB);
          }
          {
            for (int hb = 0; hb < HB; ++hb) {
              if (l == 0 || !(kC == 128 && a.cond_resident)) {
                ptx::mbar_wait(&bars->cd_full[hb], pl);
                ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&bars->cd_full[hb]), lead));
              }
              forward_entries(NB);
            }
          }
        }
        forward_entries((NB - 1) * 3 * CB + NB * KB2);
      }
    }
  } else if (warp >= 2 && warp < kSActWarp) {
    // ------------------------------------------------------------------ epilogue warps (thread = one frame)
    const int q = warp & 3;           // TMEM lane quarter this warp may read
    const int sub = (warp - 2) >> 2;  // the kSW warps of a quarter alternate 16-column chunks
    const int row = q * 32 + lane;
    const int t = t_cta0 + row;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    const bool in_seq = t < T;
    const uint32_t xc_leader = ptx::mapa(ptx::smem_u32(&bars->xc_ready), lead);
    const uint32_t gr_leader = ptx::mapa(ptx::smem_u32(&bars->g_ready[0]), lead);
    const uint32_t dr_leader = ptx::mapa(ptx::smem_u32(&bars->d2_drained[0]), lead);
    const float s2 = 0.70710678118654752f;
    // DSMEM mode: this thread's row is one of the tile's first / last 8 -> it is also a halo row of a neighbouring CTA
    const bool send_left = nb_left && row < kSHalo, send_right = nb_right && row >= 128 - kSHalo;
    const uint32_t nb_rank = send_left ? crank - 1 : (send_right ? crank + 1 : crank);
    const uint32_t nb_row = send_left ? (uint32_t)(kSHalo + 128 + row) : (uint32_t)(row - (128 - kSHalo));
    const uint32_t nb_xw = ptx::mapa(ptx::smem_u32(xw_smem), nb_rank);       // the neighbour's window, cluster address
    const uint32_t nb_bar = ptx::mapa(ptx::smem_u32(&bars->xh_full), nb_rank);
    // precomputed conditioner projection, filter half: this thread's 32 bytes of chunk ci of (layer l, block j) are the two
    // uint4 at pf_row + ((l * NB + j) * 8 + ci) * 256
    const bool pf_ok = kUseP && (t_cta0 >> 7) < a.tiles_per_track;
    const uint4* pf_row = a.pfilt + (size_t)(b * a.tiles_per_track + (t_cta0 >> 7)) * L * NB * 2048 + row * 2;
    constexpr int kChunks = 8 / kSW;  // 16-column chunks per thread and gating block
    static_assert(kChunks % 2 == 0, "the two prefetch slots alternate per chunk across blocks");

    uint32_t acc_col = 0;  // C = 128: TMEM column of this layer's accumulator, alternating halves
    for (int l = 0; l < L; ++l) {
      const uint32_t pl = (uint32_t)l & 1u;
      const int d = a.dilation[l];
      const uint32_t tcol = tmem + tlane + acc_col;   // this thread's lane, this layer's accumulator
      const bool has_l = (t - d) >= 0, has_r = (t + d) < T;
      // A track's first / last d frames lack a tap's bias term.  Warp-uniform, so that the correction is a BRANCH around the
      // rare case: written per element (if (!has_l) ...) it compiled to 64 predicated-off loads + 64 adds per 16-column
      // chunk in every thread — a third of the gating loop's instructions (profiles/r02p_stack_gating_sass.txt).
      const bool warp_edge = __any_sync(0xffffffffu, !has_l || !has_r);
      const bool last = (l == L - 1);
      // per-column biases of this layer -> smem: sb_full = centre + left + right tap terms (an interior frame's sum)
      {
        const float* sb = a.stepbias + (size_t)b * a.sb_batch_stride + (size_t)l * a.sb_layer_stride;
        const float* bo = a.bout + (size_t)l * twoC;
        for (int i = threadIdx.x - 64; i < twoC; i += kSEpi) {
          const float lft = sb[i], c = sb[twoC + i], r = sb[2 * twoC + i];
          sb_full[i] = c + lft + r;
          sb_l[i] = lft;
          sb_r[i] = r;
          bo_s[i] = bo[i];
        }
        ptx::named_bar_sync(1, kSEpi);
      }
      // filter half of the projection: chunks n and n + 1 of the layer's kChunks * NB are in flight while chunk n - 1 is gated
      uint4 pfq[2][2] = {};
      if (pf_ok) {
        const uint4* p0 = pf_row + (size_t)(l * NB * 8 + sub) * 256;
        pfq[0][0] = ldg_stream_v4(p0);
        pfq[0][1] = ldg_stream_v4(p0 + 1);
        pfq[1][0] = ldg_stream_v4(p0 + kSW * 256);
        pfq[1][1] = ldg_stream_v4(p0 + kSW * 256 + 1);
      }

      // ---- epilogue 1: gating -> G
      for (int j = 0; j < NB; ++j) {
        ptx::mbar_wait(&bars->d1_full[j], pl);
        ptx::tc_fence_after();
        uint32_t rgb[2][16], rfb[2][16];
        ptx::tmem_ld16(tcol + j * 256 + 16 * sub, rgb[0]);
        ptx::tmem_ld16(tcol + j * 256 + 128 + 16 * sub, rfb[0]);
#pragma unroll
        for (int i = 0; i < 8 / kSW; ++i) {
          const int c0 = 16 * (kSW * i + sub);
          ptx::tmem_ld_wait();
          if (i + 1 < 8 / kSW) {  // next chunk's TMEM loads fly while this chunk is gated
            ptx::tmem_ld16(tcol + j * 256 + c0 + 16 * kSW, rgb[(i + 1) & 1]);
            ptx::tmem_ld16(tcol + j * 256 + 128 + c0 + 16 * kSW, rfb[(i + 1) & 1]);
          }
          const uint32_t* rg = rgb[i & 1];
          const uint32_t* rf = rfb[i & 1];
          const int pg = j * 256 + c0, pf = pg + 128;
          const int kc0 = j * 128 + c0;  // first gated channel of the chunk = K index of GEMM2
          uint8_t* gk = g_smem + (kc0 >> 6) * kSTile;
          const uint32_t ch16 = (uint32_t)((kc0 & 63) >> 3);
          uint32_t pfw[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          if (kUseP) {
            // gate half: the bf16 values sit where this thread will store z (tile kc0 / 64 of the G buffer); read 8 bytes
            // at a time next to their use
            if ((i & (4 / kSW - 1)) == 0) ptx::mbar_wait(&bars->cd_full[kc0 >> 6], pl);
            const uint4 fa = pfq[i & 1][0], fb = pfq[i & 1][1];
            pfw[0] = fa.x; pfw[1] = fa.y; pfw[2] = fa.z; pfw[3] = fa.w;
            pfw[4] = fb.x; pfw[5] = fb.y; pfw[6] = fb.z; pfw[7] = fb.w;
            // refill the slot with chunk n + 2 of this layer
            const int n2 = j * kChunks + i + 2;
            if (pf_ok && n2 < NB * kChunks) {
              const int j2 = n2 / kChunks, ci2 = kSW * (n2 % kChunks) + sub;
              const uint4* p2 = pf_row + (size_t)((l * NB + j2) * 8 + ci2) * 256;
              pfq[i & 1][0] = ldg_stream_v4(p2);
              pfq[i & 1][1] = ldg_stream_v4(p2 + 1);
            }
          }
          uint64_t gv[8], fv[8];  // column pairs: FADD2 / FMUL2 / FFMA2 halve the issue slots of this issue-bound loop
#pragma unroll
          for (int e = 0; e < 16; e += 4) {
            const float4 bg = ptx::ld_shared_v4f(sb_full + pg + e);
            const float4 bf = ptx::ld_shared_v4f(sb_full + pf + e);
            gv[e >> 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rg[e]), __uint_as_float(rg[e + 1])), ptx::f2_pack(bg.x, bg.y));
            gv[(e >> 1) + 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rg[e + 2]), __uint_as_float(rg[e + 3])), ptx::f2_pack(bg.z, bg.w));
            fv[e >> 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rf[e]), __uint_as_float(rf[e + 1])), ptx::f2_pack(bf.x, bf.y));
            fv[(e >> 1) + 1] = ptx::f2_add(ptx::f2_pack(__uint_as_float(rf[e + 2]), __uint_as_float(rf[e + 3])), ptx::f2_pack(bf.z, bf.w));
            if (kUseP) {
              const uint2 pgw = ptx::ld_shared_v2(gk + ptx::sw128_offset((uint32_t)row, ch16 + (uint32_t)(e >> 3)) + (e & 4) * 2);
              gv[e >> 1] = ptx::f2_add(gv[e >> 1], ptx::f2_pack(ptx::bf16_lo(pgw.x), ptx::bf16_hi(pgw.x)));
              gv[(e >> 1) + 1] = ptx::f2_add(gv[(e >> 1) + 1], ptx::f2_pack(ptx::bf16_lo(pgw.y), ptx::bf16_hi(pgw.y)));
              fv[e >> 1] = ptx::f2_add(fv[e >> 1], ptx::f2_pack(ptx::bf16_lo(pfw[e >> 1]), ptx::bf16_hi(pfw[e >> 1])));
              fv[(e >> 1) + 1] = ptx::f2_add(fv[(e >> 1) + 1], ptx::f2_pack(ptx::bf16_lo(pfw[(e >> 1) + 1]), ptx::bf16_hi(pfw[(e >> 1) + 1])));
            }
          }
          if (warp_edge) {
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
          ptx::st_shared_v4(gk + ptx::sw128_offset((uint32_t)row, ch16), ptx::pack_bf16(z[0], z[1]),
                            ptx::pack_bf16(z[2], z[3]), ptx::pack_bf16(z[4], z[5]), ptx::pack_bf16(z[6], z[7]));
          ptx::st_shared_v4(gk + ptx::sw128_offset((uint32_t)row, ch16 + 1), ptx::pack_bf16(z[8], z[9]),
                            ptx::pack_bf16(z[10], z[11]), ptx::pack_bf16(z[12], z[13]), ptx::pack_bf16(z[14], z[15]));
        }
        ptx::tc_fence_before();
        ptx::fence_proxy_async_smem();  // G (generic-proxy stores) -> visible to the tensor cores' async proxy
        ptx::mbar_arrive_cluster(gr_leader + (uint32_t)j * 8u);
      }

      // ---- epilogue 2: residual -> in place over the window's centre rows (the next layer's centre tap) ;
      //      skip -> fp32 slabs in the G buffer -> TMA reduce-add (or plain store on the first layer)
      for (int j = 0; j < NB; ++j) {
        ptx::mbar_wait(&bars->d2_full[j], pl);
        ptx::tc_fence_after();
        const int res_cols = min(max(C - j * 256, 0), 256);  // residual columns in this 256-column block
        bool drained_said = false;
        if (res_cols > 0 && !last) {
          if (l == 0) ptx::mbar_wait(&bars->xw_full, 0);  // (long complete) makes the TMA-written window visible here
          if (send_left || send_right) ptx::mbar_wait(&bars->halo_free, pl);  // the neighbour's GEMM1 of this layer is done
          const int n_res = res_cols / (16 * kSW);
          uint32_t rr[2][16];
          ptx::tmem_ld16(tcol + j * 256 + 16 * sub, rr[0]);
#pragma unroll
          for (int i = 0; i < 16 / kSW; ++i) {
            if (i < n_res) {
              const int c0 = 16 * (kSW * i + sub);
              const int oc0 = j * 256 + c0;  // output channel = residual channel
              ptx::tmem_ld_wait();
              if (i + 1 < n_res) ptx::tmem_ld16(tcol + j * 256 + c0 + 16 * kSW, rr[(i + 1) & 1]);  // flies during the maths
              const uint32_t* r = rr[i & 1];
              uint8_t* xt = xw_smem + (oc0 >> 6) * kSWinBytes + kSHalo * 128;  // centre rows of the window tile
              const uint32_t ch16 = (uint32_t)((oc0 & 63) >> 3);
              uint8_t* p0 = xt + ptx::sw128_offset((uint32_t)row, ch16);
              uint8_t* p1 = xt + ptx::sw128_offset((uint32_t)row, ch16 + 1);
              const uint4 xa = ptx::ld_shared_v4(p0), xb = ptx::ld_shared_v4(p1);
              const uint32_t xo[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
              uint32_t o[8];
              const uint64_t s22 = ptx::f2_pack(s2, s2);
#pragma unroll
              for (int e = 0; e < 8; e += 2) {  // column pairs; same order of operations per lane: ((x + r) + bo) * s2
                const float4 bo = ptx::ld_shared_v4f(bo_s + oc0 + 2 * e);
                float v0, v1, v2, v3;
                ptx::f2_unpack(ptx::f2_mul(ptx::f2_add(ptx::f2_add(ptx::f2_pack(ptx::bf16_lo(xo[e]), ptx::bf16_hi(xo[e])),
                                                                   ptx::f2_pack(__uint_as_float(r[2 * e]), __uint_as_float(r[2 * e + 1]))),
                                                       ptx::f2_pack(bo.x, bo.y)), s22), v0, v1);
                ptx::f2_unpack(ptx::f2_mul(ptx::f2_add(ptx::f2_add(ptx::f2_pack(ptx::bf16_lo(xo[e + 1]), ptx::bf16_hi(xo[e + 1])),
                                                                   ptx::f2_pack(__uint_as_float(r[2 * e + 2]), __uint_as_float(r[2 * e + 3]))),
                                                       ptx::f2_pack(bo.z, bo.w)), s22), v2, v3);
                o[e] = in_seq ? ptx::pack_bf16(v0, v1) : 0u;  // rows past the end stay zero: they are the conv's zero padding
                o[e + 1] = in_seq ? ptx::pack_bf16(v2, v3) : 0u;
              }
              ptx::st_shared_v4(p0, o[0], o[1], o[2], o[3]);
              ptx::st_shared_v4(p1, o[4], o[5], o[6], o[7]);
              if (send_left || send_right) {  // the same 32 bytes into the neighbour's halo row
                const uint32_t dst = nb_xw + (uint32_t)(oc0 >> 6) * kSWinBytes;
                ptx::st_cluster_v4(dst + ptx::sw128_offset(nb_row, ch16), o[0], o[1], o[2], o[3]);
                ptx::st_cluster_v4(dst + ptx::sw128_offset(nb_row, ch16 + 1), o[4], o[5], o[6], o[7]);
              }
            }
          }
          if (j * 256 + 256 >= C) {  // all residual columns of this frame are written
            ptx::fence_proxy_async_smem();
            ptx::mbar_arrive_cluster(xc_leader);  // first: the next layer's centre tap is waiting for this
            ptx::mbar_arrive(&bars->xe_ready);
            if (res_cols == 256 && kC != 128) {
              // ... and for this: the block holds no skip columns, so this thread has read all of it out of TMEM.  Said
              // BEFORE the edge threads' cluster-scope fence below (MEMBAR.ALL.GPU + L1 invalidate, ~3 k cycles in 4 of the
              // 8 epilogue warps), during which the next layer's first MMA used to wait on a condition long true:
              // 392.4 -> 375.9 us per 20-layer launch at config 2, same box (profiles/r02h_stack_ab.log)
              ptx::tc_fence_before();
              ptx::mbar_arrive_cluster(dr_leader + (uint32_t)j * 8u);
              drained_said = true;
            }
            if (send_left || send_right) {
              ptx::fence_proxy_async_cluster_release();  // remote generic-proxy stores -> the neighbour's tensor cores
              ptx::mbar_arrive_cluster(nb_bar);
            }
          }
        }
        // skip part: columns [res_cols, 256) of this block in slabs of 32 (one 128-byte fp32 row per frame).  Each warp
        // owns whole slabs (the two warps of a lane quarter alternate) and its 32 rows of them: it stages them in a
        // private 2 x 4 KB piece of the G buffer and issues its own TMA reduce-add — no CTA-wide barrier, no shared
        // staging buffer to wait for.
        if (res_cols < 256) {
          if (j != NB - 1) __trap();  // skip columns only live in the last block: GEMM2 is done, the G buffer is free
          const int n_skip = (256 - res_cols) / 32;
          constexpr int kSlots = 4 / kSW;  // staging slots per warp: tiles sub*kSlots + m of the G buffer, rows 32q .. 32q+31
          int m = 0;
#pragma unroll 1
          for (int k = sub; k < n_skip; k += kSW, m = (m + 1) % kSlots) {
            const int c0 = res_cols + 32 * k;
            uint32_t r0[16], r1[16];
            ptx::tmem_ld16(tcol + j * 256 + c0, r0);
            ptx::tmem_ld16(tcol + j * 256 + c0 + 16, r1);
            if (k >= sub + kSW * kSlots) {  // the slot is used again: its previous TMA must have read it
              if (lane == 0) {
                if (kSlots == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
              }
              __syncwarp();
            }
            uint8_t* slab = g_smem + (sub * kSlots + m) * kSTile;
            ptx::tmem_ld_wait();
            const int oc0 = j * 256 + c0;
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
              const uint32_t* r = e < 16 ? r0 : r1;
              const float4 bo = ptx::ld_shared_v4f(bo_s + oc0 + e);
              ptx::st_shared_v4f(slab + ptx::sw128_offset((uint32_t)row, (uint32_t)(e >> 2)),
                                 __uint_as_float(r[e & 15]) + bo.x, __uint_as_float(r[(e & 15) + 1]) + bo.y,
                                 __uint_as_float(r[(e & 15) + 2]) + bo.z, __uint_as_float(r[(e & 15) + 3]) + bo.w);
            }
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              const int ch0 = oc0 - C;  // first skip channel of the slab
              if (l == 0 && a.init_skip) ptx::tma_store_3d(&tm_skip, slab + q * 4096, ch0, t_cta0 + q * 32, b);
              else ptx::tma_reduce_add_3d(&tm_skip, slab + q * 4096, ch0, t_cta0 + q * 32, b);
              ptx::bulk_commit_group();
            }
          }
          if (lane == 0) {
            ptx::bulk_wait_read_all();  // this warp's slabs are read: the G buffer may take the next conditioner tiles
            ptx::mbar_arrive(&bars->gc_free);
          }
        }
        if (!drained_said) {
          ptx::tc_fence_before();
          ptx::mbar_arrive_cluster(dr_leader + (kC == 128 ? pl : (uint32_t)j) * 8u);
        }
      }
      // the bias arrays are rewritten at the top of the next layer: every epilogue thread must be done reading them
      ptx::named_bar_sync(1, kSEpi);
      if (kC == 128) acc_col ^= 256u;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();  // the peer's smem / TMEM are in use by the leader's MMAs until here
  if (warp == 1) ptx::tmem_dealloc2(tmem, kSTmemCols);
}

}  // namespace svsk

using namespace svsk;

using StackKernelFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap,
                               DiffnetStackArgs);
static StackKernelFn stack_kernel_variant(bool use_p, bool dsmem, int C) {
  static const StackKernelFn table[8] = {
      diffnet_stack_kernel<false, false, 256>, diffnet_stack_kernel<true, false, 256>,
      diffnet_stack_kernel<false, true, 256>,  diffnet_stack_kernel<true, true, 256>,
      diffnet_stack_kernel<false, false, 128>, diffnet_stack_kernel<true, false, 128>,
      diffnet_stack_kernel<false, true, 128>,  diffnet_stack_kernel<true, true, 128>};
  return table[(use_p ? 1 : 0) | (dsmem ? 2 : 0) | (C == 128 ? 4 : 0)];
}

namespace svsk {  // diffnet_stack_duo_sm100.cu: C = 128 with two tiles per CTA pair
bool diffnet_stack_duo_applies(int C, int H);
int diffnet_stack_duo_fits(int B, int T);
int diffnet_stack_duo_launch(const svsk_diffnet_stack_params& p, void* stream);
}  // namespace svsk

static int stack_one_tile_fits(int B, int T, int C, int H);

// C = 128: two tiles per CTA pair as soon as the one-tile kernel cannot hold the whole batch on the device at once — a
// 6 x 6000 batch is 288 one-tile CTAs = two launches of 245 us in all, but 144 two-tile CTAs = one launch of 164 us.
// A batch that does fit stays with one tile per pair: each slot's chain is no shorter with two tiles, so on a device that
// is not full the kernel that spreads the tiles over twice as many SMs is the faster one (6 x 2000: 100 vs 140 us).
// SVSK_STACK_DUO=1 forces the two-tile kernel wherever it applies (tests, A/B), SVSK_STACK_NO_DUO=1 disables it.
static bool stack_use_duo(int B, int C, int H, int T) {
  if (!diffnet_stack_duo_applies(C, H)) return false;
  if (getenv("SVSK_STACK_DUO")) return true;
  return stack_one_tile_fits(B, T, C, H) != 1;
}

static int stack_smem(int C, int H, int* nentries_out, int* cond_resident_out = nullptr) {
  const int CB = C / 64, HB = H / 64;
  int gc_tiles = HB > CB ? HB : CB;
  if (gc_tiles < 4) gc_tiles = 4;
  int fixed = CB * kSWinBytes + gc_tiles * kSTile + 4 * 2 * C * (int)sizeof(float) + (int)sizeof(DiffnetStackBarriers) + 1024;
  // C = 128: resident conditioner tiles if that still leaves a ring of 5 (the depth the C = 256 kernel runs with)
  int resident = 0;
  if (C == 128 && HB > 0 && (kSSmemLimit - fixed - HB * kSTile) / kSTile >= 5) {
    resident = 1;
    fixed += HB * kSTile;
  }
  int nentries = (kSSmemLimit - fixed) / kSTile;
  if (nentries > kSMaxEntries) nentries = kSMaxEntries;
  *nentries_out = nentries;
  if (cond_resident_out) *cond_resident_out = resident;
  return fixed + nentries * kSTile;
}

// use_p: the conditioner projection is precomputed (no conditioner tiles in shared memory, none resident)
static int stack_prepare(int C, int H, int* nentries, int* smem_bytes, int* cond_resident = nullptr, bool use_p = false) {
  SVSK_REQUIRE(C == 128 || C == 256, SVSK_E_ARG, "diffnet_stack_bf16: C=%d (need 128 or 256)", C);
  SVSK_REQUIRE(H > 0 && H % 64 == 0 && H <= 512, SVSK_E_ARG, "diffnet_stack_bf16: H=%d (need a multiple of 64, at most 512)", H);
  *smem_bytes = stack_smem(C, use_p ? 0 : H, nentries, cond_resident);
  if (use_p && cond_resident) *cond_resident = 0;
  SVSK_REQUIRE(*nentries >= 3, SVSK_E_ARG, "diffnet_stack_bf16: not enough shared memory");
  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaSuccess;
    for (int v = 0; v < 8 && e == cudaSuccess; ++v) {
      StackKernelFn fn = stack_kernel_variant(v & 1, v & 2, (v & 4) ? 128 : 256);
      e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kSSmemLimit);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    }
    if (e != cudaSuccess) return fail((int)e, "diffnet_stack_bf16: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  return 0;
}

// One cluster per track (halo rows through distributed shared memory) when the track has at most 16 tiles: the cluster
// size is the next power of two (extra CTAs work on frames past the end: zeros in, nothing out).  Otherwise CTA pairs.
static int stack_cluster_size(int T) {
  const int tiles = 2 * ceil_div(T, 256);
  if (tiles > 16) return 2;
  int c = 2;
  while (c < tiles) c *= 2;
  return c;
}

static void stack_launch_config(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* attr, int B, int T, int smem_bytes, void* stream) {
  *cfg = cudaLaunchConfig_t{};
  const int csize = stack_cluster_size(T);
  cfg->gridDim = dim3(csize > 2 ? csize : 2 * ceil_div(T, 256), B);
  cfg->blockDim = dim3(kSThreads);
  cfg->dynamicSmemBytes = smem_bytes;
  cfg->stream = as_stream(stream);
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = csize;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  // cooperative: the driver starts the grid only when ALL its CTAs can be resident at once — the guarantee the
  // neighbour hand-shakes need even when other work shares the device
  // One cluster per track (DSMEM mode) has no hand-shake across clusters — the cluster launch itself co-schedules the
  // CTAs that talk to each other — so it needs no such guarantee (and no per-tile counters to reset): a plain cluster
  // launch measures 0.9 % faster per sampling pass (same-box A/B against a cooperative launch: 41.70 vs 42.07 ms).  (A programmatic-dependent-launch edge between the stack and the
  // step kernel was measured as well: no gain — the early CTAs of the next kernel only fragment the cluster placement.)
  // A track that is a single CTA pair (T <= 256) has no neighbour at all: same plain launch.
  const bool single_pair = ceil_div(T, 256) == 1;
  if (csize > 2 || single_pair) {
    cfg->attrs = attr;
    cfg->numAttrs = 1;
    return;
  }
  attr[1].id = cudaLaunchAttributeCooperative;
  attr[1].val.cooperative = 1;
  cfg->attrs = attr;
  cfg->numAttrs = 2;
}

static int stack_one_tile_fits(int B, int T, int C, int H) {
  int nentries = 0, smem_bytes = 0;
  if (stack_prepare(C, H, &nentries, &smem_bytes)) return 0;
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  stack_launch_config(&cfg, attr, B, T, smem_bytes, nullptr);
  int max_clusters = 0;
  if (cudaOccupancyMaxActiveClusters(&max_clusters, stack_kernel_variant(false, false, C), &cfg) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return (int)(cfg.gridDim.x / attr[0].val.clusterDim.x) * B <= max_clusters ? 1 : 0;
}

extern "C" int svsk_diffnet_stack_fits(int B, int T, int C, int H) {
  int rc = require_sm100();
  if (rc) return -1;
  if (B <= 0 || T <= 0 || B > 65535) return 0;
  if (stack_use_duo(B, C, H, T)) return diffnet_stack_duo_fits(B, T);
  return stack_one_tile_fits(B, T, C, H);
}

extern "C" int svsk_diffnet_stack_uses_pcond(int B, int T, int C, int H) {
  int rc = require_sm100();
  if (rc) return -1;
  if (B <= 0 || T <= 0 || B > 65535 || getenv("SVSK_STACK_NO_PCOND")) return 0;
  if (stack_use_duo(B, C, H, T)) return 0;
  return stack_one_tile_fits(B, T, C, H);
}

// [L*NB][B*T][256] (gate 128 | filter 128 per block) -> gate half channel-last [B][L][T][C], filter half in the epilogue
// threads' order [B][tiles][L][NB][8][128][16]; one CTA per (128-frame tile, layer-block), 16 bytes per thread and step.
__global__ void __launch_bounds__(256) diffnet_pcond_pack_kernel(const uint4* __restrict__ p, uint4* __restrict__ pg,
                                                                 uint4* __restrict__ pf, int B, int T, int L, int NB, int tiles) {
  const int lj = blockIdx.y, l = lj / NB, j = lj - l * NB;
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles;
  const int C = NB * 128;
  const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
  const uint4* src = p + ((size_t)lj * B + b) * T * 32;                                  // 32 uint4 per frame
  uint4* pf_blk = pf + (((size_t)(b * tiles + tile) * L + l) * NB + j) * 2048;
  for (int q = threadIdx.x; q < 128 * 32; q += 256) {
    const int row = q >> 5, c16 = q & 31;  // 8 columns c16*8 .. +7 of frame tile*128 + row
    const int t = tile * 128 + row;
    const uint4 v = t < T ? src[(size_t)t * 32 + c16] : zero;
    if (c16 < 16) {
      if (t < T) pg[(((size_t)b * L + l) * T + t) * (C / 8) + j * 16 + c16] = v;
    } else {
      const int cc = c16 - 16;             // filter columns cc*8 .. +7: chunk cc / 2, half cc & 1
      pf_blk[((cc >> 1) * 128 + row) * 2 + (cc & 1)] = v;
    }
  }
}

extern "C" int svsk_diffnet_pcond_pack_bf16(const void* p, void* pcond_gate, void* pcond_filt, int B, int T, int L, int C,
                                            void* stream) {
  SVSK_REQUIRE(p && pcond_gate && pcond_filt, SVSK_E_ARG, "diffnet_pcond_pack_bf16: null tensor");
  SVSK_REQUIRE(C == 128 || C == 256, SVSK_E_ARG, "diffnet_pcond_pack_bf16: C=%d (need 128 or 256)", C);
  SVSK_REQUIRE(B > 0 && T > 0 && L >= 1 && L <= kSMaxLayers, SVSK_E_ARG, "diffnet_pcond_pack_bf16: bad B/T/L");
  SVSK_REQUIRE(((uintptr_t)p % 16) == 0 && ((uintptr_t)pcond_gate % 16) == 0 && ((uintptr_t)pcond_filt % 16) == 0, SVSK_E_ALIGN,
               "diffnet_pcond_pack_bf16: tensors must be 16-byte aligned");
  const int NB = C / 128, tiles = 2 * ceil_div(T, 256);
  SVSK_REQUIRE((long long)B * tiles < (1ll << 31) && L * NB <= 65535, SVSK_E_ARG, "diffnet_pcond_pack_bf16: grid too large");
  int rc = require_sm100();
  if (rc) return rc;
  diffnet_pcond_pack_kernel<<<dim3((unsigned)(B * tiles), (unsigned)(L * NB)), 256, 0, as_stream(stream)>>>(
      static_cast<const uint4*>(p), static_cast<uint4*>(pcond_gate), static_cast<uint4*>(pcond_filt), B, T, L, NB, tiles);
  return check_launch("diffnet_pcond_pack_bf16");
}

extern "C" int svsk_diffnet_stack_bf16(const svsk_diffnet_stack_params* pp, void* stream) {
  SVSK_REQUIRE(pp != nullptr, SVSK_E_ARG, "diffnet_stack_bf16: null params");
  const svsk_diffnet_stack_params& p = *pp;
  SVSK_REQUIRE(p.xb_in && p.edge0 && p.edge1 && p.skip32 && p.cond && p.w1p && p.woutp && p.stepbias && p.bout && p.flags &&
                   p.dilation,
               SVSK_E_ARG, "diffnet_stack_bf16: null tensor");
  SVSK_REQUIRE(p.xb_in != p.edge0 && p.xb_in != p.edge1 && p.edge0 != p.edge1, SVSK_E_ARG,
               "diffnet_stack_bf16: xb_in / edge0 / edge1 must be three different buffers");
  SVSK_REQUIRE(p.L >= 1 && p.L <= kSMaxLayers, SVSK_E_ARG, "diffnet_stack_bf16: L=%d (1..%d)", p.L, kSMaxLayers);
  SVSK_REQUIRE(p.B > 0 && p.B <= 65535 && p.T > 0, SVSK_E_ARG, "diffnet_stack_bf16: bad B/T");
  for (int l = 0; l < p.L; ++l)
    SVSK_REQUIRE(p.dilation[l] >= 1 && p.dilation[l] <= kSHalo, SVSK_E_ARG,
                 "diffnet_stack_bf16: layer %d dilation %d outside the resident window (1..%d)", l, p.dilation[l], kSHalo);
  SVSK_REQUIRE(p.stepbias_layer_stride >= 6 * p.C && (p.stepbias_batch_stride == 0 || p.stepbias_batch_stride >= 6 * p.C),
               SVSK_E_ARG, "diffnet_stack_bf16: stepbias strides");
  SVSK_REQUIRE(((uintptr_t)p.skip32 % 16) == 0 && ((uintptr_t)p.edge0 % 16) == 0 && ((uintptr_t)p.edge1 % 16) == 0, SVSK_E_ALIGN,
               "diffnet_stack_bf16: skip32 / edge0 / edge1 must be 16-byte aligned");
  int rc = require_sm100();
  if (rc) return rc;
  SVSK_REQUIRE((p.pcond_gate == nullptr) == (p.pcond_filt == nullptr), SVSK_E_ARG,
               "diffnet_stack_bf16: pcond_gate and pcond_filt go together");
  SVSK_REQUIRE(((uintptr_t)p.pcond_gate % 16) == 0 && ((uintptr_t)p.pcond_filt % 16) == 0, SVSK_E_ALIGN,
               "diffnet_stack_bf16: pcond_gate / pcond_filt must be 16-byte aligned");
  if (stack_use_duo(p.B, p.C, p.H, p.T)) return diffnet_stack_duo_launch(p, stream);
  const bool use_p = p.pcond_gate != nullptr && !getenv("SVSK_STACK_NO_PCOND");
  int nentries = 0, smem_bytes = 0, cond_resident = 0;
  if ((rc = stack_prepare(p.C, p.H, &nentries, &smem_bytes, &cond_resident, use_p))) return rc;

  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  stack_launch_config(&cfg, attr, p.B, p.T, smem_bytes, stream);
  int max_clusters = 0;
  cudaError_t oe = cudaOccupancyMaxActiveClusters(&max_clusters, stack_kernel_variant(false, false, p.C), &cfg);
  if (oe != cudaSuccess) return fail((int)oe, "diffnet_stack_bf16: cudaOccupancyMaxActiveClusters: %s", cudaGetErrorString(oe));
  const int n_clusters = (int)(cfg.gridDim.x / attr[0].val.clusterDim.x) * p.B;
  SVSK_REQUIRE(n_clusters <= max_clusters, SVSK_E_ARG,
               "diffnet_stack_bf16: %d clusters of %d CTAs do not fit the device at once (%d); run the layers with "
               "svsk_diffnet_block3_bf16", n_clusters, (int)attr[0].val.clusterDim.x, max_clusters);

  // one cluster per track: each CTA pair fetches (and multicasts) 1/n_pairs of every weight half-tile
  const uint32_t csz = attr[0].val.clusterDim.x;
  const uint32_t w_box_rows = (csz > 2 && stack_multicast(use_p, p.C)) ? 128u / (csz / 2) : 128u;
  CUtensorMap tm_xw0, tm_e0, tm_e1, tm_cond, tm_w1, tm_wout, tm_skip;
  {
    uint64_t dims[3] = {(uint64_t)p.C, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.C * 2, (uint64_t)p.T * p.C * 2};
    uint32_t boxw[3] = {64, (uint32_t)kSWinRows, 1};
    uint32_t boxe[3] = {64, (uint32_t)kSHalo, 1};
    if ((rc = make_tmap_bf16(&tm_xw0, p.xb_in, 3, dims, str, boxw))) return rc;
    if ((rc = make_tmap_bf16(&tm_e0, p.edge0, 3, dims, str, boxe))) return rc;
    if ((rc = make_tmap_bf16(&tm_e1, p.edge1, 3, dims, str, boxe))) return rc;
    uint64_t str4[2] = {(uint64_t)p.C * 4, (uint64_t)p.T * p.C * 4};
    uint32_t box4[3] = {32, 32, 1};  // one warp's 32 rows of a 32-column skip slab
    if ((rc = make_tmap_f32(&tm_skip, p.skip32, 3, dims, str4, box4))) return rc;
  }
  if (use_p) {  // gate half of the precomputed projection, [B * L][T][C]
    uint64_t dims[3] = {(uint64_t)p.C, (uint64_t)p.T, (uint64_t)p.B * p.L};
    uint64_t str[2] = {(uint64_t)p.C * 2, (uint64_t)p.T * p.C * 2};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_cond, p.pcond_gate, 3, dims, str, box))) return rc;
  } else {
    uint64_t dims[3] = {(uint64_t)p.H, (uint64_t)p.T, (uint64_t)p.B};
    uint64_t str[2] = {(uint64_t)p.H * 2, (uint64_t)p.T * p.H * 2};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_bf16(&tm_cond, p.cond, 3, dims, str, box))) return rc;
  }
  {
    const uint64_t K1 = 3 * (uint64_t)p.C + p.H;
    uint64_t dims[3] = {K1, (uint64_t)2 * p.C, (uint64_t)p.L};
    uint64_t str[2] = {K1 * 2, K1 * 2 * 2 * p.C};
    uint32_t box[3] = {64, w_box_rows, 1};
    if ((rc = make_tmap_bf16(&tm_w1, p.w1p, 3, dims, str, box))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)p.C, (uint64_t)2 * p.C, (uint64_t)p.L};
    uint64_t str[2] = {(uint64_t)p.C * 2, (uint64_t)p.C * 2 * 2 * p.C};
    uint32_t box[3] = {64, w_box_rows, 1};
    if ((rc = make_tmap_bf16(&tm_wout, p.woutp, 3, dims, str, box))) return rc;
  }

  DiffnetStackArgs a;
  a.stepbias = p.stepbias;
  a.bout = p.bout;
  a.flags = p.flags;
  a.dsmem_halo = attr[0].val.clusterDim.x > 2 ? 1 : 0;
  a.B = p.B; a.T = p.T; a.C = p.C; a.H = p.H; a.L = p.L;
  a.sb_batch_stride = p.stepbias_batch_stride;
  a.sb_layer_stride = p.stepbias_layer_stride;
  a.init_skip = p.init_skip;
  a.nentries = nentries;
  a.cond_resident = cond_resident;
  a.use_p = use_p ? 1 : 0;
  a.pfilt = static_cast<const uint4*>(p.pcond_filt);
  a.tiles_per_track = 2 * ceil_div(p.T, 256);
  for (int l = 0; l < kSMaxLayers; ++l) a.dilation[l] = l < p.L ? p.dilation[l] : 1;

  cudaError_t e = cudaSuccess;
  if (!a.dsmem_halo) {  // the per-tile layer counters are only used when edge rows travel through global memory
    e = cudaMemsetAsync(p.flags, 0, sizeof(int) * (size_t)p.B * a.tiles_per_track, as_stream(stream));
    if (e != cudaSuccess) return fail((int)e, "diffnet_stack_bf16: flag reset: %s", cudaGetErrorString(e));
  }
  e = cudaLaunchKernelEx(&cfg, stack_kernel_variant(use_p, a.dsmem_halo != 0, p.C), tm_xw0, tm_e0, tm_e1, tm_cond, tm_w1, tm_wout,
                         tm_skip, a);
  if (e != cudaSuccess) return fail((int)e, "diffnet_stack_bf16: launch: %s", cudaGetErrorString(e));
  return check_launch("diffnet_stack_bf16");
}
