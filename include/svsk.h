/*
 * svsk.h — C ABI of libsvsk.so: hand-written sm_100a CUDA kernels for the gated dilated-Conv1d
 * residual stacks of sarulab-speech/ensemble_svs_with_interactions (NNSVS-derived).
 *
 * The reference has no FFI of its own (it is pure Python/PyTorch, SURVEY.md §8b): the seam is the
 * nn.Module protocol.  Each entry point below therefore cites the reference *function* it replaces
 * (paths relative to the reference root).  The drop-in nn.Modules in
 * ensemble_svs_with_interactions_b200/ bind these symbols with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *  - the caller owns every buffer (inputs, outputs, workspace); kernels never allocate or synchronise;
 *  - every call only enqueues work on `stream` (a cudaStream_t passed as void*) and is CUDA-graph capturable;
 *  - return value: 0 = ok; <0 = SVSK_E* argument/arch error detected before launch; >0 = cudaError_t;
 *    svsk_last_error() returns a thread-local message for the last non-zero return;
 *  - there is no CPU path: on a non-sm_100 device the tensor-core entry points return SVSK_E_ARCH;
 *  - layouts: "NCT" = [B][C][T] fp32 (the reference's layout); "NTC" = [B][T][C] channel-last
 *    (bf16 MMA operands, fp32 residual/skip masters).
 */
#ifndef SVSK_H_
#define SVSK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVSK_VERSION 100

#if defined(__GNUC__)
#define SVSK_API __attribute__((visibility("default")))
#else
#define SVSK_API
#endif

enum {
  SVSK_OK = 0,
  SVSK_E_ARG = -1,      /* bad shape / null pointer / unsupported combination */
  SVSK_E_ALIGN = -2,    /* pointer or stride alignment */
  SVSK_E_ARCH = -3,     /* device is not sm_100 */
  SVSK_E_DRIVER = -4,   /* could not obtain cuTensorMapEncodeTiled */
  SVSK_E_WORKSPACE = -5 /* workspace too small */
};

/* padding / tap-index modes of svsk_conv1d_f32 */
enum {
  SVSK_PAD_ZEROS = 0,     /* 0 outside [0,T)                       (nn.Conv1d default; DiffNet, WaveNet) */
  SVSK_PAD_REFLECT = 1,   /* i<0 -> -i ; i>=T -> 2(T-1)-i          (uSFGAN FixedBlock)                    */
  SVSK_PAD_REPLICATE = 2, /* clamp                                  (uSFGAN PeriodicityEstimator)          */
  SVSK_PAD_VALID = 3,     /* no padding: T_out = T_in-(k-1)*dil     (uSFGAN upsample conv_in)              */
  SVSK_PAD_INDEXED = 4    /* k==3: taps at idx_past[b,t], t, idx_future[b,t]; index<0 -> 0 (AdaptiveBlock) */
};

enum { SVSK_ACT_NONE = 0, SVSK_ACT_RELU = 1, SVSK_ACT_SIGMOID = 2, SVSK_ACT_MISH = 3 };

/* gate orders of svsk_gated_act_f32 */
enum {
  SVSK_GATE_SIGMOID_TANH = 0, /* sigmoid(first half) * tanh(second half): DiffNet (denoiser.py:60-61)        */
  SVSK_GATE_TANH_SIGMOID = 1  /* tanh(first half) * sigmoid(second half): WaveNet / uSFGAN                   */
};

SVSK_API const char* svsk_last_error(void);
SVSK_API int svsk_version(void);
/* 0 iff `device` is an sm_100 (B200) part; SVSK_E_ARCH otherwise; >0 cudaError_t when no driver/GPU. */
SVSK_API int svsk_device_check(int device);

/* ------------------------------------------------------------------------------------------------
 * fp32 exact path (CUDA cores), NCT layout.
 * ------------------------------------------------------------------------------------------------ */

/* General Conv1d as a sum of taps.  Replaces every nn.Conv1d / Conv1d1x1 / nn.Linear call on the path:
 *   nnsvs/diffsinger/denoiser.py:43-52,80,97-98 ; nnsvs/usfgan/layers/residual_block.py:104-120,187-201,358-366 ;
 *   nnsvs/usfgan/layers/upsample.py:165-167 ; nnsvs/wavenet/modules.py:46-62 ; nnsvs/wavenet/wavenet.py:33,52-57.
 *   y[b,co,t] = act( ( bias[co] + sum_j sum_ci w[co,ci,j] * X(b,ci,src_j(t)) + residual[b,co,t] ) * out_scale )
 *   src_j(t)  = t + (j - tap_origin) * dilation, resolved by pad_mode;
 *   X(b,ci,u) = in_relu?relu(x):x  (+ in_bias[b,ci] when u is in range: DiffNet's x + step embedding, added
 *               BEFORE zero padding, denoiser.py:57-59).
 *   accumulate != 0: y += (...) instead of y = (...).  T is the OUTPUT length. */
typedef struct svsk_conv1d_f32_params {
  const float* x;        /* [B][Cin][T_in]; T_in == T except SVSK_PAD_VALID */
  const float* w;        /* [Cout][Cin][ksize] */
  const float* bias;     /* [Cout] or NULL */
  const float* in_bias;  /* [B][Cin] or NULL */
  const float* residual; /* [B][Cout][T] or NULL (may alias y) */
  const int32_t* idx_past;   /* [B][T] (SVSK_PAD_INDEXED) */
  const int32_t* idx_future; /* [B][T] (SVSK_PAD_INDEXED) */
  float* y;              /* [B][Cout][T] */
  int32_t B, Cin, Cout, T;
  int32_t ksize, dilation, tap_origin, pad_mode;
  int32_t accumulate, act, in_relu;
  float out_scale;
} svsk_conv1d_f32_params;
SVSK_API int svsk_conv1d_f32(const svsk_conv1d_f32_params* p, void* stream);

/* nn.Linear on small batches, y[b][co] = act(bias[co] + sum_ci w[co][ci] x[b][ci]) — the step-embedding MLP and the
 * per-layer diffusion_projection (denoiser.py:49,56,84-86,113-114). */
SVSK_API int svsk_linear_f32(const float* x, const float* w, const float* bias, float* y, int Bt, int Cin, int Cout, int act,
                             void* stream);

/* z[b,h,t] = gate(y[b,h,t], y[b,H+h,t]).  denoiser.py:60-61 ; residual_block.py:140-149 ; modules.py:104-112 */
SVSK_API int svsk_gated_act_f32(const float* y, float* z, int B, int H, int T, int order, void* stream);

/* DiffNet block tail, denoiser.py:63-66:  x = (x + o[:, :C]) / sqrt(2) ;  skip (+)= o[:, C:]  (skip = when init_skip) */
SVSK_API int svsk_diffnet_residual_skip_f32(const float* o, float* x, float* skip, int B, int C, int T, int init_skip,
                                   void* stream);

/* y = alpha * act(x) elementwise over n elements (skip-sum / sqrt(L), Mish of the step MLP ...). */
SVSK_API int svsk_scale_act_f32(const float* x, float* y, size_t n, float alpha, int act, void* stream);

/* Sinusoidal step embedding, denoiser.py:14-26: out[b] = cat(sin(t_b f), cos(t_b f)), f_i = 10000^(-i/(dim/2-1)). */
SVSK_API int svsk_sinusoidal_embedding_f32(const int64_t* t, float* out, int B, int dim, void* stream);

/* One ancestral DDPM update, diffusion.py:164-204 (p_sample after the denoiser call), any layout (flat per batch):
 *   x0 = clamp(sra[t] x - srm1[t] eps, +-1) ; mean = c1[t] x0 + c2[t] x ; out = mean + [t>0] exp(.5 plv[t]) z
 * tables are the reference's registered fp32 buffers (diffusion.py:112-145); t is [B] int64. */
SVSK_API int svsk_ddpm_update_f32(const float* x, const float* eps, const float* z, float* out, const int64_t* t,
                         const float* sqrt_recip_alphas_cumprod, const float* sqrt_recipm1_alphas_cumprod,
                         const float* posterior_mean_coef1, const float* posterior_mean_coef2,
                         const float* posterior_log_variance_clipped, int B, size_t per_batch, int clip_denoised,
                         void* stream);

/* q_sample, diffusion.py:261-267: out = sac[t] x0 + somac[t] noise. */
SVSK_API int svsk_q_sample_f32(const float* x0, const float* noise, float* out, const int64_t* t,
                      const float* sqrt_alphas_cumprod, const float* sqrt_one_minus_alphas_cumprod, int B,
                      size_t per_batch, void* stream);

/* PLMS transfer get_x_pred, diffusion.py:213-230: out = x + x_delta(alphas_cumprod[t], alphas_cumprod[max(t-interval,0)]). */
SVSK_API int svsk_plms_transfer_f32(const float* x, const float* noise_t, float* out, const int64_t* t, int interval,
                           const float* alphas_cumprod, int B, size_t per_batch, void* stream);

/* out = sum_i coef[i] * in[i] over n elements, 1 <= n_in <= 4 (PLMS multistep combination, diffusion.py:236-256). */
SVSK_API int svsk_lincomb_f32(const float* const* in, const float* coef, int n_in, float* out, size_t n, void* stream);

/* Pitch-dependent tap indices, nnsvs/usfgan/utils/index.py:12-54 (bit-faithful fp32 rounding):
 *   past[b,t] = rint(-(d*dil) + (t-T)) + T   (-1 when < 0)
 *   future[b,t] = rint((d*dil) + t)           (-1 when >= T)          d is [B][T] (the (B,1,T) tensor). */
SVSK_API int svsk_pd_index(const float* d, int32_t* idx_past, int32_t* idx_future, int B, int T, int dilation, void* stream);

/* uSFGAN upsample stage, upsample.py:15-44,87-101: nearest stretch by `scale` then the (1, 2*scale+1) smoothing
 * filter (zero padding `scale`), same taps for every channel.  in [R][Tin] -> out [R][Tin*scale], R = B*C rows. */
SVSK_API int svsk_upsample_smooth_f32(const float* in, const float* taps, float* out, int R, int Tin, int scale, void* stream);

/* Periodicity mix, generator.py:505-507: h2 = a*h ; n2 = (1-a)*n ; s = h2 + n2   (h2/n2 may be NULL). */
SVSK_API int svsk_periodic_mix_f32(const float* a, const float* h, const float* n, float* s, float* h2, float* n2, size_t cnt,
                          void* stream);

/* ------------------------------------------------------------------------------------------------
 * layout / precision conversion between the two paths
 * ------------------------------------------------------------------------------------------------ */
/* [B][C][T] fp32 -> [B][T][Cp] bf16 (channels >= C zero-filled up to Cp) and optionally the fp32 NTC master. */
SVSK_API int svsk_nct_to_ntc(const float* x, void* out_bf16, float* out_f32, int B, int C, int T, int Cp, void* stream);
/* [B][T][Cp] fp32 -> [B][C][T] fp32 (first C channels), scaled by alpha. */
SVSK_API int svsk_ntc_to_nct_f32(const float* x, float* y, int B, int C, int T, int Cp, float alpha, void* stream);
/* flat fp32 -> bf16 with scale and optional ReLU (skip-sum / sqrt(L) before the tail GEMM). */
SVSK_API int svsk_cast_scale_bf16(const float* x, void* y_bf16, size_t n, float alpha, int relu, void* stream);

/* ------------------------------------------------------------------------------------------------
 * bf16 tensor-core path (tcgen05 + TMEM + TMA), NTC layout.  sm_100a only.
 * ------------------------------------------------------------------------------------------------ */

/* Fused DiffNet residual block — replaces ResidualBlock.forward, nnsvs/diffsinger/denoiser.py:54-66, one launch:
 *   D1 = W1p . [x(t-d) ; x(t) ; x(t+d) ; cond(t)]           implicit GEMM, K = 3C + H, zero padding by TMA OOB fill
 *   D1 += stepbias (per tap, masked at the sequence ends = exact `x + diffusion_step` before zero padding)
 *   G  = sigmoid(D1[gate rows]) * tanh(D1[filter rows])       TMEM -> registers -> swizzled smem (bf16)
 *   D2 = Woutp . G + bout                                     second GEMM from smem
 *   x32 <- (x32 + D2[:C]) / sqrt(2)  (fp32 master, in place) ; xb_out <- bf16(x32) ; skip32 (+)= D2[C:]
 * Weights are pre-packed by svsk_diffnet_pack_block (row permutation: 128-row gate block then its filter block).
 * Constraints: C % 128 == 0, C <= 256, H % 64 == 0, T >= 1.  xb_in and xb_out must differ (neighbour tiles read
 * xb_in halos).  stepbias is [B or 1][3][2C] fp32 in PACKED row order; stepbias_batch_stride = 0 broadcasts. */
typedef struct svsk_diffnet_block_params {
  const void* xb_in;   /* [B][T][C] bf16 */
  void* xb_out;        /* [B][T][C] bf16 */
  float* x32;          /* [B][T][C] fp32, in place */
  float* skip32;       /* [B][T][C] fp32, in place */
  const void* cond;    /* [B][T][H] bf16 */
  const void* w1p;     /* [2C][3C+H] bf16 packed */
  const void* woutp;   /* [2C][C] bf16 packed */
  const float* stepbias; /* [.][3][2C] */
  const float* bout;   /* [2C] fp32: [0,C) residual rows, [C,2C) skip rows */
  int32_t B, T, C, H;
  int32_t dilation;
  int32_t stepbias_batch_stride; /* in floats; 0 = same for every batch row */
  int32_t init_skip;   /* 1: skip32 = ..., 0: skip32 += ... */
  int32_t write_x;     /* 0 on the last layer (x is dead after it, denoiser.py:117-120) */
  int32_t reserved0;   /* must be 0 (was: time tile of the retired single-CTA kernel) */
} svsk_diffnet_block_params;

/* The per-layer kernel: CTA pair (tcgen05 cta_group::2, clusters of 2), time is the MMA M dimension (256 frames per
 * pair), with a resident activation window: the three taps of the dilated conv (denoiser.py:33-35,58) are one
 * (128 + 16)-row shared-memory tile per 64 channels addressed at row offsets -d / 0 / +d, so activations are read once
 * per tile and only weights stream through the ring.  Requires dilation <= 8 (the reference's dilation_cycle_length = 4
 * gives 1, 2, 4, 8; wider cycles are served by the fp32 kernels — DiffNet(precision="auto") selects them) and x32 /
 * skip32 / xb_out 16-byte aligned; x32 is not used (the residual stream is carried in bf16).
 * Launched with programmatic stream serialization: the packed weights w1p / woutp are read BEFORE the kernel waits for
 * its predecessor in the stream, so they must not be written by the kernel launched immediately before this one
 * (pack once, up front); every other operand may be.  Used when a track is too long for svsk_diffnet_stack_bf16. */
SVSK_API int svsk_diffnet_block3_bf16(const svsk_diffnet_block_params* p, void* stream);

/* All L residual blocks of one denoiser call in ONE launch (the loop denoiser.py:114-118): every CTA pair keeps its
 * 256-frame tile for all layers, the residual epilogue rewrites the activation window in place, and only the 8 edge
 * rows per side travel between neighbouring tiles (through edge0 / edge1 and a per-tile layer counter).  Operands are
 * the per-layer ones stacked along a leading layer dimension:
 *   w1p [L][2C][3C+H], woutp [L][2C][C] (svsk_diffnet_pack_block per layer), bout [L][2C],
 *   stepbias: row of layer l and batch row b at stepbias + b*stepbias_batch_stride + l*stepbias_layer_stride (floats),
 *   dilation[L] (host array, each 1..8), xb_in [B][T][C] bf16 = input of layer 0 (never written),
 *   edge0 / edge1 [B][T][C] bf16 scratch (only edge rows are touched; contents need not be initialised),
 *   flags: B * 2*ceil(T/256) ints of scratch (reset by this call), skip32 [B][T][C] fp32 = sum of the L skip outputs
 *   (stored if init_skip, else accumulated).  The residual stream after the last layer is not produced (it is dead,
 *   denoiser.py:117-120).
 * All CTA pairs must be resident at once (the launch is cooperative, so the driver guarantees it or waits):
 * svsk_diffnet_stack_fits(B,T,C,H) returns 1 if the device can hold them, 0 if not (then split the batch into groups of
 * tracks that fit, or run the layers one by one with svsk_diffnet_block3_bf16), -1 without an sm_100 device.
 * Tracks of at most 2048 frames run as one thread-block cluster each (edge rows through distributed shared memory,
 * weight tiles TMA-multicast); longer tracks exchange edge rows through edge0 / edge1 and the flags.
 * pcond_gate / pcond_filt (optional, both or neither): the conditioner projection of every layer,
 * conditioner_projection(cond) (denoiser.py:59), computed ONCE for a whole sampling run — cond does not change between
 * the K calls of diffusion.py:302-336 — and laid out by svsk_diffnet_pcond_pack_bf16.  With them the kernel skips the H
 * conditioner k-blocks of every layer's first GEMM (K = 3C instead of 3C + H) and adds the projection in the gating
 * epilogue; without them (a single denoiser call) the projection is part of the GEMM as before.  `cond` is required
 * either way (the two-tiles-per-pair kernel for C = 128 always projects in the GEMM). */
typedef struct svsk_diffnet_stack_params {
  const void* xb_in;
  void* edge0;
  void* edge1;
  float* skip32;
  const void* cond;      /* [B][T][H] bf16 */
  const void* w1p;
  const void* woutp;
  const float* stepbias;
  const float* bout;
  int32_t* flags;
  const int32_t* dilation; /* host pointer, L entries */
  int32_t B, T, C, H, L;
  int32_t stepbias_batch_stride;  /* floats; 0 = same for every batch row */
  int32_t stepbias_layer_stride;  /* floats; >= 6C */
  int32_t init_skip;
  const void* pcond_gate; /* [B][L][T][C] bf16 or NULL */
  const void* pcond_filt; /* [B][2*ceil(T/256)][L][2C/256][8][128][16] bf16 or NULL */
} svsk_diffnet_stack_params;
SVSK_API int svsk_diffnet_stack_bf16(const svsk_diffnet_stack_params* p, void* stream);
SVSK_API int svsk_diffnet_stack_fits(int B, int T, int C, int H);
/* 1 if svsk_diffnet_stack_bf16 would use pcond_gate / pcond_filt for this shape (the one-tile-per-pair kernel runs and
 * holds the batch), 0 if they would be ignored, -1 without an sm_100 device. */
SVSK_API int svsk_diffnet_stack_uses_pcond(int B, int T, int C, int H);
/* p[blk][n][0..255] = cond[n][:] . wcp[blk * 256 + r][:] for blk = 0 .. nblk-1 in one launch: conditioner_projection(cond)
 * of every layer and 256-row output block (denoiser.py:59), computed once for a sampling run.  cond [N][H] bf16 (N = B*T
 * frames), wcp [nblk * 256][H] bf16 (the conditioner columns of w1p, block after block), p [nblk][N][256] bf16. */
SVSK_API int svsk_diffnet_cond_project_bf16(const void* cond, const void* wcp, void* p, long long N, int H, int nblk,
                                            void* stream);
/* Lays out the per-layer conditioner projections for svsk_diffnet_stack_bf16.  p [L * 2C/256][B*T][256] bf16: for
 * layer l and 256-column output block j of the first GEMM, the projection of every frame in PACKED column order
 * (columns 0..127 = gate rows, 128..255 = filter rows of the block: cond . w1p[l][j*256 + n][3C:]^T).
 *   pcond_gate [B][L][T][C]: the gate half, channel-last (TMA-loaded into the tile the gate output overwrites);
 *   pcond_filt [B][2*ceil(T/256)][L][2C/256][8][128][16]: the filter half in the order the epilogue threads read it
 *   (128-frame tile, 16-column chunk, frame, column); frames >= T are zero. */
SVSK_API int svsk_diffnet_pcond_pack_bf16(const void* p, void* pcond_gate, void* pcond_filt, int B, int T, int L, int C,
                                          void* stream);

/* Everything between two residual-stack launches of a DDPM sampling step in one launch per 128-frame tile:
 *   eps = output_projection(relu(skip_projection(skip32 * skip_scale)))      denoiser.py:120-123
 *   x   = p_sample update of x with eps, noise z and the step's schedule coefficients, in place (the arithmetic of
 *         svsk_ddpm_update_f32; diffusion.py:164-204)
 *   xb_out = relu(input_projection(x)) as bf16 [B][T][C] for the next denoiser call (denoiser.py:109-112); pass
 *         xb_out = NULL on the last step (w_in / b_in are then unused).
 * NTC fp32 state tensors [B][T][Mp] (Mp = M rounded up to 16; padded channels carry zeros through zero weights and
 * biases), bf16 weights w_skip [C][C], w_out [Mp][C], w_in [C][Mp], fp32 biases (b_out has Mp entries), t [B] int64.
 * eps_out (optional) receives eps. */
typedef struct svsk_diffnet_step_params {
  const float* skip32;
  float* x32s;
  const float* z;
  float* eps_out;
  void* xb_out;
  const void* w_skip;
  const void* w_out;
  const void* w_in;
  const float* b_skip;
  const float* b_out;
  const float* b_in;
  const int64_t* t;
  const float* sqrt_recip_alphas_cumprod;
  const float* sqrt_recipm1_alphas_cumprod;
  const float* posterior_mean_coef1;
  const float* posterior_mean_coef2;
  const float* posterior_log_variance_clipped;
  float skip_scale;
  int32_t B, T, C, Mp, clip_denoised;
} svsk_diffnet_step_params;
SVSK_API int svsk_diffnet_step_bf16(const svsk_diffnet_step_params* p, void* stream);

/* The whole UpsampleNetwork (nnsvs/usfgan/layers/upsample.py:61-128) in one pass from frame rate to sample rate, written
 * channel-last: c [B][A][F] fp32 (the output of conv_in) -> out [B][T = F * prod(scales)][Ap] as bf16 and/or fp32
 * (Ap >= A, a multiple of 8; channels A..Ap-1 are zero).  taps: the (2 s_k + 1)-tap smoothing filters of the stages,
 * concatenated; scales: host array.  Same arithmetic as n_stages calls of svsk_upsample_smooth_f32 up to fp32 summation
 * order, including the zero padding of every stage at the sequence ends.  Needs 2 <= s_k <= 16, A <= 128 and
 * 127 / prod(scales) + 2 n_stages + 4 <= 48. */
SVSK_API int svsk_upsample_fused(const float* c, const float* taps, const int32_t* scales, int n_stages, int B, int A, int F,
                                 void* out_bf16, float* out_f32, int Ap, void* stream);

/* Pointwise 1 -> C Conv1d straight to NTC bf16 (generator.py conv_first_sine / conv_first_noise):
 * out[b][t][c] = w[c] * x[b * x_batch_stride + t] + bias[c]. */
SVSK_API int svsk_expand1_bf16(const float* x, long long x_batch_stride, const float* w, const float* bias, void* out, int B,
                               int T, int C, void* stream);

/* Pack one block's weights (fp32, reference state_dict layout) for svsk_diffnet_block_bf16.
 *   dilated_w [2C][C][3], cond_w [2C][H][1], out_w [2C][C][1]  ->  w1p [2C][3C+H] bf16, woutp [2C][C] bf16.
 * Row r of the reference maps to packed row perm(r): gate rows of channel block q at 256q..256q+127, filter rows at
 * 256q+128..256q+255.  Also applies to the stepbias/bias vectors: svsk_diffnet_packed_row(). */
SVSK_API int svsk_diffnet_pack_block(const float* dilated_w, const float* cond_w, const float* out_w, void* w1p, void* woutp,
                            int C, int H, void* stream);
SVSK_API int svsk_diffnet_packed_row(int reference_row, int C);

/* Fused uSFGAN / QPPWG residual block — replaces FixedBlock.forward / AdaptiveBlock.forward (+ pd_indexing),
 * nnsvs/usfgan/layers/residual_block.py:123-157,198-234 and nnsvs/usfgan/utils/index.py:12-54, one launch per block:
 *   D1 = W1p . [x(tap0) ; x(t) ; x(tap2) ; aux(t)] ; z = tanh(D1[:64]+b) * sigmoid(D1[64:]+b) ; D2 = Woutp . z
 *   xb_out(t) = (D2 + bout + xb_in(t)) * out_scale
 * taps: adaptive == 0: t -/+ dilation with reflect padding (needs T > dilation);
 *       adaptive != 0: idx_past[b,t] / idx_future[b,t] from svsk_pd_index (-1 = zero tap).
 * Shapes: residual 64 / gate 128 channels (the recipes' widths), aux A <= 320 with A % 8 == 0, NTC bf16 activations.
 * Persistent kernel: weights stay resident in shared memory, activations stream through a TMA / cp.async ring. */
typedef struct svsk_usfgan_block_params {
  const void* xb_in;   /* [B][T][64] bf16 */
  void* xb_out;        /* [B][T][64] bf16, != xb_in */
  const void* aux;     /* [B][T][A] bf16 */
  const void* w1p;     /* [128][192 + ceil64(A)] bf16 packed by svsk_usfgan_pack_block */
  const void* woutp;   /* [64][64] bf16 */
  const float* bias1;  /* [128] conv bias (adaptive: convP + convC + convF biases) */
  const float* bout;   /* [64] */
  const int32_t* idx_past;   /* [B][T] or NULL */
  const int32_t* idx_future; /* [B][T] or NULL */
  int32_t B, T, A;
  int32_t dilation, adaptive;
  float out_scale;     /* sqrt(0.5) in the reference */
  int32_t out_relu;    /* 1: xb_out = relu(...) — folds conv_last's leading ReLU into the last block (generator.py:461) */
  /* Frame-rate aux projection (optional; both NULL = the sample-rate `aux` above is used).  When set, `aux` and `A` are
   * ignored, w1p is [128][192] (svsk_usfgan_pack_block with A = 0) and the block adds
   *   sum_k aux_u[t][k] * aux_q[b][n][q_fpad + fbase(t) + k],   fbase = svsk_usfgan_frame_base(128*(t/128), reach, hop)
   * i.e. conv1x1_aux(upsample(c)) with the projection done at frame rate — see svsk_usfgan_aux_frames / _weights. */
  const void* aux_u;   /* [ceil128(T)][16] bf16 from svsk_usfgan_aux_weights */
  const void* aux_q;   /* this block's [128][q_ld] bf16 rows of track 0 inside svsk_usfgan_aux_frames' output */
  int64_t q_batch_stride; /* elements between tracks of aux_q */
  int32_t q_ld, q_fpad, hop, reach;
} svsk_usfgan_block_params;
SVSK_API int svsk_usfgan_block_bf16(const svsk_usfgan_block_params* p, void* stream);
/* w_taps [128][64][3] (k=3 conv, or stacked convP/convC/convF), w_aux [128][A], w_out [64][64] (fp32) -> packed bf16 */
SVSK_API int svsk_usfgan_pack_block(const float* w_taps, const float* w_aux, const float* w_out, void* w1p, void* woutp,
                                    int C, int A, int G, void* stream);

/* Frame-rate aux projection for all blocks of a generator (upsample.py:61-128 + residual_block.py:74,100,139-142):
 *   q[b][r][q_fpad + f] = sum_a w[r][a] * cin[b][f][a]      r < R (= 128 x number of blocks), f < Tf
 * cin [B][Tf][Ap] bf16 = conv_in's output at frame rate (channels padded with zeros to Ap % 8 == 0), w [R][Ap] bf16 = the
 * blocks' conv1x1_aux weights stacked, q [B][R][q_ld] bf16 — the CALLER zero-fills q first (columns outside
 * q_fpad .. q_fpad+Tf-1 are read by the block kernel and must be finite).  R % 16 == 0. */
SVSK_API int svsk_usfgan_aux_frames(const void* cin, const void* w, void* q, int B, int Tf, int Ap, int R, int q_ld, int q_fpad,
                                    void* stream);
/* u[t][k] = imp[(fbase(t) + k) mod 16][t] for t < T, 0 for T <= t < ceil128(T): the upsampler's impulse responses
 * (imp [16][T] fp32 = upsample_net.upsample applied to 16 channels holding unit impulses at the frames f = ch mod 16)
 * re-ordered into the per-tile frame window the block kernel multiplies with. */
SVSK_API int svsk_usfgan_aux_weights(const float* imp, void* u, int T, int hop, int reach, void* stream);
/* The aux upsampler itself in the same form (nnsvs/usfgan/layers/upsample.py:61-128, the stages after conv_in):
 *   out[b][t][ch] = sum_k imp[(fbase(t) + k) mod 16][t] * cin[b][ch][fbase(t) + k]      (bf16 [B][T][Ap], channels >= A zero)
 * cin [B][A][Tf] fp32 = conv_in's output, imp as for svsk_usfgan_aux_weights.  One pass at the write rate of the
 * sample-rate tensor; same hop / reach limits as the block kernel's frame window. */
SVSK_API int svsk_upsample_frames_bf16(const float* imp, const float* cin, void* out, int B, int A, int Ap, int Tf, int T,
                                       int hop, int reach, void* stream);
/* First frame of the 16-frame window of the tile starting at sample t0 (a multiple of 8, may be negative). */
SVSK_API int svsk_usfgan_frame_base(int t0, int reach, int hop);

/* General NTC bf16 Conv1d on tensor cores (weights resident in smem, persistent over 128-sample tiles):
 *   y[b][t][co] = act(bias[co] + sum_j sum_ci w[co][ci][j] x[b][t + (j - tap_origin)*dilation][ci])
 * pad_mode: SVSK_PAD_ZEROS / REFLECT / REPLICATE.  Replaces PeriodicityEstimator's convs (residual_block.py:358-366) and
 * conv_last's first 1x1 (generator.py:463).  Cin % 8 == 0, Cout % 16 == 0, Cout <= 256, packed weights must fit smem. */
typedef struct svsk_conv1d_bf16_params {
  const void* x;      /* [B][T][Cin] bf16 */
  const void* wp;     /* [Cout][ksize * ceil64(Cin)] bf16 from svsk_conv1d_pack_bf16 */
  const float* bias;  /* [Cout] or NULL */
  void* y;            /* [B][T][Cout] bf16 */
  int32_t B, T, Cin, Cout;
  int32_t ksize, dilation, tap_origin, pad_mode, act;
} svsk_conv1d_bf16_params;
SVSK_API int svsk_conv1d_bf16(const svsk_conv1d_bf16_params* p, void* stream);
SVSK_API int svsk_conv1d_pack_bf16(const float* w /* [Cout][Cin][ksize] */, void* wp, int Cout, int Cin, int ksize, void* stream);
/* s = a*h + (1-a)*n on NTC bf16 tensors of cnt elements (generator.py:505-507). */
SVSK_API int svsk_periodic_mix_bf16(const void* a, const void* h, const void* n, void* s, size_t cnt, void* stream);
/* y[r] = bias + sum_c w[c] x[r][c]: the final C -> 1 projection of conv_last (generator.py:465). */
SVSK_API int svsk_dot_rows_bf16(const void* x_bf16, const float* w, float bias, float* y, size_t rows, int C, void* stream);

/* [B][T][Cp] bf16 -> [B][C][T] fp32 (first C channels). */
SVSK_API int svsk_ntc_bf16_to_nct_f32(const void* x_bf16, float* y, int B, int C, int T, int Cp, void* stream);

/* Time-major bf16 GEMM with fused epilogue — replaces the 1x1 projections around the stacks
 * (denoiser.py:110-112,121-123 ; generator.py:461-466,492-493):
 *   Y[n][co] = act( sum_k A[n][k] W[co][k] + bias[co] )      n = B*T rows, K % 16 == 0, Cout % 16 == 0, Cout <= 256
 * A [N][lda] bf16 ; W [Cout][K] bf16 ; outputs optional: y_bf16 [N][ldy_b], y_f32 [N][ldy_f]. */
typedef struct svsk_linear_bf16_params {
  const void* a; const void* w; const float* bias;
  void* y_bf16; float* y_f32;
  int64_t N; int32_t K, Cout; int32_t lda, ldy_b, ldy_f; int32_t act;
} svsk_linear_bf16_params;
SVSK_API int svsk_linear_bf16(const svsk_linear_bf16_params* p, void* stream);

/* ---- FFConvLSTM encoder pieces (nnsvs/model.py:779-926; SURVEY.md §8(f) row 1) ---------------------------------- */

/* Recurrent half of one bidirectional nn.LSTM layer over a padded batch of packed sequences (model.py:861-868,917-919):
 *   a_t = pre_t + W_hh h_{t-1} ; c_t = sigmoid(f) c_{t-1} + sigmoid(i) tanh(g) ; h_t = sigmoid(o) tanh(c_t)
 * with gate rows in torch order i, f, g, o, h_0 = c_0 = 0; direction 1 runs from frame lengths[b]-1 down to 0; frames
 * >= lengths[b] are written as zeros (pack_padded_sequence / pad_packed_sequence).  One thread-block cluster per
 * (track, direction); W_hh lives in registers.  pre = W_ih x + b_ih + b_hh (a GEMM done by the caller), addressed as
 * pre[b*pre_stride_b + t*pre_stride_t + (dir*4H + row)*pre_stride_r]; outputs h_f32[b*hf_stride_b + t*hf_stride_t +
 * (dir*H + u)*hf_stride_c] and / or h_bf16[b*hb_stride_b + t*hb_stride_t + dir*H + u] (either may be NULL). */
typedef struct svsk_lstm_params {
  const float* pre;
  const float* w_hh;        /* [ndir][4H][H] */
  const int32_t* lengths;   /* [B] or NULL (= T) */
  float* h_f32;
  void* h_bf16;
  int64_t pre_stride_b, pre_stride_t, pre_stride_r;
  int64_t hf_stride_b, hf_stride_t, hf_stride_c;
  int64_t hb_stride_b, hb_stride_t;
  int32_t B, T, H, ndir;
} svsk_lstm_params;
SVSK_API int svsk_lstm_f32(const svsk_lstm_params* p, void* stream);
/* 1 when svsk_lstm_f32 has a cluster layout for hidden size H (H <= 256, H % 4 == 0, H / 2^k <= 32 for a k <= 3). */
SVSK_API int svsk_lstm_supported(int H);

/* Frame-major bf16 GEMM over row-shifted taps — the ff Linears (ksize 1), the three ReflectionPad1d(3) + Conv1d(k=7) +
 * BatchNorm1d(eval) + ReLU layers (model.py:846-859), the LSTM input projections and the output Linear of the encoder:
 *   Y[b][t][co] = act( bias[co] + sum_{j<ksize} sum_ci W[co][ci][j] * X[b][t + j][ci] ),  t < T
 * x: [B][Tp_x][ldx] bf16, already padded in time by the caller (Tp_x >= T + ksize - 1; see svsk_reflect_pad_rows_bf16);
 * wp: packed by svsk_tapgemm_pack_bf16; y_bf16 row (b, t) lives at ((b*Tp_y + y_row0 + t)*ldy_b), so a layer can write
 * straight into the padded input buffer of the next one; y_f32 is [B][T][ldy_f].  Cout % 16 == 0; act NONE or RELU. */
typedef struct svsk_tapgemm_bf16_params {
  const void* x; const void* wp; const float* bias;
  void* y_bf16; float* y_f32;
  int32_t B, T, Cin, Cout, ksize;
  int32_t Tp_x, ldx;
  int32_t Tp_y, y_row0, ldy_b, ldy_f;
  int32_t act;
} svsk_tapgemm_bf16_params;
SVSK_API int svsk_tapgemm_bf16(const svsk_tapgemm_bf16_params* p, void* stream);
/* wp[j][co][k] = bf16(w[co][k][j] * scale[co]) for k < Cin, 0 up to ceil64(Cin); scale (folded BatchNorm) may be NULL. */
SVSK_API int svsk_tapgemm_pack_bf16(const float* w /* [Cout][Cin][ksize] */, const float* scale, void* wp, int Cout, int Cin,
                                    int ksize, void* stream);
/* nn.ReflectionPad1d(pad) in place on buf [B][Tp][C] bf16 whose rows pad..pad+T-1 hold the data (model.py:847,851,855). */
SVSK_API int svsk_reflect_pad_rows_bf16(void* buf, int B, int Tp, int C, int T, int pad, void* stream);
/* nn.BatchNorm1d in TRAINING mode on x [B][C][T] fp32 (model.py:839-852 under module.train(); the diffusion recipe's encoders
 * run with dropout = 0, so the batch statistics are all that differs from the eval forward):
 *   svsk_bn_batch_stats_f32: mean[c], var[c] (biased) over all B*T positions of channel c, padded frames included; if
 *     running_mean / running_var are given they move by `momentum` towards (mean, unbiased variance), as torch does;
 *   svsk_bn_apply_f32: y = act((x - mean[c]) / sqrt(var[c] + eps) * gamma[c] + beta[c]), relu != 0 -> ReLU; y may be x. */
SVSK_API int svsk_bn_batch_stats_f32(const float* x, int B, int C, int T, float* mean, float* var, float* running_mean,
                                     float* running_var, float momentum, void* stream);
SVSK_API int svsk_bn_apply_f32(const float* x, float* y, const float* mean, const float* var, const float* gamma,
                               const float* beta, float eps, int relu, int B, int C, int T, void* stream);
/* Input side of the embedding front (model.py:897-910): copies x [rows][in_dim] to y_f32 [rows][ldy_f] and / or y_bf16
 * [rows][ldy_b] (zero-filled pitch) with the one-hot block [onehot_start, +onehot_len) replaced by the exact one-hot of
 * its argmax, so that emb(argmax) + fc_in(rest) becomes one GEMM with the weights [fc_in | emb^T].  onehot_len 0 = copy. */
SVSK_API int svsk_encoder_front(const float* x, float* y_f32, void* y_bf16, long long rows, int in_dim, int onehot_start,
                                int onehot_len, int ldy_f, int ldy_b, void* stream);

/* ---- FFConvLSTM encoder training (backward of model.py:893-922 with dropout = 0), fp32 on the CUDA cores ---------- */

/* svsk_lstm_f32 that also keeps what the backward needs: gates [B][ndir*4H][T] (the activated i, f, g, o of every frame
 * < lengths[b], torch row order within a direction: gates[b][(dir*4 + g)*H + u][t]) and cell [B][ndir*H][T] (c_t).
 * Frames >= lengths[b] hold zeros.  Same checks as svsk_lstm_f32; h is bit-identical to svsk_lstm_f32's. */
SVSK_API int svsk_lstm_train_f32(const svsk_lstm_params* p, float* gates, float* cell, void* stream);

/* Backward of the recurrence (torch.nn.LSTM's backward through pack_padded_sequence, model.py:917-919), in each
 * direction's own scan order reversed (the reverse direction starts at lengths[b] - 1):
 *   dh = dh_ext[t] + W_hh^T da_{t+1} ; dc = dc_{t+1} f_{t+1} + dh o (1 - tanh^2 c_t)
 *   dpre[t] = da_t = [dc g i(1-i), dc c_{t-1} f(1-f), dc i (1-g^2), dh tanh(c_t) o(1-o)]
 * dpre = dL/d(W_ih x + b_ih + b_hh) [B][ndir*4H][T], zero for frames >= lengths[b] (dh_ext there is not read).
 * dh_ext [B][ndir*H][T]; gates / cell from svsk_lstm_train_f32; w_hh [ndir][4H][H]; lengths [B] or NULL (= T).
 * H as svsk_lstm_supported.  One thread-block cluster per (track, direction), W_hh^T in registers. */
typedef struct svsk_lstm_bwd_params {
  const float* dh;
  const float* gates;
  const float* cell;
  const float* w_hh;
  const int32_t* lengths;
  float* dpre;
  int32_t B, T, H, ndir;
} svsk_lstm_bwd_params;
SVSK_API int svsk_lstm_bwd_f32(const svsk_lstm_bwd_params* p, void* stream);

/* Weight (and bias) gradient of a Conv1d / Linear, also of W_hh with a one-frame shift:
 *   dw[n][k][j] = sum_b sum_t dy[b][n][t] * x[b][k][src(t + j - origin)] ;  db[n] = sum_b sum_t dy[b][n][t]
 * dy at dy[b*dy_batch_stride + n*T + t], x at x[b*x_batch_stride + k*T + u]; src: pad_mode SVSK_PAD_ZEROS (0 outside
 * [0, T)) or SVSK_PAD_REFLECT (ReflectionPad1d, needs 0 <= origin < ksize and a reach below T).  Uses: the Linears
 * (ksize 1, origin 0), the ReflectionPad1d(3) + Conv1d(k=7) layers (origin 3, reflect), the LSTM input projections, and
 * W_hh as da^T against h of the previous step (origin 1 forward, -1 reverse: h[lengths[b]] = 0 is read).  db may be NULL.
 * 64 x 64 output tiles reduced over 32-frame chunks in a fixed order; splits > 1 splits the chunks and needs ws
 * [splits][N][K*ksize + (db != NULL)], summed in split order by a second launch.  No atomics: bit-reproducible. */
typedef struct svsk_wgrad_f32_params {
  const float* dy;
  const float* x;
  float* dw;                /* [N][K][ksize] */
  float* db;                /* [N] or NULL */
  float* ws;
  int64_t dy_batch_stride, x_batch_stride;
  int32_t B, N, K, T, ksize, origin, pad_mode, splits;
} svsk_wgrad_f32_params;
SVSK_API int svsk_wgrad_f32(const svsk_wgrad_f32_params* p, void* stream);

/* BatchNorm1d (batch statistics, model.py:839-852 under module.train()) + ReLU backward over all B*T positions of a
 * channel, padded frames included: with xhat = (x - mean) / sqrtf(var + eps) (x the BatchNorm input, mean / var the
 * forward's svsk_bn_batch_stats_f32 outputs) and y the forward's ReLU output,
 *   dz = dy [y > 0] ; dbeta = sum dz ; dgamma = sum dz xhat ; dx = gamma / sqrt(var + eps) (dz - (dbeta + xhat dgamma) / (B T))
 * All [B][C][T] fp32; dx may be dy. */
SVSK_API int svsk_bn_relu_bwd_f32(const float* dy, const float* y, const float* x, const float* mean, const float* var,
                                  const float* gamma, float eps, float* dx, float* dgamma, float* dbeta, int B, int C, int T,
                                  void* stream);

/* nn.ReflectionPad1d(pad) backward in front of a Conv1d(w [Cout][Cin][2 pad + 1]): dx [B][Cin][T] holds the gradient of
 * the padded input's centre rows (svsk_conv1d_f32 of dy with the flipped, transposed weights); this adds the padded rows
 * dXp[p] = sum_j w[:, ci, j]^T dy[p - j] into the frames they reflect: rows 0 .. pad-1 into frames pad .. 1, rows
 * T+pad .. T+2pad-1 into frames T-2 .. T-1-pad.  dy [B][Cout][T]; 1 <= pad <= 4, T > pad. */
SVSK_API int svsk_reflect_fold_f32(float* dx, const float* dy, const float* w, int B, int Cin, int Cout, int T, int pad,
                                   void* stream);

/* ---- acoustic post-processing on the device (SURVEY.md §8(f) row 3) ----------------------------------------------- */

/* nnsvs.dsp.lowpass_filter over whole batches (dsp.py:10-33; gen.py:1500-1513 calls it per feature dimension):
 * scipy.signal.filtfilt(b, a, x) with default padding on every trajectory x[bi, :lengths[bi], d] of x [B][T][D] fp32 ->
 * y (may alias x).  b, a (a[0] == 1, order+1 values each) and zi = lfilter_zi(b, a) (order values) are HOST pointers
 * read at call time; pad = 3 * (order + 1); trajectories of at most min_len (>= pad) frames, and the frames beyond
 * lengths[bi], are copied unchanged (dsp.py:26-28).  scratch: B * (T + 2 pad) * D doubles.  fp64 arithmetic. */
SVSK_API int svsk_filtfilt_f32(const float* x, float* y, double* scratch, const int32_t* lengths, const double* b,
                               const double* a, const double* zi, int order, int pad, int min_len, int B, int T, int D,
                               void* stream);
/* nnsvs.postfilters.variance_scaling per track (postfilters.py:9-46; gen.py:1410-1418): mean / population variance of
 * x[bi, t, d] over the frames t < lengths[bi] with note_mask[bi][t] != 0 (NULL mask = all frames), then
 * y = sqrt(gv[d] / var) * (x - mean) + mean on those frames for d >= offset; everything else is copied.  x, y [B][T][D]. */
SVSK_API int svsk_variance_scaling_f32(const float* x, float* y, const float* gv, const uint8_t* note_mask,
                                       const int32_t* lengths, int offset, int B, int T, int D, void* stream);
/* Feature scalers between the models (nnsvs/util.py:272-340; gen.py:1145 inverse_transform of the acoustic output,
 * gen.py predict_waveform: transform of the vocoder input): per-feature affine maps over x [rows][D] (y may alias x).
 * mode 0: y = x * a[d] + b[d]  (StandardScaler.inverse_transform with a = scale_, b = mean_; MinMaxScaler.transform with
 * a = scale_, b = min_);  mode 1: y = (x - b[d]) / a[d]  (StandardScaler.transform; MinMaxScaler.inverse_transform). */
SVSK_API int svsk_scale_features_f32(const float* x, float* y, const float* a, const float* b, int mode, long long rows, int D,
                                     void* stream);
/* Dimension-wise mixture-density head (nnsvs/mdn.py:45-74 MDNLayer.forward, :165-212 most probable component): raw
 * [rows][ld] holds the outputs of the log_pi, log_sigma and mu Linears side by side (G*D columns each, component-major).
 * log_pi <- log_softmax over the G components per output dimension, log_sigma / mu <- copies, all [rows][G][D];
 * best_sigma / best_mu [rows][D] <- exp(log_sigma) and mu of the component with the largest weight.  Any output may be
 * NULL. */
SVSK_API int svsk_mdn_head_f32(const float* raw, float* log_pi, float* log_sigma, float* mu, float* best_sigma, float* best_mu,
                               long long rows, int G, int D, int ld, void* stream);

/* Fused WaveNet residual block, fp32 — replaces ResSkipBlock._forward (nnsvs/wavenet/modules.py:88-122), one launch:
 *   y = causal_conv(x; ksize, dilation) + conv1x1c(c) + b1;  z = tanh(y[:G/2]) * sigmoid(y[G/2:])
 *   skips = (first ? 0 : skips) + conv1x1_skip(z) + b2[:S];  x_out = conv1x1_out(z) + b2[S:] + x
 * x, x_out [B][R][T], c [B][Cc][T], skips [B][S][T] fp32; x_out must not alias x.  w1t [ksize*R + Cc][G] and
 * w2t [G/2][S + R] are the layer's slices w1t[l] and w2t[l] of svsk_wavenet_train_pack_f32's pack (effective,
 * weight-norm-folded weights); b1 [G] (may be NULL), b2 [S + R] = [skip | out]. */
typedef struct svsk_wavenet_block_params {
  const float* x;
  const float* c;
  const float* w1t;
  const float* b1;
  const float* w2t;
  const float* b2;
  float* x_out;
  float* skips;
  int32_t B, T, R, G, S, Cc, ksize, dilation, first;
} svsk_wavenet_block_params;
SVSK_API int svsk_wavenet_block_f32(const svsk_wavenet_block_params* p, void* stream);


/* WaveNet autoregressive sampling, fp32 — replaces WaveNet.inference (nnsvs/wavenet/wavenet.py:89-149) for B tracks in
 * one launch.  Per track and step t < steps:
 *   x_0 = first_conv(onehot(y[t-1])) (the bias alone at t = 0); for each layer l (dilation 2^(l mod layers/stacks)):
 *   a = conv_l(x_l)[t] (taps at t - (k-1-j) d, zeros before frame 0) + b_l + cproj[b][l G + g][t];
 *   z = tanh(a[:G/2]) * sigmoid(a[G/2:]);  skip += conv1x1_skip_l(z);  x_{l+1} = conv1x1_out_l(z) + x_l;
 *   logits = last3(relu(last1(relu(skip))));  p = softmax(logits);
 *   y[t] = smallest c with u[b][t] < p_0 + .. + p_c (largest c with p_c > 0 if rounding leaves none), written one-hot.
 * cproj [B][layers G][T] holds conv1x1c of every layer on the conditioning c [B][cin][T]: svsk_conv1d_f32 with
 * w = wcond [layers G][cin][1] from svsk_wavenet_ar_pack_f32, no bias.  u [B][steps] uniforms in [0, 1) (the caller's
 * random numbers); y [B][steps][out_dim]; logits [B][steps][out_dim] or NULL; hist: workspace of B * hist_floats
 * (svsk_wavenet_ar_sizes), no initialisation needed.  steps <= T.  Shapes: svsk_wavenet_ar_supported. */
typedef struct svsk_wavenet_ar_params {
  const float* wpack;
  const float* cproj;
  const float* u;
  float* y;
  float* logits;
  float* hist;
  int32_t B, T, steps, out_dim, R, G, S, layers, stacks, ksize;
} svsk_wavenet_ar_params;
SVSK_API int svsk_wavenet_ar_f32(const svsk_wavenet_ar_params* p, void* stream);
/* 1 when svsk_wavenet_ar_f32 covers the WaveNet (out_dim, residual R, gate G, skip S channels, layers, stacks, kernel
 * size): k R <= 256, G / 2 <= 64, S <= 64, S + R <= 128, out_dim <= 256, layers <= 64 with layers / stacks <= 16. */
SVSK_API int svsk_wavenet_ar_supported(int out_dim, int R, int G, int S, int layers, int stacks, int ksize);
/* Floats of the packed weights and of the per-track ring buffer (hist) of a supported WaveNet; SVSK_E_ARG otherwise. */
SVSK_API int svsk_wavenet_ar_sizes(int out_dim, int R, int G, int S, int layers, int stacks, int ksize, long long* pack_floats,
                                   long long* hist_floats);
/* Parameters of a WaveNet as stored in its modules, all device pointers to fp32: each weight is v with its weight-norm
 * gain g ([rows], NULL = v is the weight itself), per-layer tensors stacked over the layers.  Shapes: first [R][out_dim],
 * conv [layers][G][R][ksize], cond [layers][G][cin] (no bias), skip [layers][S][G/2], out [layers][R][G/2],
 * last1 [S][S], last3 [out_dim][S]; biases [rows] per weight (conv_b may be NULL = zeros). */
typedef struct svsk_wavenet_ar_weights {
  const float *first_v, *first_g, *first_b;
  const float *conv_v, *conv_g, *conv_b;
  const float *cond_v, *cond_g;
  const float *skip_v, *skip_g, *skip_b;
  const float *out_v, *out_g, *out_b;
  const float *last1_v, *last1_g, *last1_b;
  const float *last3_v, *last3_g, *last3_b;
  int32_t out_dim, R, G, S, cin, layers, stacks, ksize;
} svsk_wavenet_ar_weights;
/* Folds weight norm with the fold of svsk_wavenet_train_pack_f32 (the same bits) and lays the weights out for
 * svsk_wavenet_ar_f32, one launch: wpack [pack_floats] and wcond [layers G][cin]. */
SVSK_API int svsk_wavenet_ar_pack_f32(const svsk_wavenet_ar_weights* w, float* wpack, float* wcond, void* stream);

/* ------------------------------------------------------------------------------------------------
 * WaveNet training (WaveNet.forward under autograd, nnsvs/wavenet/wavenet.py:60-87), fp32 on the CUDA cores.
 * L layers, residual R, gate G (G2 = G / 2), skip S, conditioning cin, out_dim classes, kernel k; Rp = R and G2p = G2
 * rounded up to multiples of 4.  Shapes: exactly those svsk_wavenet_block_f32 accepts.
 * ------------------------------------------------------------------------------------------------ */

/* svsk_wavenet_block_f32 that also writes the gate pre-activations y [B][G][T] (y = conv + conv1x1c + b1, before the
 * gate), which the backward needs.  x_out and skips are bit-identical to svsk_wavenet_block_f32's. */
typedef struct svsk_wavenet_block_train_params {
  svsk_wavenet_block_params blk;
  float* y;
} svsk_wavenet_block_train_params;
SVSK_API int svsk_wavenet_block_train_f32(const svsk_wavenet_block_train_params* p, void* stream);

/* Floats of the training weight pack (svsk_wavenet_train_pack_f32) and of the gradient arena (svsk_wavenet_wgrad_f32);
 * SVSK_E_ARG for shapes svsk_wavenet_block_f32 rejects. */
SVSK_API int svsk_wavenet_train_sizes(int out_dim, int R, int G, int S, int cin, int layers, int ksize, long long* pack_floats,
                                      long long* grad_floats);
/* Folds weight norm (w = g v / ||v|| per output row, the same arithmetic as torch._weight_norm(v, g, 0) on CUDA, so the
 * forward matches the module's eval path bit for bit; g == NULL: w = v) of every weight of w (stacked as documented
 * at svsk_wavenet_ar_weights; biases are not read) and writes, one launch, pack [pack_floats] =
 *   w1t [L][k R + cin][G]  w1t[l][j R + ci][co] = conv_l[co][ci][j], w1t[l][k R + cc][co] = conv1x1c_l[co][cc]
 *   w2t [L][G2][S + R]     w2t[l][c2][o] = conv1x1_skip_l[o][c2] for o < S, conv1x1_out_l[o - S][c2] after
 *                          (w1t[l] and w2t[l] are svsk_wavenet_block_f32's weights)
 *   wT [L][k G][Rp]        wT[l][j G + co][ci] = conv_l[co][ci][j]             (transposed conv of the backward)
 *   wB [L][R + S][G2p]     rows: conv1x1_out_l [R][G2] then conv1x1_skip_l [S][G2]
 *   wcT [cin][L G]         wcT[cc][l G + co] = conv1x1c_l[co][cc]
 *   first [R][out_dim], firstT [out_dim][R], last1 [S][S], last1T [S][S], last3 [out_dim][S], last3T [S][out_dim]
 * Padding columns of wT and wB are zero. */
SVSK_API int svsk_wavenet_train_pack_f32(const svsk_wavenet_ar_weights* w, float* pack, void* stream);

/* One step of the backward through the residual blocks, from the last down: launch l (l = L .. 0) computes
 *   g_l = g_{l+1} + sum_j conv_l[:, :, j]^T dy_l(t + (k-1-j) d_l)       (dL/dx_l; dy_in == NULL: l == L, g_l = 0)
 * and, when y_prev != NULL (l >= 1), for block l-1
 *   dz = conv1x1_out^T g_l + conv1x1_skip^T dS;  dy_{l-1} = [dz sig(b)(1 - tanh^2 a) | dz tanh(a) sig(b)(1 - sig(b))]
 * with a, b the halves of y_prev.  Tensors fp32: dy_in, dy_out [B] x [G][T] with batch stride dy_bstride (the slices of a
 * [B][L][G][T] buffer); g_next (NULL = 0), g_out [B][R][T]; dS [B][S][T] = dL/dskips (after the ReLU mask); y_prev
 * [B][G][T]; wT = pack's wT[l], wB = pack's wB[l-1].  dilation is d_l. */
typedef struct svsk_wavenet_dgrad_params {
  const float* dy_in;
  const float* wT;
  const float* g_next;
  float* g_out;
  const float* dS;
  const float* y_prev;
  const float* wB;
  float* dy_out;
  long long dy_bstride;
  int32_t B, T, R, G, S, ksize, dilation;
} svsk_wavenet_dgrad_params;
SVSK_API int svsk_wavenet_dgrad_f32(const svsk_wavenet_dgrad_params* p, void* stream);

/* Gradients of every effective weight and bias, without atomics: each CTA reduces a 64 x 64 output tile over its share
 * of the (b, t) frames in a fixed order; splits > 1 writes per-split partials to ws [splits][grad_floats] and a second
 * launch sums them in split order, so results are bit-reproducible.  dW [grad_floats] receives, in this order:
 *   conv [L][G][R][k], conv_b [L][G], cond [L][G][cin], skip [L][S][G2], skip_b [L][S], out [L][R][G2], out_b [L][R],
 *   first [R][out_dim], first_b [R], last1 [S][S], last1_b [S], last3 [out_dim][S], last3_b [out_dim].
 * Inputs (fp32): x_in [B][out_dim][T] (first_conv's input), c [B][cin][T], xs [L][B][R][T] (block inputs), ys
 * [L][B][G][T], gs [L + 1][B][R][T] (dL/dx_l, g_L = 0), dy [B][L][G][T], dS, skips (the forward's skip sum), h1
 * (last1's output before the ReLU), dh1 = dL/dh1 [B][S][T], glog = dL/dlogits [B][out_dim][T]; dilations: device int32
 * [L]. */
typedef struct svsk_wavenet_wgrad_params {
  const float *x_in, *c, *xs, *ys, *gs, *dy, *dS, *skips, *h1, *dh1, *glog;
  const int32_t* dilations;
  float* dW;
  float* ws;
  int32_t B, T, out_dim, R, G, S, cin, layers, ksize, splits;
} svsk_wavenet_wgrad_params;
SVSK_API int svsk_wavenet_wgrad_f32(const svsk_wavenet_wgrad_params* p, void* stream);

/* Weight-norm backward of the weights of w that have a gain (g != NULL), one launch: with n = ||v|| per row and dw the
 * effective weight's gradient in dW (svsk_wavenet_wgrad_f32's layout), dg = <dw, v> / n and, in place, dw <- (g / n)
 * (dw - dg v / n).  dg [first R][conv L G][cond L G][skip L S][out L R][last1 S][last3 out_dim]. */
SVSK_API int svsk_wavenet_wnorm_grad_f32(const svsk_wavenet_ar_weights* w, float* dW, float* dg, void* stream);

/* y[i] = m[i] > 0 ? x[i] : 0 (the ReLU derivative); y may alias x. */
SVSK_API int svsk_relu_mask_f32(const float* x, const float* m, float* y, long long n, void* stream);

/* Source signal and dilation factors of the uSFGAN front end from frame-level F0 (nnsvs/usfgan/utils/features.py:
 * SignalGenerator.sinusoid :145-164, dilated_factor :56-75; called per utterance by USFGANWrapper.inference,
 * nnsvs/usfgan/__init__.py:50-63).  f0 [B][F] in Hz as float64 (0 = unvoiced; the sine uses its fp32 rounding like
 * torch.FloatTensor(f0)); T = F * hop samples per track.
 *   sine_out[b * sine_batch_stride + t] = vuv * sin(2 pi cumsum((f0 / fs) mod 1)) * sine_amp
 *                                         + noise[b][t] * (vuv * noise_amp + (1 - vuv) * noise_amp / 3)    (NULL: skipped)
 *   d_out[b][t] = float(fs / f0 / dense_factor), unvoiced -> 1                                              (NULL: skipped)
 * The prefix sums are fp64 rounded to fp32 per sample — what torch.cumsum does on a CPU host.  noise [B][T] holds the
 * caller's Gaussian draws (ignored when noise_amp == 0); scratch: B * F doubles. */
SVSK_API int svsk_usfgan_source(const double* f0, const float* noise, float* sine_out, long long sine_batch_stride, float* d_out,
                                double* scratch, int B, int F, int hop, int sample_rate, int dense_factor, float sine_amp,
                                float noise_amp, void* stream);

/* ---- DiffNet training kernels (SURVEY.md §8(f) row 4: dgrad / wgrad / fused gate backward) -------------------------
 * Replace, inside the training step (nnsvs/bin/train_acoustic_multitrack.py:358-380), what autograd derives from
 * ResidualBlock.forward / DiffNet.forward (nnsvs/diffsinger/denoiser.py:54-66, 101-124).  See diffnet_train_sm100.cu. */
enum { SVSK_SEG_PLAIN = 0, SVSK_SEG_GATE_FWD = 1, SVSK_SEG_RES_SKIP = 2, SVSK_SEG_GATE_BWD = 3, SVSK_SEG_ADD_SCALE = 4 };

/* Frame-major segmented GEMM on tcgen05:
 *   D[b][t][n] = sum_s sum_k x[s][b][t + shift[s]][k] * wp[n][koff_s + k],  koff_s = kx[0] + .. + kx[s-1]
 * x[s]: [B][T][ldx[s]] bf16 (first kx[s] columns used, kx % 64 == 0); rows outside [0, T) of a track read as 0.
 * wp: [Nrows][sum kx] bf16.  The epilogue depends on `mode`:
 *  GATE_FWD  (Nrows = 2C packed rows, svsk_diffnet_train_pack): y = D + bias -> out0 [.][ld_out0] (ypre, packed columns),
 *            out1 [.][ld_out1] = sigmoid(y_gate) * tanh(y_filter) (z, channel order)
 *  RES_SKIP  (Nrows = 2C reference rows, C = Nrows / 2): o = D + bias; out0 = x' = (in0 + o[:C]) / sqrt 2 and
 *            out1 = x' + dp_next[b][:] (either may be NULL); outf (skip32, fp32) = o[C:] if init else += o[C:]
 *  GATE_BWD  (Nrows = C): dz = D; in0 = ypre (packed columns), out0 = dy (packed columns)
 *  ADD_SCALE / PLAIN: v = act(D + bias + in0) * alpha, zeroed where mask <= 0; -> out0 (bf16), out1 = v + dp_next[b][n]
 *            (bf16, dp_next [B][Nrows]) and / or outf (fp32, += if accumulate).  bias, in0, mask, dp_next optional. */
typedef struct svsk_seggemm_params {
  const void* x[4];
  int32_t ldx[4], kx[4], shift[4];
  int32_t nseg;
  const void* wp;
  int32_t Nrows, B, T, mode, C, init, act, accumulate;
  const float* bias;
  const void* in0;
  int32_t ld_in0;
  const void* mask;
  int32_t ld_mask;
  const float* dp_next; /* [B][C] fp32 */
  void* out0;
  int32_t ld_out0;
  void* out1;
  int32_t ld_out1;
  float* outf;
  int32_t ld_outf;
  float alpha;
} svsk_seggemm_params;
SVSK_API int svsk_seggemm_bf16(const svsk_seggemm_params* p, void* stream);

/* Weight gradients: dW[n][koff_s + k] (+)= sum_b sum_t p[b][n][t] * q[s][b][k][t + shift[s]], n < Prows, k < qrows[s];
 * koff_s = qrows[0] + .. + qrows[s-1].  p, q[s]: [B][rows][Tp] bf16 (time contiguous; svsk_ntc_to_nct_bf16), frames
 * outside [0, T) read as 0.  shift[s] must be a multiple of 8 frames (16-byte aligned TMA start); other shifts are
 * written into the operand by svsk_ntc_to_nct_bf16.  Column sums over time (bias gradients) are obtained by appending
 * rows of ones to a q operand.  dW [Prows][ldw] fp32.  One CTA per 128 x 128 tile of dW, whole contraction, no atomics. */
typedef struct svsk_wgrad_params {
  const void* p;
  const void* q[5];
  int32_t qrows[5], shift[5];
  int32_t nseg, Prows, B, T, Tp, ldw, accumulate;
  int32_t splits;           /* >= 1: the tracks are cut into `splits` groups, group z writes dW + z * split_stride */
  int64_t split_stride;     /* floats; the caller sums the partial results (deterministic) */
  float* dW;
} svsk_wgrad_params;
SVSK_API int svsk_wgrad_bf16(const svsk_wgrad_params* p, void* stream);

/* y[b][row0 + j * N + n][t] = x[b][t + shifts[j]][n] (0 outside [0, T)) for j < nshift (1..3), n < N, t < Tp:
 * x [B][T][ldx] bf16, y [B][out_rows][Tp] bf16; N, ldx, Tp multiples of 8.  shifts is a HOST array read at call time. */
SVSK_API int svsk_ntc_to_nct_bf16(const void* x, void* y, int B, int T, int N, int ldx, int Tp, int out_rows, int row0,
                                  int nshift, const int* shifts, void* stream);
/* Packs the stacked fp32 parameters of all L residual layers (wd [L][2C][C][3], wc [L][2C][H], wo [L][2C][C]) into the
 * bf16 operands of the kernels above: w1p [L][2C][3C+H] (packed rows), woutp [L][2C][C], woutT [L][C][2C],
 * w1T [L][C][3*2C] (K = packed dy columns per tap), wcT [L][H][2C]. */
SVSK_API int svsk_diffnet_train_pack(const float* wd, const float* wc, const float* wo, void* w1p, void* woutp, void* woutT,
                                     void* w1T, void* wcT, int L, int C, int H, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SVSK_H_ */
