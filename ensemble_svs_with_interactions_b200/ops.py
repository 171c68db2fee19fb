"""Host-side wrappers: one Python function per libsvsk entry point (include/svsk.h).

Every function only enqueues kernels on the current CUDA stream; outputs are allocated with the caching
allocator (or taken from ``out=``) so whole loops are CUDA-graph capturable.
"""
from __future__ import annotations

import ctypes as C
import functools
import math
import os
from typing import Optional, Sequence

import torch

from . import _lib as L

PAD_ZEROS, PAD_REFLECT, PAD_REPLICATE, PAD_VALID, PAD_INDEXED = 0, 1, 2, 3, 4
ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_MISH = 0, 1, 2, 3
GATE_SIGMOID_TANH, GATE_TANH_SIGMOID = 0, 1

f32 = torch.float32
bf16 = torch.bfloat16


def conv1d_f32(x, w, bias=None, *, dilation=1, tap_origin=None, pad_mode=PAD_ZEROS, in_bias=None, residual=None,
               idx=None, out=None, accumulate=False, act=ACT_NONE, in_relu=False, out_scale=1.0):
    """svsk_conv1d_f32: x [B,Cin,T_in], w [Cout,Cin,k] -> y [B,Cout,T]."""
    B, Cin, T_in = x.shape
    Cout, Cin_w, k = w.shape
    if Cin_w != Cin:
        raise RuntimeError(f"conv1d_f32: weight expects {Cin_w} input channels, got {Cin}")
    if tap_origin is None:
        tap_origin = (k - 1) // 2
    T = T_in - (k - 1) * dilation if pad_mode == PAD_VALID else T_in
    if out is None:
        if accumulate:
            raise RuntimeError("conv1d_f32: accumulate needs out=")
        out = torch.empty((B, Cout, T), device=x.device, dtype=f32)
    p = L.Conv1dF32Params()
    p.x, p.w, p.y = L.ptr(x, f32, "x"), L.ptr(w, f32, "w"), L.ptr(out, f32, "out")
    p.bias, p.in_bias, p.residual = L.ptr(bias, f32, "bias"), L.ptr(in_bias, f32, "in_bias"), L.ptr(residual, f32, "residual")
    if idx is not None:
        p.idx_past, p.idx_future = L.ptr(idx[0], torch.int32, "idx_past"), L.ptr(idx[1], torch.int32, "idx_future")
    p.B, p.Cin, p.Cout, p.T = B, Cin, Cout, T
    p.ksize, p.dilation, p.tap_origin, p.pad_mode = k, dilation, tap_origin, pad_mode
    p.accumulate, p.act, p.in_relu, p.out_scale = int(accumulate), act, int(in_relu), float(out_scale)
    L.check(L.lib().svsk_conv1d_f32(C.byref(p), L.stream_ptr()), "conv1d_f32")
    return out


def linear_f32(x, w, bias=None, act=ACT_NONE, out=None):
    """nn.Linear on [Bt,Cin] (svsk_linear_f32); w [Cout,Cin] or [Cout,Cin,1]; out: optional contiguous [Bt,Cout]."""
    Bt, Cin = x.shape
    Cout = w.shape[0]
    y = torch.empty((Bt, Cout), device=x.device, dtype=f32) if out is None else out
    if out is not None and (tuple(out.shape) != (Bt, Cout) or not out.is_contiguous()):
        raise ValueError(f"linear_f32: out must be a contiguous [{Bt}, {Cout}] tensor")
    L.check(L.lib().svsk_linear_f32(L.ptr(x, f32, "x"), L.ptr(w, f32, "w"), L.ptr(bias, f32, "bias"), L.ptr(y), Bt, Cin,
                                    Cout, act, L.stream_ptr()), "linear_f32")
    return y


def gated_act_f32(y, order):
    B, H2, T = y.shape
    z = torch.empty((B, H2 // 2, T), device=y.device, dtype=f32)
    L.check(L.lib().svsk_gated_act_f32(L.ptr(y, f32), L.ptr(z), B, H2 // 2, T, order, L.stream_ptr()), "gated_act_f32")
    return z


def diffnet_residual_skip_f32(o, x, skip, init_skip):
    B, C2, T = o.shape
    L.check(L.lib().svsk_diffnet_residual_skip_f32(L.ptr(o, f32), L.ptr(x, f32), L.ptr(skip, f32), B, C2 // 2, T,
                                                   int(init_skip), L.stream_ptr()), "diffnet_residual_skip_f32")


def scale_act_f32(x, alpha=1.0, act=ACT_NONE, out=None):
    out = torch.empty_like(x) if out is None else out
    L.check(L.lib().svsk_scale_act_f32(L.ptr(x, f32), L.ptr(out, f32), x.numel(), float(alpha), act, L.stream_ptr()),
            "scale_act_f32")
    return out


def sinusoidal_embedding_f32(t, dim):
    t = t.to(torch.int64).contiguous()
    out = torch.empty((t.shape[0], dim), device=t.device, dtype=f32)
    L.check(L.lib().svsk_sinusoidal_embedding_f32(L.ptr(t, torch.int64), L.ptr(out), t.shape[0], dim, L.stream_ptr()),
            "sinusoidal_embedding_f32")
    return out


def ddpm_update_f32(x, eps, z, t, tables, clip_denoised=True, out=None):
    """tables: dict of the reference's registered buffers (fp32 CUDA tensors)."""
    B = x.shape[0]
    out = torch.empty_like(x) if out is None else out
    L.check(L.lib().svsk_ddpm_update_f32(
        L.ptr(x, f32, "x"), L.ptr(eps, f32, "eps"), L.ptr(z, f32, "z"), L.ptr(out, f32, "out"), L.ptr(t, torch.int64, "t"),
        L.ptr(tables["sqrt_recip_alphas_cumprod"], f32), L.ptr(tables["sqrt_recipm1_alphas_cumprod"], f32),
        L.ptr(tables["posterior_mean_coef1"], f32), L.ptr(tables["posterior_mean_coef2"], f32),
        L.ptr(tables["posterior_log_variance_clipped"], f32), B, x.numel() // B, int(clip_denoised), L.stream_ptr()),
        "ddpm_update_f32")
    return out


def q_sample_f32(x0, noise, t, tables):
    B = x0.shape[0]
    out = torch.empty_like(x0)
    L.check(L.lib().svsk_q_sample_f32(L.ptr(x0, f32), L.ptr(noise, f32), L.ptr(out), L.ptr(t, torch.int64),
                                      L.ptr(tables["sqrt_alphas_cumprod"], f32),
                                      L.ptr(tables["sqrt_one_minus_alphas_cumprod"], f32), B, x0.numel() // B,
                                      L.stream_ptr()), "q_sample_f32")
    return out


def plms_transfer_f32(x, noise_t, t, interval, alphas_cumprod):
    B = x.shape[0]
    out = torch.empty_like(x)
    L.check(L.lib().svsk_plms_transfer_f32(L.ptr(x, f32), L.ptr(noise_t, f32), L.ptr(out), L.ptr(t, torch.int64),
                                           int(interval), L.ptr(alphas_cumprod, f32), B, x.numel() // B,
                                           L.stream_ptr()), "plms_transfer_f32")
    return out


def lincomb_f32(tensors: Sequence[torch.Tensor], coefs: Sequence[float]):
    n = len(tensors)
    ptrs = (C.c_void_p * n)(*[L.ptr(t, f32).value for t in tensors])
    cs = (C.c_float * n)(*[float(c) for c in coefs])
    out = torch.empty_like(tensors[0])
    L.check(L.lib().svsk_lincomb_f32(ptrs, cs, n, L.ptr(out), out.numel(), L.stream_ptr()), "lincomb_f32")
    return out


def pd_index(d, dilation):
    """d (B,1,T) fp32 -> (idx_past, idx_future) int32 [B,T]; -1 marks a zero tap."""
    B, _, T = d.shape
    ip = torch.empty((B, T), device=d.device, dtype=torch.int32)
    iff = torch.empty((B, T), device=d.device, dtype=torch.int32)
    L.check(L.lib().svsk_pd_index(L.ptr(d, f32, "d"), L.ptr(ip), L.ptr(iff), B, T, int(dilation), L.stream_ptr()),
            "pd_index")
    return ip, iff


def upsample_smooth_f32(x, taps, scale):
    """x [B,C,Tin] -> [B,C,Tin*scale]: nearest stretch then (2*scale+1)-tap smoothing."""
    B, Cc, Tin = x.shape
    out = torch.empty((B, Cc, Tin * scale), device=x.device, dtype=f32)
    L.check(L.lib().svsk_upsample_smooth_f32(L.ptr(x, f32), L.ptr(taps, f32), L.ptr(out), B * Cc, Tin, int(scale),
                                             L.stream_ptr()), "upsample_smooth_f32")
    return out


def periodic_mix_f32(a, h, n, want_parts=False):
    s = torch.empty_like(h)
    h2 = torch.empty_like(h) if want_parts else None
    n2 = torch.empty_like(h) if want_parts else None
    L.check(L.lib().svsk_periodic_mix_f32(L.ptr(a, f32), L.ptr(h, f32), L.ptr(n, f32), L.ptr(s), L.ptr(h2), L.ptr(n2),
                                          h.numel(), L.stream_ptr()), "periodic_mix_f32")
    return s, h2, n2


def nct_to_ntc(x, Cp=None, want_bf16=True, want_f32=False, out_bf16=None, out_f32=None):
    B, Cc, T = x.shape
    Cp = Cc if Cp is None else Cp
    if want_bf16 and out_bf16 is None:
        out_bf16 = torch.empty((B, T, Cp), device=x.device, dtype=bf16)
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty((B, T, Cp), device=x.device, dtype=f32)
    L.check(L.lib().svsk_nct_to_ntc(L.ptr(x, f32, "x"), L.ptr(out_bf16), L.ptr(out_f32), B, Cc, T, Cp, L.stream_ptr()),
            "nct_to_ntc")
    return out_bf16, out_f32


def ntc_to_nct_f32(x, Cc, alpha=1.0):
    B, T, Cp = x.shape
    y = torch.empty((B, Cc, T), device=x.device, dtype=f32)
    L.check(L.lib().svsk_ntc_to_nct_f32(L.ptr(x, f32, "x"), L.ptr(y), B, Cc, T, Cp, float(alpha), L.stream_ptr()),
            "ntc_to_nct_f32")
    return y


def cast_scale_bf16(x, alpha=1.0, relu=False, out=None):
    out = torch.empty(x.shape, device=x.device, dtype=bf16) if out is None else out
    L.check(L.lib().svsk_cast_scale_bf16(L.ptr(x, f32, "x"), L.ptr(out, bf16), x.numel(), float(alpha), int(relu),
                                         L.stream_ptr()), "cast_scale_bf16")
    return out


def diffnet_pack_block(dilated_w, cond_w, out_w):
    C2, Cc, _ = dilated_w.shape
    H = cond_w.shape[1]
    w1p = torch.empty((C2, 3 * Cc + H), device=dilated_w.device, dtype=bf16)
    woutp = torch.empty((C2, Cc), device=dilated_w.device, dtype=bf16)
    L.check(L.lib().svsk_diffnet_pack_block(L.ptr(dilated_w.contiguous(), f32), L.ptr(cond_w.contiguous(), f32),
                                            L.ptr(out_w.contiguous(), f32), L.ptr(w1p), L.ptr(woutp), Cc, H,
                                            L.stream_ptr()), "diffnet_pack_block")
    return w1p, woutp


def diffnet_packed_rows(Cc):
    """perm[r] = packed row of reference row r (host-side, for bias / step-weight packing)."""
    l = L.lib()
    return torch.tensor([l.svsk_diffnet_packed_row(r, Cc) for r in range(2 * Cc)], dtype=torch.long)


def diffnet_block_bf16(xb_in, xb_out, x32, skip32, cond, w1p, woutp, stepbias, bout, *, dilation, stepbias_batch_stride,
                       init_skip, write_x=True):
    """One residual block per launch (svsk_diffnet_block3_bf16: CTA pair, resident activation window; dilation <= 8)."""
    B, T, Cc = xb_in.shape
    p = L.DiffnetBlockParams()
    p.xb_in, p.xb_out = L.ptr(xb_in, bf16, "xb_in"), L.ptr(xb_out, bf16, "xb_out")
    p.x32, p.skip32 = L.ptr(x32, f32, "x32"), L.ptr(skip32, f32, "skip32")
    p.cond, p.w1p, p.woutp = L.ptr(cond, bf16, "cond"), L.ptr(w1p, bf16, "w1p"), L.ptr(woutp, bf16, "woutp")
    p.stepbias, p.bout = L.ptr(stepbias, f32, "stepbias"), L.ptr(bout, f32, "bout")
    p.B, p.T, p.C, p.H = B, T, Cc, cond.shape[2]
    p.dilation, p.stepbias_batch_stride = int(dilation), int(stepbias_batch_stride)
    p.init_skip, p.write_x, p.reserved0 = int(init_skip), int(write_x), 0
    L.check(L.lib().svsk_diffnet_block3_bf16(C.byref(p), L.stream_ptr()), "diffnet_block_bf16")


def wavenet_block_f32(x, c, w1t, b1, w2t, b2, skips, *, ksize, dilation, first, out=None):
    """One fused ResSkipBlock (svsk_wavenet_block_f32): x [B,R,T], c [B,Cc,T] -> new x; skips [B,S,T] set or accumulated."""
    B, R, T = x.shape
    out = torch.empty_like(x) if out is None else out
    p = L.WavenetBlockParams()
    p.x, p.c, p.w1t, p.b1 = L.ptr(x, f32, "x"), L.ptr(c, f32, "c"), L.ptr(w1t, f32, "w1t"), L.ptr(b1, f32, "b1")
    p.w2t, p.b2, p.x_out, p.skips = L.ptr(w2t, f32, "w2t"), L.ptr(b2, f32, "b2"), L.ptr(out, f32, "x_out"), L.ptr(skips, f32, "skips")
    p.B, p.T, p.R, p.G, p.S, p.Cc = B, T, R, w1t.shape[1], skips.shape[1], c.shape[1]
    p.ksize, p.dilation, p.first = int(ksize), int(dilation), int(first)
    L.check(L.lib().svsk_wavenet_block_f32(C.byref(p), L.stream_ptr()), "wavenet_block_f32")
    return out


def wavenet_ar_supported(out_dim, R, G, S, layers, stacks, ksize):
    return bool(L.lib().svsk_wavenet_ar_supported(out_dim, R, G, S, layers, stacks, ksize))


def wavenet_ar_sizes(out_dim, R, G, S, layers, stacks, ksize):
    """(floats of the packed weights, floats of one track's tap ring buffer) of svsk_wavenet_ar_f32."""
    pack, hist = C.c_longlong(), C.c_longlong()
    rc = L.lib().svsk_wavenet_ar_sizes(out_dim, R, G, S, layers, stacks, ksize, C.byref(pack), C.byref(hist))
    if rc != 0:
        raise RuntimeError(f"libsvsk wavenet_ar_sizes failed (code {rc}): {L.lib().svsk_last_error().decode()}")
    return pack.value, hist.value


_AR_WEIGHTS = ("first_v", "first_g", "first_b", "conv_v", "conv_g", "conv_b", "cond_v", "cond_g", "skip_v", "skip_g", "skip_b",
               "out_v", "out_g", "out_b", "last1_v", "last1_g", "last1_b", "last3_v", "last3_g", "last3_b")


def wavenet_ar_pack_f32(w, *, out_dim, R, G, S, cin, layers, stacks, ksize):
    """svsk_wavenet_ar_pack_f32.  w: dict of the fields of svsk_wavenet_ar_weights (fp32 CUDA tensors, per-layer ones
    stacked over the layers; the *_g gains and conv_b may be None) -> (wpack [pack_floats], wcond [layers*G, cin, 1])."""
    npack, _ = wavenet_ar_sizes(out_dim, R, G, S, layers, stacks, ksize)
    dev = w["first_v"].device
    wpack = torch.empty(npack, device=dev, dtype=f32)
    wcond = torch.empty((layers * G, cin, 1), device=dev, dtype=f32)
    p = L.WavenetArWeights()
    for n in _AR_WEIGHTS:
        setattr(p, n, L.ptr(w.get(n), f32, n).value)
    p.out_dim, p.R, p.G, p.S, p.cin, p.layers, p.stacks, p.ksize = out_dim, R, G, S, cin, layers, stacks, ksize
    L.check(L.lib().svsk_wavenet_ar_pack_f32(C.byref(p), L.ptr(wpack), L.ptr(wcond), L.stream_ptr()), "wavenet_ar_pack_f32")
    return wpack, wcond


def wavenet_ar_f32(wpack, cproj, u, *, out_dim, R, G, S, layers, stacks, ksize, logits=None):
    """svsk_wavenet_ar_f32: steps = u.shape[1] autoregressive WaveNet steps for B tracks in one launch.
    wpack from wavenet_ar_pack_f32; cproj [B, layers*G, T] = conv1d_f32(c, wcond) (no bias); u [B, steps] uniforms in
    [0, 1).  Returns the one-hot samples [B, steps, out_dim]; logits: optional [B, steps, out_dim] output."""
    npack, nhist = wavenet_ar_sizes(out_dim, R, G, S, layers, stacks, ksize)
    if u.dim() != 2 or cproj.dim() != 3:
        raise ValueError(f"wavenet_ar_f32: u must be [B, steps] and cproj [B, layers*G, T], got {tuple(u.shape)} and "
                         f"{tuple(cproj.shape)}")
    B, steps = u.shape
    T = cproj.shape[2]
    if tuple(cproj.shape[:2]) != (B, layers * G):
        raise ValueError(f"wavenet_ar_f32: cproj must be [B={B}, layers*G={layers * G}, T], got {tuple(cproj.shape)}")
    if steps < 1 or steps > T:
        raise ValueError(f"wavenet_ar_f32: steps={steps} must be in [1, T={T}] (one conditioning frame per step)")
    if wpack.dim() != 1 or wpack.numel() != npack:
        raise ValueError(f"wavenet_ar_f32: wpack must hold {npack} floats, got {tuple(wpack.shape)}")
    if logits is not None and tuple(logits.shape) != (B, steps, out_dim):
        raise ValueError(f"wavenet_ar_f32: logits must be [{B}, {steps}, {out_dim}], got {tuple(logits.shape)}")
    p = L.WavenetArParams()
    p.wpack, p.cproj, p.u = L.ptr(wpack, f32, "wpack"), L.ptr(cproj, f32, "cproj"), L.ptr(u, f32, "u")
    p.logits = L.ptr(logits, f32, "logits")
    y = torch.empty((B, steps, out_dim), device=u.device, dtype=f32)
    hist = torch.empty(B * nhist, device=u.device, dtype=f32)
    p.y, p.hist = L.ptr(y), L.ptr(hist)
    p.B, p.T, p.steps, p.out_dim, p.R, p.G, p.S = B, T, steps, out_dim, R, G, S
    p.layers, p.stacks, p.ksize = layers, stacks, ksize
    L.check(L.lib().svsk_wavenet_ar_f32(C.byref(p), L.stream_ptr()), "wavenet_ar_f32")
    return y


def _shape(name, t, shape):
    if t is None or tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name} must be {list(shape)}, got {None if t is None else list(t.shape)}")


def wavenet_block_train_f32(x, c, w1t, b1, w2t, b2, skips, y, *, ksize, dilation, first, out=None):
    """svsk_wavenet_block_train_f32: wavenet_block_f32 that also writes the gate pre-activations y [B, G, T]."""
    B, R, T = x.shape
    G = w1t.shape[1]
    _shape("wavenet_block_train_f32: y", y, (B, G, T))
    out = torch.empty_like(x) if out is None else out
    p = L.WavenetBlockTrainParams()
    q = p.blk
    q.x, q.c, q.w1t, q.b1 = L.ptr(x, f32, "x"), L.ptr(c, f32, "c"), L.ptr(w1t, f32, "w1t"), L.ptr(b1, f32, "b1")
    q.w2t, q.b2, q.x_out, q.skips = L.ptr(w2t, f32, "w2t"), L.ptr(b2, f32, "b2"), L.ptr(out, f32, "x_out"), L.ptr(skips, f32, "skips")
    q.B, q.T, q.R, q.G, q.S, q.Cc = B, T, R, G, skips.shape[1], c.shape[1]
    q.ksize, q.dilation, q.first = int(ksize), int(dilation), int(first)
    p.y = L.ptr(y, f32, "y")
    L.check(L.lib().svsk_wavenet_block_train_f32(C.byref(p), L.stream_ptr()), "wavenet_block_train_f32")
    return out


@functools.lru_cache(maxsize=64)
def wavenet_train_sizes(out_dim, R, G, S, cin, layers, ksize):
    """(floats of the training weight pack, floats of the gradient arena); raises for shapes the block rejects."""
    pack, grad = C.c_longlong(), C.c_longlong()
    rc = L.lib().svsk_wavenet_train_sizes(out_dim, R, G, S, cin, layers, ksize, C.byref(pack), C.byref(grad))
    if rc != 0:
        raise RuntimeError(f"libsvsk wavenet_train_sizes failed (code {rc}): {L.lib().svsk_last_error().decode()}")
    return pack.value, grad.value


@functools.lru_cache(maxsize=64)
def wavenet_train_layout(out_dim, R, G, S, cin, layers, ksize):
    """{name: (offset, shape)} of the weight pack and of the gradient arena (include/svsk.h, svsk_wavenet_train_pack_f32
    and svsk_wavenet_wgrad_f32), checked against wavenet_train_sizes."""
    Ly, k, G2 = layers, ksize, G // 2
    Rp, G2p = (R + 3) // 4 * 4, (G2 + 3) // 4 * 4

    def lay(items):
        out, o = {}, 0
        for name, shape in items:
            out[name] = (o, shape)
            o += math.prod(shape)
        return out, o

    pack, npk = lay([("w1t", (Ly, k * R + cin, G)), ("w2t", (Ly, G2, S + R)), ("wT", (Ly, k * G, Rp)), ("wB", (Ly, R + S, G2p)),
                     ("wcT", (cin, Ly * G, 1)), ("first", (R, out_dim, 1)), ("firstT", (out_dim, R, 1)), ("last1", (S, S, 1)),
                     ("last1T", (S, S, 1)), ("last3", (out_dim, S, 1)), ("last3T", (S, out_dim, 1))])
    grad, ngr = lay([("conv", (Ly, G, R, k)), ("conv_b", (Ly, G)), ("cond", (Ly, G, cin, 1)), ("skip", (Ly, S, G2, 1)),
                     ("skip_b", (Ly, S)), ("out", (Ly, R, G2, 1)), ("out_b", (Ly, R)), ("first", (R, out_dim, 1)),
                     ("first_b", (R,)), ("last1", (S, S, 1)), ("last1_b", (S,)), ("last3", (out_dim, S, 1)), ("last3_b", (out_dim,))])
    if (npk, ngr) != wavenet_train_sizes(out_dim, R, G, S, cin, layers, ksize):
        raise RuntimeError("wavenet_train_layout: layout disagrees with libsvsk")
    return pack, grad


# the weights in the order of svsk_wavenet_wnorm_grad_f32's dg vector
_WN_NAMES = ("first", "conv", "cond", "skip", "out", "last1", "last3")


def _ar_weights_struct(w, out_dim, R, G, S, cin, layers, ksize):
    p = L.WavenetArWeights()
    for n in _AR_WEIGHTS:
        setattr(p, n, L.ptr(w.get(n), f32, n).value)
    p.out_dim, p.R, p.G, p.S, p.cin, p.layers, p.stacks, p.ksize = out_dim, R, G, S, cin, layers, 1, ksize
    return p


def _check_train_weights(w, out_dim, R, G, S, cin, layers, ksize):
    G2 = G // 2
    shapes = {"first": (R, out_dim, 1), "conv": (layers, G, R, ksize), "cond": (layers, G, cin, 1), "skip": (layers, S, G2, 1),
              "out": (layers, R, G2, 1), "last1": (S, S, 1), "last3": (out_dim, S, 1)}
    for n, shp in shapes.items():
        _shape(f"wavenet weights: {n}_v", w.get(n + "_v"), shp)
        if w.get(n + "_g") is not None and w[n + "_g"].numel() != math.prod(shp[:-2]):
            raise ValueError(f"wavenet weights: {n}_g must hold {math.prod(shp[:-2])} gains, got {list(w[n + '_g'].shape)}")


def wavenet_train_pack_f32(w, *, out_dim, R, G, S, cin, layers, ksize):
    """svsk_wavenet_train_pack_f32.  w: the *_v / *_g tensors of svsk_wavenet_ar_weights (fp32, contiguous, stacked over
    the layers; *_g None = no weight norm) -> {name: view} of one pack tensor (wavenet_train_layout)."""
    _check_train_weights(w, out_dim, R, G, S, cin, layers, ksize)
    lay, _ = wavenet_train_layout(out_dim, R, G, S, cin, layers, ksize)
    n = sum(math.prod(s) for _, s in lay.values())
    pack = torch.empty(n, device=w["conv_v"].device, dtype=f32)
    p = _ar_weights_struct(w, out_dim, R, G, S, cin, layers, ksize)
    L.check(L.lib().svsk_wavenet_train_pack_f32(C.byref(p), L.ptr(pack), L.stream_ptr()), "wavenet_train_pack_f32")
    return {k: pack[o:o + math.prod(s)].view(s) for k, (o, s) in lay.items()}


def wavenet_wnorm_grad_f32(w, dW, *, out_dim, R, G, S, cin, layers, ksize):
    """svsk_wavenet_wnorm_grad_f32: turns the effective weights' gradients in dW (the arena of wavenet_wgrad_f32) into
    those of the weight_v tensors, in place, and returns {name: gradient of the gain, shaped like the stacked weight_g}
    for the weights that have a gain."""
    _check_train_weights(w, out_dim, R, G, S, cin, layers, ksize)
    _, ngr = wavenet_train_sizes(out_dim, R, G, S, cin, layers, ksize)
    _shape("wavenet_wnorm_grad_f32: dW", dW, (ngr,))
    rows = {"first": R, "conv": layers * G, "cond": layers * G, "skip": layers * S, "out": layers * R, "last1": S, "last3": out_dim}
    dg = torch.empty(sum(rows.values()), device=dW.device, dtype=f32)
    p = _ar_weights_struct(w, out_dim, R, G, S, cin, layers, ksize)
    L.check(L.lib().svsk_wavenet_wnorm_grad_f32(C.byref(p), L.ptr(dW, f32, "dW"), L.ptr(dg), L.stream_ptr()),
            "wavenet_wnorm_grad_f32")
    out, o = {}, 0
    for n in _WN_NAMES:
        if w.get(n + "_g") is not None:
            out[n] = dg[o:o + rows[n]].view(w[n + "_g"].shape)
        o += rows[n]
    return out


def wavenet_dgrad_f32(*, dy_in, wT, g_next, g_out, dS, y_prev, wB, dy_out, ksize, dilation):
    """svsk_wavenet_dgrad_f32 (one launch of the backward through the blocks).  dy_in / dy_out: [B, G, T] slices of a
    [B, L, G, T] buffer (or None); g_next (or None), g_out [B, R, T]; dS [B, S, T]; y_prev [B, G, T] or None."""
    B, R, T = g_out.shape
    S = dS.shape[1]
    _shape("wavenet_dgrad_f32: dS", dS, (B, S, T))
    if g_next is not None:
        _shape("wavenet_dgrad_f32: g_next", g_next, (B, R, T))
    G = (dy_in if dy_in is not None else y_prev).shape[1] if (dy_in is not None or y_prev is not None) else 0
    bstride = None
    for name, t in (("dy_in", dy_in), ("dy_out", dy_out)):
        if t is not None:
            if t.dim() != 3 or tuple(t.shape) != (B, G, T) or t.stride(2) != 1 or t.stride(1) != T:
                raise ValueError(f"wavenet_dgrad_f32: {name} must be a [{B}, {G}, {T}] slice with rows of T frames")
            if bstride is not None and t.stride(0) != bstride:
                raise ValueError("wavenet_dgrad_f32: dy_in and dy_out must share the batch stride")
            bstride = t.stride(0)
    if y_prev is not None:
        _shape("wavenet_dgrad_f32: y_prev", y_prev, (B, G, T))
        if dy_out is None or wB is None:
            raise ValueError("wavenet_dgrad_f32: y_prev needs wB and dy_out")
        _shape("wavenet_dgrad_f32: wB", wB, (R + S, (G // 2 + 3) // 4 * 4))
    if dy_in is not None:
        _shape("wavenet_dgrad_f32: wT", wT, (ksize * G, (R + 3) // 4 * 4))
    p = L.WavenetDgradParams()

    def sl(t, name):
        if t is None:
            return C.c_void_p(0)
        if not t.is_cuda or t.dtype != f32:
            raise RuntimeError(f"{name} must be a CUDA fp32 tensor")
        return C.c_void_p(t.data_ptr())

    p.dy_in, p.dy_out = sl(dy_in, "dy_in"), sl(dy_out, "dy_out")
    p.wT, p.wB = L.ptr(wT, f32, "wT"), L.ptr(wB, f32, "wB")
    p.g_next, p.g_out, p.dS, p.y_prev = L.ptr(g_next, f32, "g_next"), L.ptr(g_out, f32, "g_out"), L.ptr(dS, f32, "dS"), L.ptr(y_prev, f32, "y_prev")
    p.dy_bstride = bstride if bstride is not None else G * T
    p.B, p.T, p.R, p.G, p.S, p.ksize, p.dilation = B, T, R, G, S, int(ksize), int(dilation)
    L.check(L.lib().svsk_wavenet_dgrad_f32(C.byref(p), L.stream_ptr()), "wavenet_dgrad_f32")


def wavenet_wgrad_splits(B, T, out_dim, R, G, S, cin, layers, ksize, target=2 * 148):
    """Frame splits of svsk_wavenet_wgrad_f32: enough CTAs for about two waves on a B200, at least 8 chunks of 32 frames
    per split."""
    t = lambda M, N: -(-M // 64) * -(-N // 64)
    tiles = layers * (t(G, ksize * R + cin + 1) + t(R, G // 2 + 1) + t(S, G // 2 + 1)) + t(out_dim, S + 1) + t(S, S + 1) + t(R, out_dim + 1)
    chunks = B * -(-T // 32)
    return max(1, min(-(-target // tiles), chunks // 8, 64))


def wavenet_wgrad_f32(*, x_in, c, xs, ys, gs, dy, dS, skips, h1, dh1, glog, dilations, ksize, splits=1):
    """svsk_wavenet_wgrad_f32 -> the gradient arena (wavenet_train_layout's second dict).  Shapes as in include/svsk.h;
    dilations: int32 CUDA tensor [L]."""
    B, out_dim, T = x_in.shape
    cin = c.shape[1]
    Ly, _, R, _ = xs.shape
    G, S = ys.shape[2], dS.shape[1]
    for name, t, shp in (("c", c, (B, cin, T)), ("xs", xs, (Ly, B, R, T)), ("ys", ys, (Ly, B, G, T)), ("gs", gs, (Ly + 1, B, R, T)),
                         ("dy", dy, (B, Ly, G, T)), ("dS", dS, (B, S, T)), ("skips", skips, (B, S, T)), ("h1", h1, (B, S, T)),
                         ("dh1", dh1, (B, S, T)), ("glog", glog, (B, out_dim, T)), ("dilations", dilations, (Ly,))):
        _shape(f"wavenet_wgrad_f32: {name}", t, shp)
    _, ngr = wavenet_train_sizes(out_dim, R, G, S, cin, Ly, ksize)
    dev = x_in.device
    dW = torch.empty(ngr, device=dev, dtype=f32)
    ws = torch.empty(splits * ngr, device=dev, dtype=f32) if splits > 1 else None
    p = L.WavenetWgradParams()
    for name, t in (("x_in", x_in), ("c", c), ("xs", xs), ("ys", ys), ("gs", gs), ("dy", dy), ("dS", dS), ("skips", skips),
                    ("h1", h1), ("dh1", dh1), ("glog", glog)):
        setattr(p, name, L.ptr(t, f32, name).value)
    p.dilations = L.ptr(dilations, torch.int32, "dilations").value
    p.dW, p.ws = L.ptr(dW).value, L.ptr(ws).value
    p.B, p.T, p.out_dim, p.R, p.G, p.S, p.cin, p.layers, p.ksize, p.splits = B, T, out_dim, R, G, S, cin, Ly, int(ksize), int(splits)
    L.check(L.lib().svsk_wavenet_wgrad_f32(C.byref(p), L.stream_ptr()), "wavenet_wgrad_f32")
    return dW


def relu_mask_f32(x, m, out=None):
    """svsk_relu_mask_f32: x where m > 0, else 0 (out may be x)."""
    _shape("relu_mask_f32: m", m, x.shape)
    out = torch.empty_like(x) if out is None else out
    _shape("relu_mask_f32: out", out, x.shape)
    L.check(L.lib().svsk_relu_mask_f32(L.ptr(x, f32, "x"), L.ptr(m, f32, "m"), L.ptr(out, f32, "out"), x.numel(), L.stream_ptr()),
            "relu_mask_f32")
    return out


def usfgan_source(f0, *, hop, sample_rate, dense_factor=4, sine_amp=0.1, noise_amp=0.0, noise=None, sine_out=None,
                  want_sine=True, want_d=True):
    """f0 [B, F] float64 CUDA (Hz, 0 = unvoiced) -> (sine [B, 1, F*hop] fp32 or None, d [B, 1, F*hop] fp32 or None): the
    sine-based source signal (with `noise` [B, 1, F*hop] added at noise_amp / noise_amp/3) and the dilation factors.
    sine_out: optional [B, Cs, F*hop] fp32 tensor whose channel 0 receives the sine (the generator's in_signal)."""
    B, F = f0.shape
    T = F * int(hop)
    dev = f0.device
    sine, stride = None, 0
    if want_sine:
        if sine_out is None:
            sine_out = torch.empty((B, 1, T), device=dev, dtype=f32)
        if sine_out.dim() != 3 or sine_out.shape[0] != B or sine_out.shape[2] != T or not sine_out.is_contiguous():
            raise ValueError(f"usfgan_source: sine_out must be a contiguous [B={B}, channels, T={T}] tensor")
        sine, stride = sine_out, sine_out.stride(0)
    if noise_amp > 0 and want_sine and (noise is None or noise.numel() != B * T):
        raise ValueError("usfgan_source: noise_amp > 0 needs the Gaussian draws, [B, 1, T]")
    d = torch.empty((B, 1, T), device=dev, dtype=f32) if want_d else None
    scratch = torch.empty((B, F), device=dev, dtype=torch.float64)
    L.check(L.lib().svsk_usfgan_source(L.ptr(f0, torch.float64, "f0"), L.ptr(noise, f32, "noise") if noise_amp > 0 else C.c_void_p(0),
                                       L.ptr(sine, f32, "sine_out"), stride, L.ptr(d, f32), L.ptr(scratch), B, F, int(hop),
                                       int(sample_rate), int(dense_factor), float(sine_amp), float(noise_amp), L.stream_ptr()),
            "usfgan_source")
    return sine, d


# ------------------------------------------------------------------------------------------------ training kernels
SEG_PLAIN, SEG_GATE_FWD, SEG_RES_SKIP, SEG_GATE_BWD, SEG_ADD_SCALE = 0, 1, 2, 3, 4


def seggemm_bf16(segments, wp, *, mode, bias=None, in0=None, mask=None, dp_next=None, out0=None, out1=None, outf=None,
                 alpha=1.0, act=ACT_NONE, init=True, accumulate=False):
    """D[b,t,n] = sum_s x_s[b, t + shift_s, :kx_s] . wp[n, koff_s:koff_s + kx_s]  with the epilogue `mode` of
    svsk_seggemm_bf16.  segments: list of (x [B,T,ld] bf16, kx, shift); wp [Nrows, sum kx] bf16."""
    x0 = segments[0][0]
    B, T = x0.shape[0], x0.shape[1]
    p = L.SegGemmParams()
    p.nseg = len(segments)
    for s, (x, kx, shift) in enumerate(segments):
        if x.shape[0] != B or x.shape[1] != T:
            raise ValueError("seggemm_bf16: all segments must be [B, T, .]")
        p.x[s] = L.ptr(x, bf16, f"segment {s}").value
        p.ldx[s], p.kx[s], p.shift[s] = x.shape[2], int(kx), int(shift)
    if wp.shape[1] != sum(int(k) for _, k, _ in segments):
        raise ValueError(f"seggemm_bf16: wp has K = {wp.shape[1]}, segments sum to {sum(int(k) for _, k, _ in segments)}")
    p.wp = L.ptr(wp, bf16, "wp")
    p.Nrows, p.B, p.T, p.mode = wp.shape[0], B, T, int(mode)
    p.C = wp.shape[0] // 2 if mode == SEG_RES_SKIP else wp.shape[0]
    p.init, p.act, p.accumulate, p.alpha = int(init), int(act), int(accumulate), float(alpha)
    p.bias, p.dp_next = L.ptr(bias, f32, "bias"), L.ptr(dp_next, f32, "dp_next")
    for name, t in (("in0", in0), ("mask", mask), ("out0", out0), ("out1", out1)):
        setattr(p, name, L.ptr(t, bf16, name))
        setattr(p, "ld_" + name, 0 if t is None else t.shape[-1])
    p.outf, p.ld_outf = L.ptr(outf, f32, "outf"), 0 if outf is None else outf.shape[-1]
    L.check(L.lib().svsk_seggemm_bf16(C.byref(p), L.stream_ptr()), "seggemm_bf16")


def wgrad_bf16(p_nct, q_segments, dW, *, T, accumulate=False):
    """dW[..., n, koff_s + k] (+)= sum_{b,t} p[b, n, t] q_s[b, k, t + shift_s].  p_nct [B, Prows, Tp] bf16,
    q_segments: list of (q [B, rows, Tp] bf16, shift); dW [Prows, >= sum rows] fp32 — or [S, Prows, ld]: the tracks are
    cut into S groups whose partial results land in dW[0] .. dW[S-1] (sum them; more CTAs, still no atomics)."""
    B, Prows, Tp = p_nct.shape
    p = L.WgradParams()
    p.p = L.ptr(p_nct, bf16, "p")
    p.nseg = len(q_segments)
    for s, (q, shift) in enumerate(q_segments):
        if q.shape[0] != B or q.shape[2] != Tp:
            raise ValueError("wgrad_bf16: operands must share B and the time pitch")
        p.q[s] = L.ptr(q, bf16, f"q {s}").value
        p.qrows[s], p.shift[s] = q.shape[1], int(shift)
    p.Prows, p.B, p.T, p.Tp, p.ldw, p.accumulate = Prows, B, int(T), Tp, dW.shape[-1], int(accumulate)
    p.splits, p.split_stride = (dW.shape[0], dW.stride(0)) if dW.dim() == 3 else (1, 0)
    if dW.shape[-2] != Prows:
        raise ValueError(f"wgrad_bf16: dW has {dW.shape[-2]} rows, p has {Prows}")
    p.dW = L.ptr(dW, f32, "dW")
    L.check(L.lib().svsk_wgrad_bf16(C.byref(p), L.stream_ptr()), "wgrad_bf16")


def wgrad_splits(B, tiles, budget=160):
    """How many track groups a wgrad launch of `tiles` CTAs per group should use: the largest divisor of B that keeps the
    grid within about one wave (the kernel is bound by what ONE SM can pull from L2, so it wants many CTAs)."""
    best = 1
    for s in range(1, B + 1):
        if B % s == 0 and tiles * s <= budget:
            best = s
    return best


def ntc_to_nct_bf16(x, N=None, out=None, row0=0, shifts=(0,)):
    """out[b, row0 + j * N + n, t] = x[b, t + shifts[j], n] for every t < Tp, 0 where frame t + shifts[j] is outside
    [0, T), for up to three shifts: x [B, T, ld] bf16 (first N columns), out [B, rows, Tp] bf16 (Tp = T rounded up to 8;
    a fresh `out` has exactly len(shifts) * N rows).  The padding columns t in [T, Tp) follow the same rule, so they hold
    x[t + shift] wherever that frame exists: they are not zero, and svsk_wgrad_bf16 never reads them.  The other rows of
    `out` are left as they are."""
    B, T, ld = x.shape
    N = ld if N is None else N
    Tp = (T + 7) // 8 * 8
    if out is None:
        out = torch.empty((B, len(shifts) * N, Tp), device=x.device, dtype=bf16)
    sh = (C.c_int * 3)(*([int(v) for v in shifts] + [0] * (3 - len(shifts))))
    L.check(L.lib().svsk_ntc_to_nct_bf16(L.ptr(x, bf16, "x"), L.ptr(out, bf16, "out"), B, T, N, ld, out.shape[2], out.shape[1],
                                         int(row0), len(shifts), sh, L.stream_ptr()), "ntc_to_nct_bf16")
    return out


def diffnet_train_pack(wd, wc, wo):
    """Stacked fp32 parameters (wd [L,2C,C,3], wc [L,2C,H], wo [L,2C,C]) -> dict of the bf16 operands of the training kernels."""
    Ln, C2, Cc, _ = wd.shape
    H = wc.shape[2]
    dev = wd.device
    out = dict(w1p=torch.empty((Ln, C2, 3 * Cc + H), device=dev, dtype=bf16), woutp=torch.empty((Ln, C2, Cc), device=dev, dtype=bf16),
               woutT=torch.empty((Ln, Cc, C2), device=dev, dtype=bf16), w1T=torch.empty((Ln, Cc, 3 * C2), device=dev, dtype=bf16),
               wcT=torch.empty((Ln, H, C2), device=dev, dtype=bf16))
    L.check(L.lib().svsk_diffnet_train_pack(L.ptr(wd, f32, "wd"), L.ptr(wc, f32, "wc"), L.ptr(wo, f32, "wo"),
                                            L.ptr(out["w1p"]), L.ptr(out["woutp"]), L.ptr(out["woutT"]), L.ptr(out["w1T"]),
                                            L.ptr(out["wcT"]), Ln, Cc, H, L.stream_ptr()), "diffnet_train_pack")
    return out


def diffnet_stack_fits(B, T, Cc, H):
    """True if the one-launch residual stack (svsk_diffnet_stack_bf16) can hold all its CTA pairs on the device at once."""
    return L.lib().svsk_diffnet_stack_fits(int(B), int(T), int(Cc), int(H)) == 1


def diffnet_stack_uses_pcond(B, T, Cc, H):
    """True if svsk_diffnet_stack_bf16 would use a precomputed conditioner projection for this shape."""
    return L.lib().svsk_diffnet_stack_uses_pcond(int(B), int(T), int(Cc), int(H)) == 1


def diffnet_cond_project(cond, wcp):
    """cond [B,T,H] bf16, wcp [nblk,256,H] bf16 -> p [nblk, B*T, 256] bf16 in one launch."""
    B, T, H = cond.shape
    nblk = wcp.shape[0]
    p = torch.empty((nblk, B * T, 256), device=cond.device, dtype=bf16)
    L.check(L.lib().svsk_diffnet_cond_project_bf16(L.ptr(cond, bf16, "cond"), L.ptr(wcp, bf16, "wcp"), L.ptr(p), B * T, H, nblk,
                                                   L.stream_ptr()), "diffnet_cond_project_bf16")
    return p


def diffnet_pcond_pack(p, B, T, nl, Cc):
    """p [L*2C/256, B*T, 256] bf16 (packed column order per output block) -> (pcond_gate [B,L,T,C],
    pcond_filt [B, tiles, L, 2C/256, 8, 128, 16]) for diffnet_stack_bf16(pcond=...)."""
    NB = Cc // 128
    tiles = 2 * ((T + 255) // 256)
    if tuple(p.shape) != (nl * NB, B * T, 256):
        raise ValueError(f"diffnet_pcond_pack: p must be [{nl * NB}, {B * T}, 256], got {tuple(p.shape)}")
    pg = torch.empty((B, nl, T, Cc), device=p.device, dtype=bf16)
    pf = torch.empty((B, tiles, nl, NB, 8, 128, 16), device=p.device, dtype=bf16)
    L.check(L.lib().svsk_diffnet_pcond_pack_bf16(L.ptr(p, bf16, "p"), L.ptr(pg), L.ptr(pf), B, T, nl, Cc, L.stream_ptr()),
            "diffnet_pcond_pack_bf16")
    return pg, pf


def diffnet_stack_bf16(xb_in, edge0, edge1, skip32, cond, w1p_all, woutp_all, stepbias, bout_all, flags, dilations, *,
                       stepbias_batch_stride, stepbias_layer_stride, init_skip=True, pcond=None):
    """All residual blocks in one launch.  w1p_all [L,2C,3C+H], woutp_all [L,2C,C], bout_all [L,2C]; stepbias: any fp32
    tensor whose element (layer l, batch row b) row starts at l*layer_stride + b*batch_stride floats.  pcond: optional
    (pcond_gate, pcond_filt) of diffnet_pcond_pack for the same tracks (the conditioner projection computed once per
    sampling run instead of inside every call)."""
    B, T, Cc = xb_in.shape
    nl = w1p_all.shape[0]
    p = L.DiffnetStackParams()
    p.xb_in, p.edge0, p.edge1 = L.ptr(xb_in, bf16, "xb_in"), L.ptr(edge0, bf16, "edge0"), L.ptr(edge1, bf16, "edge1")
    p.skip32, p.cond = L.ptr(skip32, f32, "skip32"), L.ptr(cond, bf16, "cond")
    p.w1p, p.woutp = L.ptr(w1p_all, bf16, "w1p"), L.ptr(woutp_all, bf16, "woutp")
    if not stepbias.is_cuda or stepbias.dtype != f32:
        raise RuntimeError("stepbias must be a CUDA float32 tensor")
    p.stepbias, p.bout = C.c_void_p(stepbias.data_ptr()), L.ptr(bout_all, f32, "bout")
    p.flags = L.ptr(flags, torch.int32, "flags")
    if flags.numel() < B * 2 * ((T + 255) // 256):
        raise ValueError("diffnet_stack_bf16: flags too small")
    dil = (C.c_int32 * nl)(*[int(d) for d in dilations])
    p.dilation = C.cast(dil, C.POINTER(C.c_int32))
    p.B, p.T, p.C, p.H, p.L = B, T, Cc, cond.shape[2], nl
    p.stepbias_batch_stride, p.stepbias_layer_stride = int(stepbias_batch_stride), int(stepbias_layer_stride)
    p.init_skip = int(init_skip)
    if pcond is not None:
        pg, pf = pcond
        if tuple(pg.shape) != (B, nl, T, Cc) or pf.shape[0] != B or not pg.is_contiguous() or not pf.is_contiguous():
            raise ValueError("diffnet_stack_bf16: pcond does not match the batch")
        p.pcond_gate, p.pcond_filt = L.ptr(pg, bf16, "pcond_gate"), L.ptr(pf, bf16, "pcond_filt")
    L.check(L.lib().svsk_diffnet_stack_bf16(C.byref(p), L.stream_ptr()), "diffnet_stack_bf16")


def upsample_fused_supported(scales, A):
    hop = 1
    for sc in scales:
        hop *= int(sc)
    return (1 <= len(scales) <= 6 and all(2 <= int(sc) <= 16 for sc in scales) and A <= 128
            and sum(2 * int(sc) + 1 for sc in scales) <= 128 and 127 // hop + 2 * len(scales) + 4 <= 48)


def upsample_fused(c, taps, scales, *, want_bf16=True, want_f32=False):
    """UpsampleNetwork in one pass: c [B,A,F] fp32 -> NTC [B, F*prod(scales), Ap] (bf16 and/or fp32), Ap = A rounded up to 8."""
    B, A, F = c.shape
    hop = 1
    for sc in scales:
        hop *= int(sc)
    Ap = (A + 7) // 8 * 8
    ob = torch.empty((B, F * hop, Ap), device=c.device, dtype=bf16) if want_bf16 else None
    of = torch.empty((B, F * hop, Ap), device=c.device, dtype=f32) if want_f32 else None
    sc = (C.c_int32 * len(scales))(*[int(x) for x in scales])
    L.check(L.lib().svsk_upsample_fused(L.ptr(c, f32, "c"), L.ptr(taps, f32, "taps"), sc, len(scales), B, A, F, L.ptr(ob, bf16),
                                        L.ptr(of, f32), Ap, L.stream_ptr()), "upsample_fused")
    return ob, of


def expand1_bf16(x_row, w, bias, Cc):
    """x_row: [B, T] fp32 view whose rows are contiguous (any batch stride) -> [B, T, Cc] bf16 = w * x + bias."""
    B, T = x_row.shape
    if not x_row.is_cuda or x_row.dtype != f32 or x_row.stride(1) != 1:
        raise RuntimeError("expand1_bf16: x_row must be a CUDA float32 [B, T] view with unit time stride")
    out = torch.empty((B, T, Cc), device=x_row.device, dtype=bf16)
    L.check(L.lib().svsk_expand1_bf16(C.c_void_p(x_row.data_ptr()), x_row.stride(0) if B > 1 else T, L.ptr(w, f32, "w"),
                                      L.ptr(bias, f32, "bias"), L.ptr(out), B, T, Cc, L.stream_ptr()), "expand1_bf16")
    return out


def diffnet_step_bf16(skip32, x32s, z, t, tables, w_skip, b_skip, w_out, b_out, *, skip_scale, w_in=None, b_in=None, xb_out=None,
                      eps_out=None, clip_denoised=True):
    """Tail projections + DDPM update (x32s in place) + the next call's input projection (into xb_out, if given).
    tables: the five schedule vectors of ddpm_update_f32, in its order."""
    B, T, Cc = skip32.shape
    p = L.DiffnetStepParams()
    p.skip32, p.x32s, p.z = L.ptr(skip32, f32, "skip32"), L.ptr(x32s, f32, "x32s"), L.ptr(z, f32, "z")
    p.eps_out, p.xb_out = L.ptr(eps_out, f32, "eps_out"), L.ptr(xb_out, bf16, "xb_out")
    p.w_skip, p.w_out, p.w_in = L.ptr(w_skip, bf16, "w_skip"), L.ptr(w_out, bf16, "w_out"), L.ptr(w_in, bf16, "w_in")
    p.b_skip, p.b_out, p.b_in = L.ptr(b_skip, f32, "b_skip"), L.ptr(b_out, f32, "b_out"), L.ptr(b_in, f32, "b_in")
    p.t = L.ptr(t, torch.int64, "t")
    p.sra, p.srm1, p.c1, p.c2, p.plv = [L.ptr(x, f32, "schedule table") for x in tables]
    p.skip_scale = float(skip_scale)
    p.B, p.T, p.C, p.Mp, p.clip_denoised = B, T, Cc, x32s.shape[2], int(clip_denoised)
    L.check(L.lib().svsk_diffnet_step_bf16(C.byref(p), L.stream_ptr()), "diffnet_step_bf16")


def linear_bf16(a, w, bias=None, *, act=ACT_NONE, want_bf16=False, want_f32=False, out_bf16=None, out_f32=None):
    """a [..., K] bf16 (row-major rows), w [Cout, K] bf16 -> [..., Cout]."""
    K = a.shape[-1]
    N = a.numel() // K
    Cout = w.shape[0]
    lead = a.shape[:-1]
    if want_bf16 and out_bf16 is None:
        out_bf16 = torch.empty((*lead, Cout), device=a.device, dtype=bf16)
    if want_f32 and out_f32 is None:
        out_f32 = torch.empty((*lead, Cout), device=a.device, dtype=f32)
    p = L.LinearBf16Params()
    p.a, p.w, p.bias = L.ptr(a, bf16, "a"), L.ptr(w, bf16, "w"), L.ptr(bias, f32, "bias")
    p.y_bf16, p.y_f32 = L.ptr(out_bf16, bf16), L.ptr(out_f32, f32)
    p.N, p.K, p.Cout = N, K, Cout
    p.lda, p.ldy_b, p.ldy_f, p.act = K, Cout, Cout, act
    L.check(L.lib().svsk_linear_bf16(C.byref(p), L.stream_ptr()), "linear_bf16")
    return out_bf16, out_f32


def ntc_bf16_to_nct_f32(x, Cc):
    B, T, Cp = x.shape
    y = torch.empty((B, Cc, T), device=x.device, dtype=f32)
    L.check(L.lib().svsk_ntc_bf16_to_nct_f32(L.ptr(x, bf16, "x"), L.ptr(y), B, Cc, T, Cp, L.stream_ptr()),
            "ntc_bf16_to_nct_f32")
    return y


def usfgan_pack_block(w_taps, w_aux, w_out):
    """w_taps [128,64,3] (k=3 conv, or stacked convP/convC/convF), w_aux [128,A] (A % 8 == 0) or None (frame-rate aux
    projection: the block's w1p holds the taps only), w_out [64,64] -> bf16."""
    G, Cc, _ = w_taps.shape
    A = 0 if w_aux is None else w_aux.shape[1]
    Ap = (A + 63) // 64 * 64
    w1p = torch.empty((G, 3 * Cc + Ap), device=w_taps.device, dtype=bf16)
    woutp = torch.empty((Cc, G // 2), device=w_taps.device, dtype=bf16)
    L.check(L.lib().svsk_usfgan_pack_block(L.ptr(w_taps.contiguous(), f32),
                                           None if w_aux is None else L.ptr(w_aux.contiguous(), f32),
                                           L.ptr(w_out.contiguous(), f32), L.ptr(w1p), L.ptr(woutp), Cc, A, G,
                                           L.stream_ptr()), "usfgan_pack_block")
    return w1p, woutp


class UsfganAuxFrames:
    """Operands of the frame-rate aux projection of one generator call (csrc/usfgan_fr.cuh): ``u`` [ceil128(T), 16] bf16,
    ``q`` [B, R, q_ld] bf16 (R = 128 x blocks, in the order the stacks were listed), and the window geometry."""

    def __init__(self, u, q, q_fpad, hop, reach):
        self.u, self.q, self.q_fpad, self.hop, self.reach = u, q, int(q_fpad), int(hop), int(reach)

    def block(self, index):
        """(aux_q view of block ``index``, batch stride in elements, q_ld)."""
        return self.q[:, 128 * index:128 * (index + 1)], self.q.stride(0), self.q.stride(1)


def usfgan_frame_window_ok(hop, reach):
    """A 128-sample tile must fit its frames into the 16-frame window (8 for the reach + 7 of alignment slack)."""
    return hop >= 1 and (127 + 2 * reach) // hop <= 7 and 2 * reach < 15 * hop


def usfgan_aux_frames(cin_ntc, w_all, Tf, T, hop, reach):
    """cin_ntc [B, Tf, Ap] bf16 (conv_in's output, channel-last), w_all [R, Ap] bf16 -> q [B, R, q_ld] bf16 with frame f at
    column q_fpad + f and zeros elsewhere (svsk_usfgan_aux_frames)."""
    B, Tf_, Ap = cin_ntc.shape
    assert Tf_ == Tf
    R = w_all.shape[0]
    fpad = -L.lib().svsk_usfgan_frame_base(0, int(reach), int(hop))
    last = L.lib().svsk_usfgan_frame_base((T - 1) // 128 * 128, int(reach), int(hop))
    q_ld = (max(fpad + Tf, fpad + last + 16) + 7) // 8 * 8
    q = torch.empty((B, R, q_ld), device=cin_ntc.device, dtype=bf16)   # 0.5 GB at config 3: only the pad columns are zeroed
    q[:, :, :fpad].zero_()
    q[:, :, fpad + Tf:].zero_()
    L.check(L.lib().svsk_usfgan_aux_frames(L.ptr(cin_ntc, bf16, "cin"), L.ptr(w_all, bf16, "w_all"), L.ptr(q), B, Tf, Ap, R,
                                           q_ld, fpad, L.stream_ptr()), "usfgan_aux_frames")
    return q, fpad


def usfgan_aux_weights(imp, hop, reach):
    """imp [16, T] fp32 (the upsampler applied to unit impulses at the frames f = channel mod 16) -> u [ceil128(T), 16]
    bf16 (svsk_usfgan_aux_weights)."""
    T = imp.shape[1]
    u = torch.empty(((T + 127) // 128 * 128, 16), device=imp.device, dtype=bf16)
    L.check(L.lib().svsk_usfgan_aux_weights(L.ptr(imp, f32, "imp"), L.ptr(u), T, int(hop), int(reach), L.stream_ptr()),
            "usfgan_aux_weights")
    return u


def upsample_frames_bf16(imp, cin, T, hop, reach, Ap=None):
    """imp [16, T] fp32 (as for usfgan_aux_weights), cin [B, A, Tf] fp32 (conv_in's output) -> upsampled aux features
    [B, T, Ap] bf16 channel-last (svsk_upsample_frames_bf16)."""
    B, A, Tf = cin.shape
    Ap = (A + 7) // 8 * 8 if Ap is None else Ap
    out = torch.empty((B, T, Ap), device=cin.device, dtype=bf16)
    L.check(L.lib().svsk_upsample_frames_bf16(L.ptr(imp, f32, "imp"), L.ptr(cin, f32, "cin"), L.ptr(out), B, A, Ap, Tf, int(T),
                                              int(hop), int(reach), L.stream_ptr()), "upsample_frames_bf16")
    return out


def conv1d_pack_bf16(w):
    """w [Cout,Cin,k] fp32 -> [Cout, k*ceil64(Cin)] bf16 (tap-major K)."""
    Cout, Cin, k = w.shape
    wp = torch.empty((Cout, k * ((Cin + 63) // 64 * 64)), device=w.device, dtype=bf16)
    L.check(L.lib().svsk_conv1d_pack_bf16(L.ptr(w.contiguous(), f32), L.ptr(wp), Cout, Cin, k, L.stream_ptr()),
            "conv1d_pack_bf16")
    return wp


def conv1d_bf16(x, wp, bias, Cout, ksize, *, dilation=1, tap_origin=None, pad_mode=PAD_ZEROS, act=ACT_NONE, out=None):
    """x [B,T,Cin] bf16 NTC -> [B,T,Cout] bf16 on the tcgen05 conv kernel."""
    B, T, Cin = x.shape
    if tap_origin is None:
        tap_origin = (ksize - 1) // 2
    out = torch.empty((B, T, Cout), device=x.device, dtype=bf16) if out is None else out
    p = L.Conv1dBf16Params()
    p.x, p.wp, p.bias, p.y = L.ptr(x, bf16, "x"), L.ptr(wp, bf16, "wp"), L.ptr(bias, f32, "bias"), L.ptr(out, bf16, "out")
    p.B, p.T, p.Cin, p.Cout = B, T, Cin, Cout
    p.ksize, p.dilation, p.tap_origin, p.pad_mode, p.act = ksize, dilation, tap_origin, pad_mode, act
    L.check(L.lib().svsk_conv1d_bf16(C.byref(p), L.stream_ptr()), "conv1d_bf16")
    return out


def periodic_mix_bf16(a, h, n):
    s = torch.empty_like(h)
    L.check(L.lib().svsk_periodic_mix_bf16(L.ptr(a, bf16), L.ptr(h, bf16), L.ptr(n, bf16), L.ptr(s), h.numel(),
                                           L.stream_ptr()), "periodic_mix_bf16")
    return s


def dot_rows_bf16(x, w, bias):
    """x [..., C] bf16, w [C] fp32 -> [...] fp32."""
    Cc = x.shape[-1]
    y = torch.empty(x.shape[:-1], device=x.device, dtype=f32)
    L.check(L.lib().svsk_dot_rows_bf16(L.ptr(x, bf16), L.ptr(w, f32), float(bias), L.ptr(y), y.numel(), Cc,
                                       L.stream_ptr()), "dot_rows_bf16")
    return y


def usfgan_block_bf16(xb_in, xb_out, aux, w1p, woutp, bias1, bout, *, dilation=1, idx=None, out_scale=math.sqrt(0.5),
                      out_relu=False, frames=None, frames_block=0):
    """One fused uSFGAN Fixed / Adaptive block (svsk_usfgan_block_bf16).  ``aux`` [B,T,A8] bf16 at sample rate, or
    ``frames`` (UsfganAuxFrames) + ``frames_block`` for the frame-rate aux projection (then w1p holds the taps only)."""
    B, T, Cc = xb_in.shape
    p = L.UsfganBlockParams()
    p.xb_in, p.xb_out = L.ptr(xb_in, bf16, "xb_in"), L.ptr(xb_out, bf16, "xb_out")
    p.w1p, p.woutp = L.ptr(w1p, bf16), L.ptr(woutp, bf16)
    p.bias1, p.bout = L.ptr(bias1, f32), L.ptr(bout, f32)
    if idx is not None:
        p.idx_past, p.idx_future = L.ptr(idx[0], torch.int32), L.ptr(idx[1], torch.int32)
    p.B, p.T = B, T
    if frames is not None:
        qv, qbs, qld = frames.block(frames_block)
        if frames.q.shape[0] != B or frames.u.shape[0] < (T + 127) // 128 * 128:
            raise RuntimeError(f"usfgan_block_bf16: frame-rate aux operands are for another shape (q {tuple(frames.q.shape)}, "
                               f"u {tuple(frames.u.shape)}, x {tuple(xb_in.shape)})")
        p.aux_u, p.aux_q = frames.u.data_ptr(), qv.data_ptr()
        p.q_batch_stride, p.q_ld, p.q_fpad, p.hop, p.reach = qbs, qld, frames.q_fpad, frames.hop, frames.reach
        p.A = 0
    else:
        p.aux = L.ptr(aux, bf16, "aux")
        p.A = aux.shape[2]
    p.dilation, p.adaptive, p.out_scale = int(dilation), int(idx is not None), float(out_scale)
    p.out_relu = int(out_relu)
    L.check(L.lib().svsk_usfgan_block_bf16(C.byref(p), L.stream_ptr()), "usfgan_block_bf16")


# ---- FFConvLSTM encoder pieces (include/svsk.h, "FFConvLSTM encoder pieces") ---------------------------------------
def lstm_supported(H):
    return bool(L.lib().svsk_lstm_supported(int(H)))


def lstm_f32(pre, w_hh, lengths, H, *, pre_layout, h_f32=None, h_bf16=None):
    """svsk_lstm_f32.  pre: gate pre-activations of both directions, ``pre_layout`` "ntc" = [B, T, ndir*4H] or "nct" =
    [B, ndir*4H, T] (fp32); w_hh [ndir, 4H, H]; lengths int32 [B] or None.  h_f32: [B, 2H, T] (NCT) output or None;
    h_bf16: [B, T, >= 2H] bf16 output or None."""
    ndir = w_hh.shape[0]
    if pre_layout == "ntc":
        B, T, R = pre.shape
        sb, st_, sr = T * R, R, 1
    elif pre_layout == "nct":
        B, R, T = pre.shape
        sb, st_, sr = T * R, 1, T
    else:
        raise ValueError("pre_layout must be 'ntc' or 'nct'")
    if R != ndir * 4 * H or tuple(w_hh.shape) != (ndir, 4 * H, H):
        raise RuntimeError(f"lstm_f32: pre has {R} gate rows, w_hh is {tuple(w_hh.shape)}; expected {ndir * 4 * H} and ({ndir}, {4 * H}, {H})")
    p = L.LstmParams()
    p.pre, p.w_hh, p.lengths = L.ptr(pre, f32, "pre"), L.ptr(w_hh, f32, "w_hh"), L.ptr(lengths, torch.int32, "lengths")
    p.pre_stride_b, p.pre_stride_t, p.pre_stride_r = sb, st_, sr
    if h_f32 is not None:
        if tuple(h_f32.shape) != (B, ndir * H, T):
            raise RuntimeError("lstm_f32: h_f32 must be [B, ndir*H, T]")
        p.h_f32 = L.ptr(h_f32, f32, "h_f32")
        p.hf_stride_b, p.hf_stride_t, p.hf_stride_c = ndir * H * T, 1, T
    if h_bf16 is not None:
        if h_bf16.shape[0] != B or h_bf16.shape[1] != T or h_bf16.shape[2] < ndir * H:
            raise RuntimeError("lstm_f32: h_bf16 must be [B, T, >= ndir*H]")
        p.h_bf16 = L.ptr(h_bf16, bf16, "h_bf16")
        p.hb_stride_b, p.hb_stride_t = T * h_bf16.shape[2], h_bf16.shape[2]
    p.B, p.T, p.H, p.ndir = B, T, H, ndir
    L.check(L.lib().svsk_lstm_f32(C.byref(p), L.stream_ptr()), "lstm_f32")


def tapgemm_pack_bf16(w, scale=None):
    """w [Cout, Cin, k] (or [Cout, Cin]) fp32 -> packed [k, Cout, ceil64(Cin)] bf16 with ``scale`` [Cout] folded in."""
    if w.dim() == 2:
        w = w.unsqueeze(-1)
    w = w.contiguous()
    Cout, Cin, k = w.shape
    wp = torch.empty((k, Cout, (Cin + 63) // 64 * 64), device=w.device, dtype=bf16)
    L.check(L.lib().svsk_tapgemm_pack_bf16(L.ptr(w, f32, "w"), L.ptr(scale, f32, "scale"), L.ptr(wp), Cout, Cin, k,
                                           L.stream_ptr()), "tapgemm_pack_bf16")
    return wp


def tapgemm_bf16(x, wp, bias, Cin, *, T, act=ACT_NONE, y_bf16=None, y_row0=0, y_f32=None):
    """svsk_tapgemm_bf16.  x [B, Tp_x, ldx] bf16 (time-padded by the caller), wp from tapgemm_pack_bf16;
    y_bf16 [B, Tp_y, ldy_b] receives frame t at row y_row0 + t; y_f32 [B, T, ldy_f]."""
    B, Tp_x, ldx = x.shape
    k, Cout, _ = wp.shape
    p = L.TapGemmBf16Params()
    p.x, p.wp, p.bias = L.ptr(x, bf16, "x"), L.ptr(wp, bf16, "wp"), L.ptr(bias, f32, "bias")
    p.B, p.T, p.Cin, p.Cout, p.ksize, p.Tp_x, p.ldx, p.act = B, T, Cin, Cout, k, Tp_x, ldx, act
    if y_bf16 is not None:
        p.y_bf16, p.Tp_y, p.y_row0, p.ldy_b = L.ptr(y_bf16, bf16, "y_bf16"), y_bf16.shape[1], y_row0, y_bf16.shape[2]
    if y_f32 is not None:
        if y_f32.shape[0] != B or y_f32.shape[1] != T:
            raise RuntimeError("tapgemm_bf16: y_f32 must be [B, T, ldy_f]")
        p.y_f32, p.ldy_f = L.ptr(y_f32, f32, "y_f32"), y_f32.shape[2]
    L.check(L.lib().svsk_tapgemm_bf16(C.byref(p), L.stream_ptr()), "tapgemm_bf16")


def reflect_pad_rows_bf16(buf, T, pad):
    B, Tp, Cc = buf.shape
    L.check(L.lib().svsk_reflect_pad_rows_bf16(L.ptr(buf, bf16, "buf"), B, Tp, Cc, T, pad, L.stream_ptr()), "reflect_pad_rows_bf16")


def encoder_front(x, onehot_start, onehot_len, *, y_f32=None, y_bf16=None):
    """x [rows, in_dim] fp32 -> copies with the one-hot block replaced by one-hot(argmax) (svsk_encoder_front)."""
    rows, in_dim = x.shape
    L.check(L.lib().svsk_encoder_front(L.ptr(x, f32, "x"), L.ptr(y_f32, f32, "y_f32"), L.ptr(y_bf16, bf16, "y_bf16"), rows, in_dim,
                                       onehot_start, onehot_len, 0 if y_f32 is None else y_f32.shape[1],
                                       0 if y_bf16 is None else y_bf16.shape[1], L.stream_ptr()), "encoder_front")


def batchnorm_train_f32(x, gamma, beta, running_mean, running_var, *, eps, momentum, relu=True, out=None, stats=None):
    """nn.BatchNorm1d in training mode (+ ReLU) on x [B, C, T] fp32: batch statistics over all B*T positions, running
    buffers updated as torch does (svsk_bn_batch_stats_f32 + svsk_bn_apply_f32).  In place unless ``out`` [B, C, T] is
    given (x is then kept, as the backward needs it); ``stats``: (mean, var) [C] tensors that receive the batch
    statistics.  Returns the output."""
    B, Cc, T = x.shape
    if out is None:
        out = x
    _shape("batchnorm_train_f32: out", out, x.shape)
    if stats is None:
        stats = (torch.empty((Cc,), device=x.device, dtype=f32), torch.empty((Cc,), device=x.device, dtype=f32))
    mean, var = stats
    _shape("batchnorm_train_f32: mean", mean, (Cc,))
    _shape("batchnorm_train_f32: var", var, (Cc,))
    L.check(L.lib().svsk_bn_batch_stats_f32(L.ptr(x, f32, "x"), B, Cc, T, L.ptr(mean), L.ptr(var), L.ptr(running_mean, f32),
                                            L.ptr(running_var, f32), float(momentum), L.stream_ptr()), "bn_batch_stats_f32")
    L.check(L.lib().svsk_bn_apply_f32(L.ptr(x, f32, "x"), L.ptr(out, f32, "out"), L.ptr(mean), L.ptr(var), L.ptr(gamma, f32),
                                      L.ptr(beta, f32), float(eps), int(relu), B, Cc, T, L.stream_ptr()), "bn_apply_f32")
    return out


# ---- FFConvLSTM encoder training (include/svsk.h, "FFConvLSTM encoder training") ------------------------------------
def lstm_train_f32(pre, w_hh, lengths, H, *, h_f32, gates, cell):
    """svsk_lstm_train_f32: lstm_f32 with pre [B, ndir*4H, T] ("nct") and h_f32 [B, ndir*H, T] that also writes the
    activated gates [B, ndir*4H, T] and the cell states [B, ndir*H, T] the backward needs."""
    ndir = w_hh.shape[0]
    B, R, T = pre.shape
    _shape("lstm_train_f32: w_hh", w_hh, (ndir, 4 * H, H))
    _shape("lstm_train_f32: pre", pre, (B, ndir * 4 * H, T))
    _shape("lstm_train_f32: h_f32", h_f32, (B, ndir * H, T))
    _shape("lstm_train_f32: gates", gates, (B, ndir * 4 * H, T))
    _shape("lstm_train_f32: cell", cell, (B, ndir * H, T))
    p = L.LstmParams()
    p.pre, p.w_hh, p.lengths = L.ptr(pre, f32, "pre"), L.ptr(w_hh, f32, "w_hh"), L.ptr(lengths, torch.int32, "lengths")
    p.pre_stride_b, p.pre_stride_t, p.pre_stride_r = R * T, 1, T
    p.h_f32 = L.ptr(h_f32, f32, "h_f32")
    p.hf_stride_b, p.hf_stride_t, p.hf_stride_c = ndir * H * T, 1, T
    p.B, p.T, p.H, p.ndir = B, T, H, ndir
    L.check(L.lib().svsk_lstm_train_f32(C.byref(p), L.ptr(gates, f32, "gates"), L.ptr(cell, f32, "cell"), L.stream_ptr()),
            "lstm_train_f32")


def lstm_bwd_f32(dh, gates, cell, w_hh, lengths, H, out=None):
    """svsk_lstm_bwd_f32: dL/dpre [B, ndir*4H, T] from dL/dh [B, ndir*H, T] and lstm_train_f32's gates / cell."""
    ndir = w_hh.shape[0]
    B, _, T = dh.shape
    _shape("lstm_bwd_f32: w_hh", w_hh, (ndir, 4 * H, H))
    _shape("lstm_bwd_f32: dh", dh, (B, ndir * H, T))
    _shape("lstm_bwd_f32: gates", gates, (B, ndir * 4 * H, T))
    _shape("lstm_bwd_f32: cell", cell, (B, ndir * H, T))
    if lengths is not None:
        _shape("lstm_bwd_f32: lengths", lengths, (B,))
    out = torch.empty((B, ndir * 4 * H, T), device=dh.device, dtype=f32) if out is None else out
    _shape("lstm_bwd_f32: out", out, (B, ndir * 4 * H, T))
    p = L.LstmBwdParams()
    p.dh, p.gates, p.cell = L.ptr(dh, f32, "dh"), L.ptr(gates, f32, "gates"), L.ptr(cell, f32, "cell")
    p.w_hh, p.lengths, p.dpre = L.ptr(w_hh, f32, "w_hh"), L.ptr(lengths, torch.int32, "lengths"), L.ptr(out, f32, "out")
    p.B, p.T, p.H, p.ndir = B, T, H, ndir
    L.check(L.lib().svsk_lstm_bwd_f32(C.byref(p), L.stream_ptr()), "lstm_bwd_f32")
    return out


def _frames_view(name, t):
    """Batch stride of a [B, C, T] fp32 CUDA tensor whose rows are T contiguous frames (a channel slice is fine)."""
    if t.dim() != 3 or t.stride(2) != 1 or t.stride(1) != t.shape[2]:
        raise ValueError(f"{name} must be [B, C, T] with rows of T contiguous frames, got shape {list(t.shape)} strides {t.stride()}")
    if not t.is_cuda or t.dtype != f32:
        raise RuntimeError(f"{name} must be a CUDA fp32 tensor: libsvsk has no CPU path")
    return t.stride(0)


def wgrad_f32_splits(B, T, N, ncols, target=2 * 148):
    """Frame splits of svsk_wgrad_f32: about two waves of CTAs on a B200, at least 4 chunks of 32 frames per split."""
    tiles = -(-N // 64) * -(-ncols // 64)
    return max(1, min(-(-target // tiles), (B * -(-T // 32)) // 4, 64))


def wgrad_f32(dy, x, *, ksize=1, origin=0, pad_mode=PAD_ZEROS, bias=True, dw=None):
    """svsk_wgrad_f32: dw [N, K, ksize] = sum_b sum_t dy[b, n, t] x[b, k, t + j - origin] (zero / reflect padded) and,
    with ``bias``, db [N] = sum dy.  dy [B, N, T], x [B, K, T] (channel slices of larger tensors allowed).  -> (dw, db)."""
    B, N, T = dy.shape
    if x.dim() != 3 or x.shape[0] != B or x.shape[2] != T:
        raise ValueError(f"wgrad_f32: x must be [{B}, K, {T}], got {list(x.shape)}")
    K = x.shape[1]
    dsb, xsb = _frames_view("wgrad_f32: dy", dy), _frames_view("wgrad_f32: x", x)
    dw = torch.empty((N, K, ksize), device=dy.device, dtype=f32) if dw is None else dw
    _shape("wgrad_f32: dw", dw, (N, K, ksize))
    db = torch.empty((N,), device=dy.device, dtype=f32) if bias else None
    ncols = K * ksize + int(bias)
    splits = wgrad_f32_splits(B, T, N, ncols)
    ws = torch.empty((splits, N, ncols), device=dy.device, dtype=f32) if splits > 1 else None
    p = L.WgradF32Params()
    p.dy, p.x = C.c_void_p(dy.data_ptr()), C.c_void_p(x.data_ptr())
    p.dw, p.db, p.ws = L.ptr(dw, f32, "dw"), L.ptr(db), L.ptr(ws)
    p.dy_batch_stride, p.x_batch_stride = dsb, xsb
    p.B, p.N, p.K, p.T, p.ksize, p.origin, p.pad_mode, p.splits = B, N, K, T, int(ksize), int(origin), int(pad_mode), splits
    L.check(L.lib().svsk_wgrad_f32(C.byref(p), L.stream_ptr()), "wgrad_f32")
    return dw, db


def bn_relu_bwd_f32(dy, y, x, mean, var, gamma, *, eps, out=None):
    """svsk_bn_relu_bwd_f32: BatchNorm1d (batch statistics) + ReLU backward on [B, C, T] -> (dx, dgamma, dbeta).
    y: the forward's ReLU output, x: the BatchNorm input, mean / var: its batch statistics; out may be dy."""
    B, Cc, T = dy.shape
    for name, t in (("y", y), ("x", x)):
        _shape(f"bn_relu_bwd_f32: {name}", t, (B, Cc, T))
    for name, t in (("mean", mean), ("var", var), ("gamma", gamma)):
        _shape(f"bn_relu_bwd_f32: {name}", t, (Cc,))
    out = torch.empty_like(dy) if out is None else out
    _shape("bn_relu_bwd_f32: out", out, (B, Cc, T))
    dgamma = torch.empty((Cc,), device=dy.device, dtype=f32)
    dbeta = torch.empty((Cc,), device=dy.device, dtype=f32)
    L.check(L.lib().svsk_bn_relu_bwd_f32(L.ptr(dy, f32, "dy"), L.ptr(y, f32, "y"), L.ptr(x, f32, "x"), L.ptr(mean, f32, "mean"),
                                         L.ptr(var, f32, "var"), L.ptr(gamma, f32, "gamma"), float(eps), L.ptr(out, f32, "out"),
                                         L.ptr(dgamma), L.ptr(dbeta), B, Cc, T, L.stream_ptr()), "bn_relu_bwd_f32")
    return out, dgamma, dbeta


def reflect_fold_f32(dx, dy, w):
    """svsk_reflect_fold_f32, in place on dx [B, Cin, T]: adds the ReflectionPad1d rows of the Conv1d w [Cout, Cin, k]
    (pad = (k - 1) / 2) whose output gradient is dy [B, Cout, T].  Returns dx."""
    B, Cin, T = dx.shape
    Cout, Cin_w, k = w.shape
    if Cin_w != Cin or k % 2 == 0:
        raise ValueError(f"reflect_fold_f32: w must be [Cout, {Cin}, odd k], got {list(w.shape)}")
    _shape("reflect_fold_f32: dy", dy, (B, Cout, T))
    L.check(L.lib().svsk_reflect_fold_f32(L.ptr(dx, f32, "dx"), L.ptr(dy, f32, "dy"), L.ptr(w, f32, "w"), B, Cin, Cout, T,
                                          (k - 1) // 2, L.stream_ptr()), "reflect_fold_f32")
    return dx


# ---- acoustic post-processing (include/svsk.h, "acoustic post-processing on the device") ----------------------------
def filtfilt_f32(x, b, a, zi, *, min_len, lengths=None, out=None):
    """svsk_filtfilt_f32.  x [B, T, D] fp32; b, a, zi: float64 sequences (host); lengths int32 [B] or None."""
    B, T, D = x.shape
    order = len(a) - 1
    pad = 3 * (order + 1)
    out = torch.empty_like(x) if out is None else out
    scratch = torch.empty((B, T + 2 * pad, D), device=x.device, dtype=torch.float64)
    arr = lambda v: (C.c_double * len(v))(*[float(t) for t in v])
    L.check(L.lib().svsk_filtfilt_f32(L.ptr(x, f32, "x"), L.ptr(out, f32, "out"), L.ptr(scratch), L.ptr(lengths, torch.int32, "lengths"),
                                      arr(b), arr(a), arr(zi), order, pad, int(min_len), B, T, D, L.stream_ptr()), "filtfilt_f32")
    return out


def variance_scaling_f32(x, gv, *, offset=2, note_mask=None, lengths=None, out=None):
    """svsk_variance_scaling_f32.  x [B, T, D] fp32, gv [D] fp32, note_mask uint8 [B, T] or None, lengths int32 [B] or None."""
    B, T, D = x.shape
    out = torch.empty_like(x) if out is None else out
    L.check(L.lib().svsk_variance_scaling_f32(L.ptr(x, f32, "x"), L.ptr(out, f32, "out"), L.ptr(gv, f32, "gv"),
                                              L.ptr(note_mask, torch.uint8, "note_mask"), L.ptr(lengths, torch.int32, "lengths"),
                                              int(offset), B, T, D, L.stream_ptr()), "variance_scaling_f32")
    return out


def scale_features_f32(x, a, b, mode, out=None):
    """svsk_scale_features_f32 over the last dimension of x (fp32, contiguous): mode 0 x*a+b, mode 1 (x-b)/a."""
    D = x.shape[-1]
    out = torch.empty_like(x) if out is None else out
    L.check(L.lib().svsk_scale_features_f32(L.ptr(x, f32, "x"), L.ptr(out, f32, "out"), L.ptr(a, f32, "a"), L.ptr(b, f32, "b"), int(mode),
                                            x.numel() // D, D, L.stream_ptr()), "scale_features_f32")
    return out


def mdn_head_f32(raw, G, D, *, want_params=True, want_best=False):
    """svsk_mdn_head_f32.  raw [B, T, ld] fp32 ([log_pi | log_sigma | mu] columns) -> (log_pi, log_sigma, mu) [B, T, G, D]
    and / or (best_sigma, best_mu) [B, T, D]."""
    B, T, ld = raw.shape
    mk = lambda *shape: torch.empty(shape, device=raw.device, dtype=f32)
    lp, ls, mu = (mk(B, T, G, D), mk(B, T, G, D), mk(B, T, G, D)) if want_params else (None, None, None)
    bs, bm = (mk(B, T, D), mk(B, T, D)) if want_best else (None, None)
    L.check(L.lib().svsk_mdn_head_f32(L.ptr(raw, f32, "raw"), L.ptr(lp), L.ptr(ls), L.ptr(mu), L.ptr(bs), L.ptr(bm), B * T, G, D, ld,
                                      L.stream_ptr()), "mdn_head_f32")
    return (lp, ls, mu), (bs, bm)
