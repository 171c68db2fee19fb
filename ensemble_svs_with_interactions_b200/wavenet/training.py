"""Training-time WaveNet forward AND backward on libsvsk kernels: ``WaveNet.forward`` under autograd
(nnsvs/wavenet/wavenet.py:60-87), trained through ``loss.backward()`` like the reference.

The whole network is ONE ``torch.autograd.Function`` over the parameters stacked over the layers (a differentiable
``torch.stack``, so every ``nn.Parameter`` still receives its own ``.grad``):

forward (_forward, which the inference path of WaveNet.forward runs too, so the output is the same bits)
    pack      = fold weight norm of every weight into the layouts below          svsk_wavenet_train_pack_f32, 1 launch
    x_0       = first_conv(x)                                                    svsk_conv1d_f32
    x_{l+1}, skips (+)=, y_l = block_l(x_l, c)                                   svsk_wavenet_block_train_f32, L launches
    h1 = last1(relu(skips));  logits = last3(relu(h1))                           svsk_conv1d_f32 x 2
backward (dlogits = upstream gradient)
    dh1 = last3^T dlogits . [h1 > 0];  dS = last1^T dh1 . [skips > 0]            svsk_conv1d_f32 + svsk_relu_mask_f32, x 2
    g_l = dL/dx_l and dy_{l-1} = dL/dy_{l-1}, last block first                   svsk_wavenet_dgrad_f32, L + 1 launches
    every weight / bias gradient                                                 svsk_wavenet_wgrad_f32, 1-2 launches
    weight norm: dg, dv from the effective weights' gradients                    svsk_wavenet_wnorm_grad_f32, 1 launch
    dc = [conv1x1c_0 .. conv1x1c_{L-1}]^T [dy_0 .. dy_{L-1}] (one 1x1 conv); dx = first_conv^T g_0, when asked for

Numerics: fp32 on the CUDA cores throughout, like the forward; no atomics, so gradients are bit-reproducible.
"""
from __future__ import annotations

import torch

from .. import ops

f32 = torch.float32
_CPU_ERROR = "WaveNet runs on CUDA (sm_100a) only: libsvsk has no CPU path"

# the weights as in svsk_wavenet_ar_weights: (name, how to get the conv holders from the network)
_GROUPS = (
    ("first", lambda n: [n.first_conv]),
    ("conv", lambda n: [f.conv for f in n.main_conv_layers]),
    ("cond", lambda n: [f.conv1x1c for f in n.main_conv_layers]),
    ("skip", lambda n: [f.conv1x1_skip for f in n.main_conv_layers]),
    ("out", lambda n: [f.conv1x1_out for f in n.main_conv_layers]),
    ("last1", lambda n: [n.last_conv_layers[1]]),
    ("last3", lambda n: [n.last_conv_layers[3]]),
)
_STACKED = {"conv", "cond", "skip", "out"}
_BIASED = ("first", "conv", "skip", "out", "last1", "last3")


def _stack(mods, attr, stacked):
    ts = [getattr(m, attr) for m in mods]
    if any(t is None for t in ts):
        return None
    t = torch.stack(ts) if stacked else ts[0]
    return t.to(f32).contiguous()


def _params(net):
    """[(key, tensor or None)] of the Function's parameter inputs: v, g (None without weight norm) of every weight, then
    the biases (conv_b None when a block's conv has no bias)."""
    out = []
    for name, mods in _GROUPS:
        ms = mods(net)
        st = name in _STACKED
        if hasattr(ms[0], "weight_g"):
            out += [(name + "_v", _stack(ms, "weight_v", st)), (name + "_g", _stack(ms, "weight_g", st))]
        else:
            out += [(name + "_v", _stack(ms, "weight", st)), (name + "_g", None)]
    for name, mods in _GROUPS:
        if name in _BIASED:
            out.append((name + "_b", _stack(mods(net), "bias", name in _STACKED)))
    return out


def _dims(net):
    """(sizes as the ops wrappers take them, dilation of every block)."""
    blocks = net.main_conv_layers
    f0 = blocks[0]
    if len({f.kernel_size for f in blocks}) != 1:
        raise RuntimeError("WaveNet on libsvsk: all blocks must share one kernel size")
    return (dict(out_dim=net.first_conv.in_channels, R=net.first_conv.out_channels, G=f0.conv.out_channels,
                 S=f0.conv1x1_skip.out_channels, cin=f0.conv1x1c.in_channels, layers=len(blocks), ksize=f0.kernel_size),
            tuple(int(f.dilation) for f in blocks))


def _pack(dims, w):
    """The weight pack of the forward (wavenet_train_layout's views) plus "b2", the blocks' [skip | out] biases."""
    pk = ops.wavenet_train_pack_f32({n: w[n] for n in w if not n.endswith("_b")}, **dims)
    return dict(pk, b2=torch.cat([w["skip_b"], w["out_b"]], dim=1))


def _forward(dims, dilations, pk, w, c, x, train):
    """Forward kernels after the pack: logits [B, out_dim, T] and what the backward keeps.  train: the blocks also store
    their gate pre-activations ys (svsk_wavenet_block_train_f32), else ys is None."""
    L, k = dims["layers"], dims["ksize"]
    B, _, T = x.shape
    R, G, S = dims["R"], dims["G"], dims["S"]
    xs = torch.empty((L + 1, B, R, T), device=x.device, dtype=f32)
    ops.conv1d_f32(x, pk["first"], w["first_b"], out=xs[0])
    skips = torch.empty((B, S, T), device=x.device, dtype=f32)
    ys = torch.empty((L, B, G, T), device=x.device, dtype=f32) if train else None
    for l in range(L):
        b1 = None if w["conv_b"] is None else w["conv_b"][l]
        blk = (xs[l], c, pk["w1t"][l], b1, pk["w2t"][l], pk["b2"][l], skips)
        kw = dict(ksize=k, dilation=dilations[l], first=(l == 0), out=xs[l + 1])
        if train:
            ops.wavenet_block_train_f32(*blk, ys[l], **kw)
        else:
            ops.wavenet_block_f32(*blk, **kw)
    h1 = ops.conv1d_f32(skips, pk["last1"], w["last1_b"], in_relu=True)
    logits = ops.conv1d_f32(h1, pk["last3"], w["last3_b"], in_relu=True)
    return logits, (pk, xs, ys, skips, h1)


def _backward(dims, dilations, dil_dev, c, x, w, saved, glog, need_c, need_x):
    """Backward kernels -> (dc [B, cin, T] or None, dx [B, out_dim, T] or None, {parameter key: gradient})."""
    pk, xs, ys, skips, h1 = saved
    L, k = dims["layers"], dims["ksize"]
    B, _, T = x.shape
    R, G, S = dims["R"], dims["G"], dims["S"]
    dh1 = ops.conv1d_f32(glog, pk["last3T"])
    ops.relu_mask_f32(dh1, h1, out=dh1)
    dS = ops.conv1d_f32(dh1, pk["last1T"])
    ops.relu_mask_f32(dS, skips, out=dS)
    gs = torch.empty((L + 1, B, R, T), device=x.device, dtype=f32)
    dy = torch.empty((B, L, G, T), device=x.device, dtype=f32)
    for l in range(L, -1, -1):
        ops.wavenet_dgrad_f32(dy_in=dy[:, l] if l < L else None, wT=pk["wT"][l] if l < L else None,
                              g_next=gs[l + 1] if l < L - 1 else None, g_out=gs[l], dS=dS,
                              y_prev=ys[l - 1] if l > 0 else None, wB=pk["wB"][l - 1] if l > 0 else None,
                              dy_out=dy[:, l - 1] if l > 0 else None, ksize=k, dilation=dilations[l] if l < L else 1)
    splits = ops.wavenet_wgrad_splits(B, T, **dims)
    dW = ops.wavenet_wgrad_f32(x_in=x, c=c, xs=xs[:L], ys=ys, gs=gs, dy=dy, dS=dS, skips=skips, h1=h1, dh1=dh1, glog=glog,
                               dilations=dil_dev, ksize=k, splits=splits)
    dg = ops.wavenet_wnorm_grad_f32({n: w[n] for n in w if not n.endswith("_b")}, dW, **dims)
    _, lay = ops.wavenet_train_layout(**dims)
    view = lambda name: dW[lay[name][0]:lay[name][0] + _numel(lay[name][1])].view(lay[name][1])
    grads = {}
    for name, _ in _GROUPS:
        grads[name + "_v"] = view(name).view(w[name + "_v"].shape)
        grads[name + "_g"] = dg.get(name)
    for name in _BIASED:
        grads[name + "_b"] = None if w[name + "_b"] is None else view(name + "_b").view(w[name + "_b"].shape)
    dc = ops.conv1d_f32(dy.view(B, L * G, T), pk["wcT"]) if need_c else None
    dx = ops.conv1d_f32(gs[0], pk["firstT"]) if need_x else None
    return dc, dx, grads


def _numel(shape):
    n = 1
    for s in shape:
        n *= s
    return n


class _WaveNetFn(torch.autograd.Function):
    """logits (B, T, out_dim) = WaveNet(c (B, T, cin), x (B, T, out_dim)) given the stacked parameters."""

    @staticmethod
    def forward(ctx, dims, dilations, keys, c, x, *params):
        w = dict(zip(keys, params))
        ct = c.to(f32).transpose(1, 2).contiguous()
        xt = x.to(f32).transpose(1, 2).contiguous()
        logits, saved = _forward(dims, dilations, _pack(dims, w), w, ct, xt, train=True)
        ctx.dims, ctx.dilations, ctx.keys = dims, dilations, keys
        ctx.c_dtype, ctx.x_dtype = c.dtype, x.dtype
        ctx.saved = saved               # kernel outputs only (not inputs / parameters): no version tracking needed
        ctx.save_for_backward(ct, xt, *params)
        return logits.transpose(1, 2)

    @staticmethod
    def backward(ctx, g):
        ct, xt, *params = ctx.saved_tensors
        w = dict(zip(ctx.keys, params))
        glog = g.to(f32).transpose(1, 2).contiguous()
        dil_dev = torch.tensor(ctx.dilations, dtype=torch.int32, device=glog.device)
        dc, dx, grads = _backward(ctx.dims, ctx.dilations, dil_dev, ct, xt, w, ctx.saved, glog, ctx.needs_input_grad[3],
                                  ctx.needs_input_grad[4])
        ctx.saved = None
        dc = None if dc is None else dc.transpose(1, 2).to(ctx.c_dtype)
        dx = None if dx is None else dx.transpose(1, 2).to(ctx.x_dtype)
        return (None, None, None, dc, dx) + tuple(grads[k] if p is not None else None for k, p in zip(ctx.keys, params))


def wavenet_forward_with_grad(net, c, x):
    """WaveNet.forward under autograd: logits (B, T, out_dim) with a grad_fn; the forward is bit-identical to the eval
    path's."""
    if not x.is_cuda or not c.is_cuda:
        raise RuntimeError(_CPU_ERROR)
    dims, dilations = _dims(net)
    items = _params(net)
    keys = tuple(k_ for k_, _ in items)
    return _WaveNetFn.apply(dims, dilations, keys, c, x, *[t for _, t in items])
