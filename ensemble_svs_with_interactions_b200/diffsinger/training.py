"""Training-time DiffNet forward AND backward on libsvsk kernels (SURVEY.md §8(f) row 4).

The reference trains the denoiser through autograd over ``DiffNet.forward`` (nnsvs/diffsinger/denoiser.py:101-124) inside
``train_step`` (nnsvs/bin/train_acoustic_multitrack.py:358-380).  Here the whole convolutional part — input projection,
the L gated residual blocks, skip / output projections — is ONE ``torch.autograd.Function`` whose forward and backward
are hand-written tcgen05 kernels (csrc/diffnet_train_sm100.cu):

forward, per block l  (NTC bf16 activations; kept for the backward: xd_l, ypre_l, z_l)
    ypre_l, z_l = GATE_FWD ( [xd_l(t-d) | xd_l(t) | xd_l(t+d) | cond(t)] . W1p_l + b1_l )        xd_l = x_l + dp_l
    x_{l+1}, xd_{l+1}, skip += RES_SKIP ( z_l . Woutp_l + bout_l )
backward, per block l  (u_l = dL/dx_l / sqrt 2, dS = dL/dskip: the same for every block)
    dy_l   = GATE_BWD ( [u_{l+1} | dS] . Wout_l )                  dz GEMM with the gate derivative fused
    u_l    = ADD_SCALE( [dy_l(t+d) | dy_l(t) | dy_l(t-d)] . W1_l^T + u_{l+1} ) / sqrt 2          dgrad (transposed conv)
    dW1_l  = dy_l^T . [xd_l(t-d) | xd_l(t) | xd_l(t+d) | cond]     wgrad: contraction over all frames, no atomics
    dWout_l = [u_{l+1} | dS]^T . z_l
    bias and step-embedding gradients = column sums of dy_l over time: indicator rows appended to the wgrad operand

Only the [B, C]-sized step-embedding MLP (sinusoid -> Linear -> Mish -> Linear -> per-layer Linear, 1e-5 of the FLOPs) stays
ordinary differentiable PyTorch: its output ``dp`` [L, B, C] is an input of the Function and receives its gradient from
it.  Parameters remain ordinary ``nn.Parameter``s (they enter the Function stacked over the layers, a differentiable
``torch.stack``), so DistributedDataParallel's hooks and the NCCL gradient all-reduce work as with the reference model
(nnsvs/train_util.py:1444-1446).

Numerics: bf16 GEMM operands and bf16 stored activations / gradients, fp32 accumulation, ``tanh.approx`` in the gate and
in its derivative — the backward differentiates exactly the function the forward computes (up to the bf16 rounding of
the stored tensors).  Models that resolve to precision "fp32" (C not in {128, 256}, H % 64 != 0, or forced) have no
tensor-core kernels at all: their forward stays libsvsk's fp32 path and their backward differentiates
``torch_restatement`` below (``_DiffNetFp32Fn``).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from .. import ops

BACKWARD_IMPL = "libsvsk tcgen05 kernels (seggemm dgrad / gate backward, wgrad)"

f32 = torch.float32
bf16 = torch.bfloat16


def _mish(x):
    return x * torch.tanh(F.softplus(x))


def _step_embedding(net, t):
    """mlp(SinusoidalPosEmb(t)) in differentiable PyTorch (denoiser.py:14-26, 84-86, 113-114) -> [B, C]."""
    C = net.residual_channels
    half = C // 2
    freq = torch.exp(torch.arange(half, device=t.device) * -(math.log(10000) / (half - 1)))
    arg = t.to(f32)[:, None] * freq[None, :]
    e = torch.cat((arg.sin(), arg.cos()), dim=-1)
    return F.linear(_mish(F.linear(e, net.mlp[0].weight, net.mlp[0].bias)), net.mlp[2].weight, net.mlp[2].bias)


def torch_restatement(net, spec, t, cond):
    """Differentiable fp32 re-statement of DiffNet.forward: the training path of precision="fp32" models, and the
    autograd reference of the gradient parity tests."""
    C = net.residual_channels
    x = F.relu(F.conv1d(spec[:, 0], net.input_projection.weight, net.input_projection.bias))
    e = _step_embedding(net, t)
    skip = 0
    for layer in net.residual_layers:
        dp = F.linear(e, layer.diffusion_projection.weight, layer.diffusion_projection.bias)[:, :, None]
        y = F.conv1d(x + dp, layer.dilated_conv.weight, layer.dilated_conv.bias, padding=layer.dilation,
                     dilation=layer.dilation)
        y = y + F.conv1d(cond, layer.conditioner_projection.weight, layer.conditioner_projection.bias)
        z = torch.sigmoid(y[:, :C]) * torch.tanh(y[:, C:])
        o = F.conv1d(z, layer.output_projection.weight, layer.output_projection.bias)
        x = (x + o[:, :C]) / math.sqrt(2.0)
        skip = skip + o[:, C:]
    x = skip / math.sqrt(len(net.residual_layers))
    x = F.relu(F.conv1d(x, net.skip_projection.weight, net.skip_projection.bias))
    x = F.conv1d(x, net.output_projection.weight, net.output_projection.bias)
    return x[:, None]


def _pad_cols(w, cols):
    """[R, K] -> [R, cols] bf16, zero padded."""
    out = torch.zeros((w.shape[0], cols), device=w.device, dtype=bf16)
    out[:, :w.shape[1]] = w
    return out


def _pad_rows(w, rows):
    out = torch.zeros((rows, w.shape[1]), device=w.device, dtype=bf16)
    out[:w.shape[0]] = w
    return out


_PERM = {}


def _perm(C, device):
    """perm[r] = packed row of reference row r of the 2C conv outputs (gate / filter rows of 128 channels side by side)."""
    key = (C, str(device))
    if key not in _PERM:
        _PERM[key] = ops.diffnet_packed_rows(C).to(device)
    return _PERM[key]


def _stack_forward(dilations, spec, cond, dp, Wd, bd, Wc, bc, Wo, bo, Win, bin_, Wsk, bsk, Wout, bout):
    """Forward kernels.  Returns (eps [B,1,M,T] fp32, saved tensors for _stack_backward, dims)."""
    B, _, M, T = spec.shape
    L, C2, C, _ = Wd.shape
    H = Wc.shape[2]
    dev = spec.device
    M64 = (M + 63) // 64 * 64
    M16 = (M + 15) // 16 * 16
    perm = _perm(C, dev)
    pk = ops.diffnet_train_pack(Wd.contiguous(), Wc.reshape(L, C2, H).contiguous(), Wo.reshape(L, C2, C).contiguous())
    b1p = torch.empty((L, C2), device=dev, dtype=f32)
    b1p[:, perm] = bd + bc
    bo = bo.contiguous()
    dp = dp.contiguous()
    specb, _ = ops.nct_to_ntc(spec[:, 0].to(f32).contiguous(), Cp=M64)
    condb, _ = ops.nct_to_ntc(cond.to(f32).contiguous())
    win_p = _pad_cols(Win[:, :, 0], M64)                                      # [C, M64]
    xd_all = torch.empty((L, B, T, C), device=dev, dtype=bf16)
    ypre_all = torch.empty((L, B, T, C2), device=dev, dtype=bf16)
    z_all = torch.empty((L, B, T, C), device=dev, dtype=bf16)
    x0 = torch.empty((B, T, C), device=dev, dtype=bf16)
    xa, xb = torch.empty_like(x0), torch.empty_like(x0)
    skip32 = torch.empty((B, T, C), device=dev, dtype=f32)
    # head: x0 = relu(Win spec + b);  xd_0 = x0 + dp_0
    ops.seggemm_bf16([(specb, M64, 0)], win_p, mode=ops.SEG_PLAIN, bias=bin_.contiguous(), act=ops.ACT_RELU, out0=x0,
                     out1=xd_all[0], dp_next=dp[0])
    cur = x0
    for l in range(L):
        d = int(dilations[l])
        xd = xd_all[l]
        ops.seggemm_bf16([(xd, C, -d), (xd, C, 0), (xd, C, d), (condb, H, 0)], pk["w1p"][l], mode=ops.SEG_GATE_FWD,
                         bias=b1p[l], out0=ypre_all[l], out1=z_all[l])
        last = l == L - 1
        nxt = xa if cur is not xa else xb
        ops.seggemm_bf16([(z_all[l], C, 0)], pk["woutp"][l], mode=ops.SEG_RES_SKIP, bias=bo[l], in0=cur,
                         out0=None if last else nxt, out1=None if last else xd_all[l + 1],
                         dp_next=None if last else dp[l + 1], outf=skip32, init=(l == 0))
        cur = nxt
    # tail: h = relu(Wskip S / sqrt L + b);  eps = Wout h + b
    Sb = ops.cast_scale_bf16(skip32, alpha=1.0 / math.sqrt(L))
    h = torch.empty((B, T, C), device=dev, dtype=bf16)
    ops.seggemm_bf16([(Sb, C, 0)], Wsk[:, :, 0].to(bf16).contiguous(), mode=ops.SEG_PLAIN, bias=bsk.contiguous(),
                     act=ops.ACT_RELU, out0=h)
    bout_p = torch.zeros((M16,), device=dev, dtype=f32)
    bout_p[:M] = bout
    eps32 = torch.empty((B, T, M16), device=dev, dtype=f32)
    ops.seggemm_bf16([(h, C, 0)], _pad_rows(Wout[:, :, 0].to(bf16), M16), mode=ops.SEG_PLAIN, bias=bout_p, outf=eps32)
    saved = (specb, condb, xd_all, ypre_all, z_all, x0, Sb, h, Wd, Wsk, Wout, Win, pk["woutT"], pk["w1T"], pk["wcT"])
    dims = (B, M, T, L, C, H, M64, M16)
    return ops.ntc_to_nct_f32(eps32, M)[:, None], saved, dims


_INDICATORS = {}


def _indicator_rows(B, T, Tp, d, device):
    """Rows appended to a wgrad operand so that column sums over time come out of the same GEMM (bf16 ones are exact, the
    accumulation is fp32).  d is None: [B, 16, Tp], row 0 = 1 on every frame of every track (-> sums over all tracks).
    d >= 0: [B, R, Tp], R = 3 B rounded up to 16; in track b only rows 3b, 3b+1, 3b+2 are non-zero: all frames, the
    first d frames, the last d frames (-> per-track sums, for the step-embedding gradient)."""
    key = (B, T, Tp, d, str(device))
    if key not in _INDICATORS:
        if d is None:
            ind = torch.zeros((B, 16, Tp), device=device, dtype=bf16)
            ind[:, 0, :T] = 1
        else:
            ind = torch.zeros((B, (3 * B + 15) // 16 * 16, Tp), device=device, dtype=bf16)
            for b in range(B):
                ind[b, 3 * b, :T] = 1
                ind[b, 3 * b + 1, :min(d, T)] = 1
                ind[b, 3 * b + 2, max(T - d, 0):T] = 1
        if len(_INDICATORS) > 64:
            _INDICATORS.clear()
        _INDICATORS[key] = ind
    return _INDICATORS[key]


def _stack_backward(saved, dims, dilations, d_eps, need_spec, need_cond):
    """Backward kernels.  Returns the gradients of (spec, cond, dp, Wd, bd, Wc, bc, Wo, bo, Win, bin, Wsk, bsk, Wout, bout)."""
    specb, condb, xd_all, ypre_all, z_all, x0, Sb, h, Wd, Wsk, Wout, Win, woutT, w1T, wcT = saved
    B, M, T, L, C, H, M64, M16 = dims
    C2 = 2 * C
    K1 = 3 * C + H
    dev = d_eps.device
    perm = _perm(C, dev)
    rs2 = 1.0 / math.sqrt(2.0)
    Tp = (T + 7) // 8 * 8
    ones = _indicator_rows(B, T, Tp, None, dev)                                   # [B, 16, Tp]
    ind = {d: _indicator_rows(B, T, Tp, d, dev) for d in set(dilations)}          # [B, R, Tp] per dilation
    R = next(iter(ind.values())).shape[1]
    # ---- tail
    deb, _ = ops.nct_to_ntc(d_eps[:, 0].to(f32).contiguous(), Cp=M64)            # [B, T, M64] bf16
    dh = torch.empty((B, T, C), device=dev, dtype=bf16)
    ops.seggemm_bf16([(deb, M64, 0)], _pad_cols(Wout[:, :, 0].t(), M64), mode=ops.SEG_PLAIN, mask=h, out0=dh)
    dS = torch.empty((B, T, C), device=dev, dtype=bf16)
    ops.seggemm_bf16([(dh, C, 0)], Wsk[:, :, 0].t().to(bf16).contiguous(), mode=ops.SEG_PLAIN, alpha=1.0 / math.sqrt(L), out0=dS)
    debT, hT, dhT, SbT = (ops.ntc_to_nct_bf16(t_) for t_ in (deb, h, dh, Sb))
    S1 = ops.wgrad_splits(B, ((C + 127) // 128) * ((C + 127) // 128 + 1))
    dWout = torch.empty((S1, M64, C + 16), device=dev, dtype=f32)                 # last 16 columns: [sum over frames, 0 ..]
    ops.wgrad_bf16(debT, [(hT, 0), (ones, 0)], dWout, T=T)
    dWsk = torch.empty((S1, C, C + 16), device=dev, dtype=f32)
    ops.wgrad_bf16(dhT, [(SbT, 0), (ones, 0)], dWsk, T=T)
    # ---- residual blocks, last to first
    Sa = ops.wgrad_splits(B, (C2 // 128) * ((3 * C + 127) // 128 + (H + 127) // 128 + (R + 127) // 128))
    Sb_ = ops.wgrad_splits(B, (C2 // 128) * ((C + 127) // 128 + 1))
    dW1 = torch.empty((L, Sa, C2, K1 + R), device=dev, dtype=f32)                 # packed rows; last R columns: sums of dy
    dWo = torch.empty((L, Sb_, C2, C + 16), device=dev, dtype=f32)                # column C: sums of [u_{l+1} ; dS]
    condT = ops.ntc_to_nct_bf16(condb)
    doT = torch.zeros((B, C2, Tp), device=dev, dtype=bf16)                        # [u_{l+1} ; dS] channel-major
    ops.ntc_to_nct_bf16(dS, out=doT, row0=C)
    xdT = torch.empty((B, 3 * C, Tp), device=dev, dtype=bf16)                     # xd_l(t - d) ; xd_l(t) ; xd_l(t + d)
    zT = torch.empty((B, C, Tp), device=dev, dtype=bf16)
    dyT = torch.empty((B, C2, Tp), device=dev, dtype=bf16)
    dy = torch.empty((B, T, C2), device=dev, dtype=bf16)
    ua = torch.zeros((B, T, C), device=dev, dtype=bf16)                          # u_L = 0: x after the last block is dead
    ub = torch.empty_like(ua)
    dcond32 = torch.empty((B, T, H), device=dev, dtype=f32) if need_cond else None
    u_next = ua
    for l in reversed(range(L)):
        d = dilations[l]
        ops.seggemm_bf16([(u_next, C, 0), (dS, C, 0)], woutT[l], mode=ops.SEG_GATE_BWD, in0=ypre_all[l], out0=dy)
        ops.ntc_to_nct_bf16(dy, out=dyT)
        # the tap shifts are written by the transpose (a TMA box must start 16-byte aligned along time)
        ops.ntc_to_nct_bf16(xd_all[l], out=xdT, shifts=(-d, 0, d))
        ops.ntc_to_nct_bf16(z_all[l], out=zT)
        ops.wgrad_bf16(dyT, [(xdT, 0), (condT, 0), (ind[d], 0)], dW1[l], T=T)
        ops.wgrad_bf16(doT, [(zT, 0), (ones, 0)], dWo[l], T=T)
        if need_cond:
            ops.seggemm_bf16([(dy, C2, 0)], wcT[l], mode=ops.SEG_PLAIN, outf=dcond32, accumulate=(l != L - 1))
        u = ub if u_next is ua else ua
        # transposed conv: tap j of the forward read x(t + s_j), s = (-d, 0, +d), so dx(t) gathers dy(t - s_j)
        ops.seggemm_bf16([(dy, C2, d), (dy, C2, 0), (dy, C2, -d)], w1T[l], mode=ops.SEG_ADD_SCALE, in0=u_next,
                         alpha=rs2 if l > 0 else 1.0, mask=None if l > 0 else x0, out0=u)
        u_next = u
        if l > 0:
            ops.ntc_to_nct_bf16(u_next, out=doT, row0=0)
    dpre0 = u_next                                                               # dL/d(pre-activation of the head) [B, T, C]
    # ---- head
    dWin = torch.empty((S1, C, M64 + 16), device=dev, dtype=f32)
    ops.wgrad_bf16(ops.ntc_to_nct_bf16(dpre0), [(ops.ntc_to_nct_bf16(specb), 0), (ones, 0)], dWin, T=T)
    g_spec = None
    if need_spec:
        dsp = torch.empty((B, T, M16), device=dev, dtype=f32)
        ops.seggemm_bf16([(dpre0, C, 0)], _pad_rows(Win[:, :, 0].t().to(bf16), M16), mode=ops.SEG_PLAIN, outf=dsp)
        g_spec = ops.ntc_to_nct_f32(dsp, M)[:, None]
    g_cond = ops.ntc_to_nct_f32(dcond32, H) if need_cond else None
    # ---- sum the track groups' partial results and unpack (a handful of batched tensor ops over all layers)
    dW1r = dW1.sum(1)[:, perm]                                                   # [L, 2C (reference rows), K1 + R]
    dWo_s, dWout_s, dWsk_s, dWin_s = dWo.sum(1), dWout.sum(0), dWsk.sum(0), dWin.sum(0)
    gWd = dW1r[:, :, :3 * C].reshape(L, C2, 3, C).permute(0, 1, 3, 2).contiguous()
    gWc = dW1r[:, :, 3 * C:K1].reshape(L, C2, H, 1).contiguous()
    csr = dW1r[:, :, K1:K1 + 3 * B].reshape(L, C2, B, 3).permute(0, 2, 3, 1)      # [L, B, 3, 2C]: all / first d / last d frames
    gb1 = csr[:, :, 0].sum(1)
    gbo = dWo_s[:, :, C].contiguous()
    # step projection: dp_l enters the conv through every tap that exists at a frame (zero padding comes after the add)
    taps = torch.stack([csr[:, :, 0] - csr[:, :, 1], csr[:, :, 0], csr[:, :, 0] - csr[:, :, 2]], dim=2)   # [L, B, 3, 2C]
    g_dp = torch.einsum("lbjr,lrcj->lbc", taps, Wd)
    return (g_spec, g_cond, g_dp, gWd, gb1, gWc, gb1, dWo_s[:, :, :C].reshape(L, C2, C, 1).contiguous(), gbo,
            dWin_s[:, :M, None].contiguous(), dWin_s[:, M64].contiguous(), dWsk_s[:, :C, None].contiguous(), dWsk_s[:, C].contiguous(),
            dWout_s[:M, :C, None].contiguous(), dWout_s[:M, C].contiguous())


class _GraphedStack:
    """CUDA graphs of _stack_forward / _stack_backward for one shape: static input buffers, two captured graphs (the
    ~45 + ~260 launches of a training step's stack become two replays; the step is launch-bound otherwise: 10.1 ms of
    host time against ~2 ms of kernels at 6 x 1000 frames)."""

    def __init__(self, dilations, tensors, need_spec, need_cond):
        self.dilations, self.need_spec, self.need_cond = dilations, need_spec, need_cond
        self.s_in = [torch.empty_like(t_, memory_format=torch.contiguous_format) for t_ in tensors]
        for s_, t_ in zip(self.s_in, tensors):
            s_.copy_(t_)
        self.pending = False            # a forward whose backward has not run yet owns the saved activations
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):   # warm-up outside capture (function attributes, tensor-map cache, allocator)
            eps, saved, dims = _stack_forward(dilations, *self.s_in)
            self.s_deps = torch.zeros_like(eps)
            _stack_backward(saved, dims, dilations, self.s_deps, need_spec, need_cond)
        torch.cuda.current_stream().wait_stream(side)
        n0 = _launch_count()
        self.g_fwd = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_fwd):
            self.eps, self.saved, self.dims = _stack_forward(dilations, *self.s_in)
        self.n_fwd = _launch_count() - n0
        self.g_bwd = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_bwd, pool=self.g_fwd.pool()):
            self.grads = _stack_backward(self.saved, self.dims, dilations, self.s_deps, need_spec, need_cond)
        self.n_bwd = _launch_count() - n0 - self.n_fwd
        _set_launch_count(n0)           # capture enqueues nothing; replays are counted when they happen

    def forward(self, tensors):
        for s_, t_ in zip(self.s_in, tensors):
            s_.copy_(t_)
        self.g_fwd.replay()
        _set_launch_count(_launch_count() + self.n_fwd)
        self.pending = True
        return self.eps.clone()

    def backward(self, d_eps):
        self.s_deps.copy_(d_eps)
        self.g_bwd.replay()
        _set_launch_count(_launch_count() + self.n_bwd)
        self.pending = False
        # clones: autograd may keep the returned tensors as .grad, and the next replay rewrites the static buffers
        return tuple(None if g is None else g.clone() for g in self.grads)


def _launch_count():
    from .. import _lib
    return _lib.launch_count


def _set_launch_count(v):
    from .. import _lib
    _lib.launch_count = v


_GRAPHS = {}          # shape key -> _GraphedStack (at most _MAX_GRAPHS, least recently used first out)
_SEEN = {}            # shape key -> times seen (a graph is captured the second time a shape comes by)
_MAX_GRAPHS = 2


def _graph_for(key, dilations, tensors, need_spec, need_cond):
    if torch.cuda.is_current_stream_capturing():
        return None
    g = _GRAPHS.get(key)
    if g is not None:
        _GRAPHS[key] = _GRAPHS.pop(key)      # most recently used last
        return None if g.pending else g
    _SEEN[key] = _SEEN.get(key, 0) + 1
    if len(_SEEN) > 64:
        _SEEN.clear()
    if _SEEN[key] < 2:
        return None
    while len(_GRAPHS) >= _MAX_GRAPHS:
        old = next(iter(_GRAPHS))
        if _GRAPHS[old].pending:
            return None
        del _GRAPHS[old]
    g = _GRAPHS[key] = _GraphedStack(dilations, tensors, need_spec, need_cond)
    return g


class _DiffNetStackFn(torch.autograd.Function):
    """eps = DiffNet(spec, cond) given the per-layer step projections dp [L, B, C] and the parameters stacked over the layers."""

    @staticmethod
    def forward(ctx, dilations, spec, cond, dp, *params):
        tensors = (spec, cond, dp) + params
        need_spec, need_cond = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        key = (dilations, need_spec, need_cond) + tuple((tuple(t_.shape), t_.dtype) for t_ in tensors) + (str(spec.device),)
        ctx.dilations = dilations
        ctx.graph = _graph_for(key, dilations, tensors, need_spec, need_cond)
        if ctx.graph is not None:
            return ctx.graph.forward(tensors)
        eps, saved, ctx.dims = _stack_forward(dilations, *tensors)
        ctx.save_for_backward(*saved)
        return eps

    @staticmethod
    def backward(ctx, d_eps):
        if ctx.graph is not None:
            return (None,) + ctx.graph.backward(d_eps)
        return (None,) + _stack_backward(ctx.saved_tensors, ctx.dims, ctx.dilations, d_eps, ctx.needs_input_grad[1],
                                         ctx.needs_input_grad[2])


class _DiffNetFp32Fn(torch.autograd.Function):
    """precision="fp32" models (widths the tensor-core kernels do not cover, or forced): the forward is libsvsk's exact
    fp32 path like every other call; the backward differentiates the PyTorch re-statement.  Not the training path of any
    recipe (C = 256 / 128 resolve to bf16) — it keeps small / odd models trainable."""

    @staticmethod
    def forward(ctx, net, spec, t, cond, *params):
        ctx.net = net
        ctx.save_for_backward(spec, t, cond)
        with torch.no_grad():
            return net._forward_no_grad(spec, t, cond)

    @staticmethod
    def backward(ctx, grad_out):
        net = ctx.net
        spec, t, cond = ctx.saved_tensors
        params = list(net.parameters())
        with torch.enable_grad():
            spec_ = spec.detach().requires_grad_(ctx.needs_input_grad[1])
            cond_ = cond.detach().requires_grad_(ctx.needs_input_grad[3])
            out = torch_restatement(net, spec_, t, cond_)
            wanted = [x for x in (spec_, cond_) if x.requires_grad] + [p for p in params if p.requires_grad]
            grads = list(torch.autograd.grad(out, wanted, grad_out.to(out.dtype), allow_unused=True))
        g_spec = grads.pop(0) if spec_.requires_grad else None
        g_cond = grads.pop(0) if cond_.requires_grad else None
        g_params = [grads.pop(0) if p.requires_grad else None for p in params]
        return (None, g_spec, None, g_cond, *g_params)


def diffnet_forward_with_grad(net, spec, diffusion_step, cond):
    """DiffNet.forward under autograd.  bf16 models: forward and backward are the kernel Function above."""
    t = diffusion_step.reshape(-1).to(torch.int64)
    if net.resolved_precision() != "bf16":
        return _DiffNetFp32Fn.apply(net, spec, t, cond, *net.parameters())
    layers = net.residual_layers
    e = _step_embedding(net, t)                                                          # [B, C]
    Wdp = torch.stack([ly.diffusion_projection.weight for ly in layers])                 # [L, C, C]
    bdp = torch.stack([ly.diffusion_projection.bias for ly in layers])
    dp = torch.einsum("bk,lck->lbc", e, Wdp) + bdp[:, None]
    st = lambda name, attr: torch.stack([getattr(getattr(ly, name), attr) for ly in layers])
    return _DiffNetStackFn.apply(
        tuple(int(ly.dilation) for ly in layers), spec, cond, dp,
        st("dilated_conv", "weight"), st("dilated_conv", "bias"), st("conditioner_projection", "weight"),
        st("conditioner_projection", "bias"), st("output_projection", "weight"), st("output_projection", "bias"),
        net.input_projection.weight, net.input_projection.bias, net.skip_projection.weight, net.skip_projection.bias,
        net.output_projection.weight, net.output_projection.bias)
