"""DiffNet denoiser — drop-in for ``nnsvs.diffsinger.denoiser.DiffNet`` (nnsvs/diffsinger/denoiser.py:69-124).

Same constructor kwargs, ``forward(spec, diffusion_step, cond)`` signature and ``state_dict`` keys/shapes.  The
``nn.Conv1d`` / ``nn.Linear`` sub-modules only HOLD the parameters (so checkpoints load with strict=True); the
arithmetic runs in libsvsk:

* ``precision="bf16"``: all residual layers of a call in one tcgen05 launch (svsk_diffnet_stack_bf16; one launch per
  layer, svsk_diffnet_block3_bf16, for tracks too long for it) + tcgen05 1x1 projections (svsk_linear_bf16); bf16
  residual stream and MMA operands, fp32 accumulation and skip sum.
* ``precision="fp32"``: CUDA-core kernels in the reference's own fp32 arithmetic (svsk_conv1d_f32 ...).
* ``precision="auto"`` (default): bf16 when the shapes fit the tensor-core kernels (C in {128,256}, H % 64 == 0,
  dilations <= 8, i.e. dilation_cycle_length <= 4 as in every recipe), else fp32.  Both are CUDA kernels of this library; there is no PyTorch/CPU path for the forward pass.
"""
from __future__ import annotations

import math
from math import sqrt

import os

import torch
import torch.nn as nn

from .. import ops

f32 = torch.float32
bf16 = torch.bfloat16


def _ceil_to(v, m):
    return (v + m - 1) // m * m


class Mish(nn.Module):
    """Parameter-free placeholder keeping ``mlp`` indices (mlp.0 / mlp.2) identical to denoiser.py:84-86.
    The activation itself runs inside svsk_conv1d_f32 (SVSK_ACT_MISH)."""

    def forward(self, x):  # pragma: no cover - never on the product path
        raise RuntimeError("Mish is evaluated inside libsvsk; call DiffNet.forward")


class SinusoidalPosEmb(nn.Module):
    """denoiser.py:14-26, evaluated by svsk_sinusoidal_embedding_f32."""

    def __init__(self, dim):
        super().__init__()
        self.dim = dim

    def forward(self, x):
        return ops.sinusoidal_embedding_f32(x, self.dim)


def Conv1d(*args, **kwargs):
    """Parameter holder with the reference's kaiming-normal init (denoiser.py:29-32)."""
    layer = nn.Conv1d(*args, **kwargs)
    nn.init.kaiming_normal_(layer.weight)
    return layer


class ResidualBlock(nn.Module):
    """Parameter holder for one gated block (denoiser.py:40-52); computed by DiffNet's engine."""

    def __init__(self, encoder_hidden, residual_channels, dilation):
        super().__init__()
        self.dilation = dilation
        self.dilated_conv = Conv1d(residual_channels, 2 * residual_channels, 3, padding=dilation, dilation=dilation)
        self.diffusion_projection = nn.Linear(residual_channels, residual_channels)
        self.conditioner_projection = Conv1d(encoder_hidden, 2 * residual_channels, 1)
        self.output_projection = Conv1d(residual_channels, 2 * residual_channels, 1)

    def forward(self, x, conditioner, diffusion_step):
        """Stand-alone block call in fp32 (same maths as denoiser.py:54-66)."""
        dp = ops.linear_f32(diffusion_step.contiguous(), self.diffusion_projection.weight, self.diffusion_projection.bias)
        return _block_fp32(self, x.contiguous(), conditioner.contiguous(), dp)


def _block_fp32(layer: ResidualBlock, x, cond, dp, skip=None, init_skip=True):
    y = ops.conv1d_f32(x, layer.dilated_conv.weight, layer.dilated_conv.bias, dilation=layer.dilation, tap_origin=1,
                       pad_mode=ops.PAD_ZEROS, in_bias=dp)
    ops.conv1d_f32(cond, layer.conditioner_projection.weight, layer.conditioner_projection.bias, out=y, accumulate=True)
    z = ops.gated_act_f32(y, ops.GATE_SIGMOID_TANH)
    o = ops.conv1d_f32(z, layer.output_projection.weight, layer.output_projection.bias)
    if skip is None:
        C = x.shape[1]
        x_new = x.clone()
        skip = torch.empty_like(x)
        ops.diffnet_residual_skip_f32(o, x_new, skip, True)
        return x_new, skip
    ops.diffnet_residual_skip_f32(o, x, skip, init_skip)
    return x, skip


_STACK_FIT_CACHE = {}
_PCOND_BUDGET_BYTES = 16 << 30   # buffers of the precomputed conditioner projection (cond_projection_bf16)


def _stack_tracks_per_launch(B, T, C, H):
    """Largest number of tracks whose CTA pairs all fit the device at once (0 if not even one track does)."""
    key = (B, T, C, H)
    if key not in _STACK_FIT_CACHE:
        b = B
        while b > 0 and not ops.diffnet_stack_fits(b, T, C, H):
            b -= 1
        if len(_STACK_FIT_CACHE) > 256:
            _STACK_FIT_CACHE.clear()
        _STACK_FIT_CACHE[key] = b
    return _STACK_FIT_CACHE[key]


class _Bf16Plan:
    """Packed weights of one DiffNet for the tensor-core path (rebuilt when any parameter changes)."""

    def __init__(self, net: "DiffNet", device):
        C, H, M, L = net.residual_channels, net.encoder_hidden_dim, net.in_dim, len(net.residual_layers)
        self.C, self.H, self.M, self.L = C, H, M, L
        self.Mp = _ceil_to(M, 16)
        with torch.no_grad():
            perm = ops.diffnet_packed_rows(C).to(device)  # reference row -> packed row
            w_in = torch.zeros((C, self.Mp), device=device, dtype=f32)
            w_in[:, :M] = net.input_projection.weight[:, :, 0]
            self.w_in = w_in.to(bf16).contiguous()
            self.b_in = net.input_projection.bias.detach().to(f32).contiguous()
            self.w_skip = net.skip_projection.weight[:, :, 0].to(bf16).contiguous()
            self.b_skip = net.skip_projection.bias.detach().to(f32).contiguous()
            w_out = torch.zeros((self.Mp, C), device=device, dtype=f32)
            w_out[:M] = net.output_projection.weight[:, :, 0]
            self.w_out = w_out.to(bf16).contiguous()
            b_out = torch.zeros((self.Mp,), device=device, dtype=f32)
            b_out[:M] = net.output_projection.bias
            self.b_out = b_out
            # per-layer operands live in tensors stacked along a leading layer dimension (what the one-launch stack
            # kernel reads); the per-layer entries below are views of them
            K1 = 3 * C + H
            self.w1p_all = torch.empty((L, 2 * C, K1), device=device, dtype=bf16)
            self.woutp_all = torch.empty((L, 2 * C, C), device=device, dtype=bf16)
            self.bout_all = torch.empty((L, 2 * C), device=device, dtype=f32)
            self.wcp_all = None  # [L * 2C/256, 256, H]: conditioner columns of w1p_all per 256-row output block (below)
            self.dilations = [int(layer.dilation) for layer in net.residual_layers]
            self.layers = []
            for i, layer in enumerate(net.residual_layers):
                dw = layer.dilated_conv.weight.detach().to(f32)
                cw = layer.conditioner_projection.weight.detach().to(f32)
                ow = layer.output_projection.weight.detach().to(f32)
                w1p, woutp = ops.diffnet_pack_block(dw, cw, ow)
                self.w1p_all[i].copy_(w1p)
                self.woutp_all[i].copy_(woutp)
                self.bout_all[i].copy_(layer.output_projection.bias.detach().to(f32))
                # step-embedding taps: stepw[j*2C + perm[r]] = dilated_w[r, :, j]  (so that stepbias = stepw @ dp + stepb
                # gives, per tap j, W_j . (diffusion_projection(e)) in packed row order); the conv and conditioner
                # biases ride on the centre tap, which every frame has.
                stepw = torch.zeros((3 * 2 * C, C), device=device, dtype=f32)
                stepb = torch.zeros((3 * 2 * C,), device=device, dtype=f32)
                for j in range(3):
                    stepw[j * 2 * C + perm] = dw[:, :, j]
                stepb[2 * C + perm] = layer.dilated_conv.bias.detach().to(f32) + layer.conditioner_projection.bias.detach().to(f32)
                self.layers.append(dict(
                    w1p=self.w1p_all[i], woutp=self.woutp_all[i], dilation=layer.dilation, bout=self.bout_all[i],
                    stepw=stepw.unsqueeze(-1).contiguous(), stepb=stepb,
                    dpw=layer.diffusion_projection.weight.detach().to(f32).contiguous(),
                    dpb=layer.diffusion_projection.bias.detach().to(f32).contiguous()))
            self.wcp_all = self.w1p_all[:, :, 3 * C:].reshape(L * (2 * C // 256), 256, H).contiguous()
        self.step_table = None  # [L, K, 3*2C], filled by GaussianDiffusion for t = 0..K-1


class DiffNet(nn.Module):
    def __init__(self, in_dim=80, encoder_hidden_dim=256, residual_layers=20, residual_channels=256,
                 dilation_cycle_length=4, precision="auto"):
        super().__init__()
        self.in_dim = in_dim
        self.encoder_hidden_dim = encoder_hidden_dim
        self.residual_channels = residual_channels
        self.precision = precision

        self.input_projection = Conv1d(in_dim, residual_channels, 1)
        self.diffusion_embedding = SinusoidalPosEmb(residual_channels)
        dim = residual_channels
        self.mlp = nn.Sequential(nn.Linear(dim, dim * 4), Mish(), nn.Linear(dim * 4, dim))
        self.residual_layers = nn.ModuleList(
            [ResidualBlock(encoder_hidden_dim, residual_channels, 2 ** (i % dilation_cycle_length))
             for i in range(residual_layers)])
        self.skip_projection = Conv1d(residual_channels, residual_channels, 1)
        self.output_projection = Conv1d(residual_channels, in_dim, 1)
        nn.init.zeros_(self.output_projection.weight)
        self._plan = None
        self._plan_key = None

    # ------------------------------------------------------------------ precision / plans
    def resolved_precision(self) -> str:
        max_dil = max((int(layer.dilation) for layer in self.residual_layers), default=1)
        ok = self.residual_channels in (128, 256) and self.encoder_hidden_dim % 64 == 0 and max_dil <= 8
        if self.precision == "auto":
            return "bf16" if ok else "fp32"
        if self.precision == "bf16" and not ok:
            raise RuntimeError("DiffNet precision='bf16' needs residual_channels in {128,256}, encoder_hidden_dim % 64 == 0 "
                               f"and dilations <= 8 (got {self.residual_channels}, {self.encoder_hidden_dim}, {max_dil}); "
                               "precision='fp32' / 'auto' run such shapes on the fp32 kernels")
        if self.precision not in ("bf16", "fp32"):
            raise RuntimeError(f"unknown precision {self.precision!r}")
        return self.precision

    def _param_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def bf16_plan(self) -> _Bf16Plan:
        key = self._param_key()
        if self._plan is None or self._plan_key != key:
            self._plan = _Bf16Plan(self, self.input_projection.weight.device)
            self._plan_key = key
        return self._plan

    # ------------------------------------------------------------------ step embedding (denoiser.py:113-114)
    def step_embedding(self, t):
        """mlp(SinusoidalPosEmb(t)) -> (Bt, C) fp32, all in libsvsk."""
        emb = self.diffusion_embedding(t)
        h = ops.linear_f32(emb, self.mlp[0].weight, self.mlp[0].bias, act=ops.ACT_MISH)
        return ops.linear_f32(h, self.mlp[2].weight, self.mlp[2].bias)

    def step_bias_bf16(self, t):
        """[L, Bt, 3*2C] tap biases for the fused kernels (packed row order), layer-major."""
        plan = self.bf16_plan()
        e = self.step_embedding(t)
        out = torch.empty((plan.L, e.shape[0], 6 * plan.C), device=e.device, dtype=f32)
        for i, lw in enumerate(plan.layers):
            dp = ops.linear_f32(e, lw["dpw"], lw["dpb"])
            ops.linear_f32(dp, lw["stepw"], lw["stepb"], out=out[i])
        return out

    # ------------------------------------------------------------------ engines
    def project_in_bf16(self, x32s, plan=None, out=None):
        """relu(input_projection(x)) (denoiser.py:109-112) as bf16 [B,T,C], from the fp32 NTC state [B,T,Mp]."""
        plan = self.bf16_plan() if plan is None else plan
        B, T, _ = x32s.shape
        xb0 = torch.empty((B, T, plan.C), device=x32s.device, dtype=bf16) if out is None else out
        ops.linear_bf16(ops.cast_scale_bf16(x32s), plan.w_in, plan.b_in, act=ops.ACT_RELU, out_bf16=xb0)
        return xb0

    def cond_projection_bf16(self, condb, plan=None):
        """conditioner_projection(cond) of ALL layers (denoiser.py:59) for a run of denoiser calls on the same cond
        (the K steps of diffusion.py:302-336): computed once, handed to every residual_stack_bf16 call of the run as
        ``pcond``.  Returns None when the stack kernel that would run this shape projects inside its GEMM."""
        plan = self.bf16_plan() if plan is None else plan
        B, T, H = condb.shape
        stack_b = _stack_tracks_per_launch(B, T, plan.C, H) if os.environ.get("SVSK_DIFFNET_STACK", "1") != "0" else 0
        if not stack_b or not ops.diffnet_stack_uses_pcond(stack_b, T, plan.C, H):
            return None
        # three buffers of B * T * L * 2C bf16 each (GEMM output, gate half + filter half): 0.74 GB at BASELINE config 2,
        # 2.2 GB for a 6 x 6000 batch; a batch for which they would not be small next to the model's own tensors keeps the
        # projection inside the GEMM (_PCOND_BUDGET_BYTES, 16 GB)
        tiles = 2 * ((T + 255) // 256)
        need = 2 * B * plan.L * 2 * plan.C * (2 * T + tiles * 128)
        if need > _PCOND_BUDGET_BYTES:
            return None
        p = ops.diffnet_cond_project(condb.contiguous(), plan.wcp_all)
        return ops.diffnet_pcond_pack(p, B, T, plan.L, plan.C)

    def residual_stack_bf16(self, xb0, condb, stepbias, plan=None, pcond=None):
        """The L residual blocks (denoiser.py:114-118) on xb0 [B,T,C] bf16 (clobbered); returns the fp32 sum of the skip
        outputs [B,T,C].  stepbias [L, Bt, 3*2C] fp32 (any layer stride; Bt = B rows, or 1 row shared by the batch).
        pcond: result of cond_projection_bf16(condb) for a run of calls on the same conditioner."""
        plan = self.bf16_plan() if plan is None else plan
        B, T, C = xb0.shape
        L = plan.L
        dev = xb0.device
        if stepbias.dim() != 3 or stepbias.shape[0] != L or stepbias.shape[1] not in (1, B) or stepbias.stride(2) != 1:
            raise ValueError(f"stepbias must be [L={L}, 1 or B={B}, {6 * C}], got {tuple(stepbias.shape)}")
        sb_layer = stepbias.stride(0)
        per_row = stepbias.shape[1] == B and B > 1
        sb_batch = stepbias.stride(1) if per_row else 0
        xb1 = torch.empty((B, T, C), device=dev, dtype=bf16)
        skip32 = torch.empty((B, T, C), device=dev, dtype=f32)
        stack_b = 0  # tracks per launch of the one-launch residual stack (0: run the layers one kernel at a time)
        if os.environ.get("SVSK_DIFFNET_STACK", "1") != "0":
            stack_b = _stack_tracks_per_launch(B, T, C, plan.H)
        if stack_b:
            # one launch for all L blocks of `stack_b` tracks: every CTA pair keeps its 256-frame tile across the layers,
            # neighbouring tiles exchange 8 edge rows per layer.  All pairs of a launch must be resident at once, so a
            # batch that exceeds one wave (e.g. 6 x 6000 frames) is split into groups of tracks.
            xb2 = torch.empty((B, T, C), device=dev, dtype=bf16)
            flags = torch.empty((B * 2 * ((T + 255) // 256),), device=dev, dtype=torch.int32)
            for b0 in range(0, B, stack_b):
                b1 = min(B, b0 + stack_b)
                ops.diffnet_stack_bf16(xb0[b0:b1], xb1[b0:b1], xb2[b0:b1], skip32[b0:b1], condb[b0:b1], plan.w1p_all,
                                       plan.woutp_all, stepbias[:, b0:b1] if per_row else stepbias, plan.bout_all, flags,
                                       plan.dilations, stepbias_batch_stride=sb_batch, stepbias_layer_stride=sb_layer,
                                       pcond=None if pcond is None else (pcond[0][b0:b1], pcond[1][b0:b1]))
        else:
            cur, nxt = xb0, xb1
            for i, lw in enumerate(plan.layers):
                ops.diffnet_block_bf16(cur, nxt, skip32, skip32, condb, lw["w1p"], lw["woutp"], stepbias[i], lw["bout"],
                                       dilation=lw["dilation"], stepbias_batch_stride=sb_batch, init_skip=(i == 0),
                                       write_x=(i < L - 1))
                cur, nxt = nxt, cur
        return skip32

    def denoise_ntc_bf16(self, x32s, condb, stepbias, plan=None):
        """x32s [B,T,Mp] fp32 (channels >= M are ignored), condb [B,T,H] bf16, stepbias as in residual_stack_bf16.
        Returns eps [B,T,Mp] fp32 (padded channels = 0)."""
        plan = self.bf16_plan() if plan is None else plan
        skip32 = self.residual_stack_bf16(self.project_in_bf16(x32s, plan), condb, stepbias, plan)
        skipb = ops.cast_scale_bf16(skip32, alpha=1.0 / sqrt(plan.L))
        hb, _ = ops.linear_bf16(skipb, plan.w_skip, plan.b_skip, act=ops.ACT_RELU, want_bf16=True)
        _, eps = ops.linear_bf16(hb, plan.w_out, plan.b_out, want_f32=True)
        return eps

    def denoise_nct_fp32(self, x_in, cond, t):
        """x_in [B,M,T], cond [B,H,T], t [B] -> eps [B,M,T]; the reference's fp32 arithmetic."""
        L = len(self.residual_layers)
        x = ops.conv1d_f32(x_in, self.input_projection.weight, self.input_projection.bias, act=ops.ACT_RELU)
        e = self.step_embedding(t)
        skip = torch.empty_like(x)
        for i, layer in enumerate(self.residual_layers):
            dp = ops.linear_f32(e, layer.diffusion_projection.weight, layer.diffusion_projection.bias)
            _block_fp32(layer, x, cond, dp, skip, init_skip=(i == 0))
        s = ops.scale_act_f32(skip, alpha=1.0 / sqrt(L))
        h = ops.conv1d_f32(s, self.skip_projection.weight, self.skip_projection.bias, act=ops.ACT_RELU)
        return ops.conv1d_f32(h, self.output_projection.weight, self.output_projection.bias)

    def _forward_no_grad(self, spec, diffusion_step, cond):
        x_in = spec[:, 0].to(f32).contiguous()
        cond = cond.to(f32).contiguous()
        t = diffusion_step.reshape(-1).to(torch.int64).contiguous()
        if self.resolved_precision() == "fp32":
            return self.denoise_nct_fp32(x_in, cond, t)[:, None]
        plan = self.bf16_plan()
        _, x32s = ops.nct_to_ntc(x_in, Cp=plan.Mp, want_bf16=False, want_f32=True)
        condb, _ = ops.nct_to_ntc(cond)
        sb = self.step_bias_bf16(t)
        eps = self.denoise_ntc_bf16(x32s, condb, sb)
        return ops.ntc_to_nct_f32(eps, plan.M)[:, None]

    def forward(self, spec, diffusion_step, cond):
        """
        :param spec: [B, 1, M, T]
        :param diffusion_step: [B] (int64 step indices)
        :param cond: [B, H, T]
        :return: [B, 1, M, T]
        """
        if not spec.is_cuda:
            raise RuntimeError("DiffNet runs on CUDA (sm_100a) only: libsvsk has no CPU path")
        needs_grad = torch.is_grad_enabled() and (
            spec.requires_grad or cond.requires_grad or any(p.requires_grad for p in self.parameters()))
        if needs_grad:
            from .training import diffnet_forward_with_grad
            return diffnet_forward_with_grad(self, spec, diffusion_step, cond)
        with torch.no_grad():
            return self._forward_no_grad(spec, diffusion_step, cond)
