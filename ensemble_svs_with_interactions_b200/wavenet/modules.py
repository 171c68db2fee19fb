"""WaveNet building blocks with the module tree of ``nnsvs.wavenet.modules`` (modules.py:6-140)."""
import torch
from torch import nn

from .. import ops
from . import conv

f32 = torch.float32


def _w(m):
    if hasattr(m, "weight_g"):
        return torch._weight_norm(m.weight_v, m.weight_g, 0).detach()
    return m.weight.detach()


def Conv1d(in_channels, out_channels, kernel_size, *args, **kwargs):
    """Weight-normalized Conv1d holder (modules.py:6-9)."""
    return nn.utils.weight_norm(conv.Conv1d(in_channels, out_channels, kernel_size, *args, **kwargs))


def Conv1d1x1(in_channels, out_channels, bias=True):
    return Conv1d(in_channels, out_channels, kernel_size=1, bias=bias)


class ResSkipBlock(nn.Module):
    """Causal dilated gated block with local conditioning (modules.py:17-140)."""

    def __init__(self, residual_channels, gate_channels, kernel_size, skip_out_channels, dilation=1, cin_channels=80,
                 *args, **kwargs):
        super().__init__()
        self.kernel_size, self.dilation = kernel_size, dilation
        self.padding = (kernel_size - 1) * dilation
        self.conv = Conv1d(residual_channels, gate_channels, kernel_size, *args, padding=self.padding,
                           dilation=dilation, **kwargs)
        self.conv1x1c = Conv1d1x1(cin_channels, gate_channels, bias=False)
        gate_out_channels = gate_channels // 2
        self.conv1x1_out = Conv1d1x1(gate_out_channels, residual_channels)
        self.conv1x1_skip = Conv1d1x1(gate_out_channels, skip_out_channels)

    @torch.no_grad()
    def forward(self, x, c):
        """x (B, R, T), c (B, cin, T) -> (x_out, skips) fp32, one launch (svsk_wavenet_block_f32): "pad (k-1)d both sides
        then trim right" (modules.py:99-101) == taps at t-(k-1-j)d, zero for t < 0; tanh on the first half of the gate
        channels, sigmoid on the second; x + res without a sqrt(1/2).  WaveNet runs its blocks from one pack of all layers
        (wavenet/training.py); this lays out the same w1t / w2t for one block (include/svsk.h)."""
        x = x.to(f32).contiguous()
        k, R = self.kernel_size, x.shape[1]
        w1t = torch.cat([_w(self.conv).to(f32).permute(2, 1, 0).reshape(k * R, -1), _w(self.conv1x1c).to(f32)[:, :, 0].t()])
        w2t = torch.cat([_w(self.conv1x1_skip)[:, :, 0], _w(self.conv1x1_out)[:, :, 0]]).to(f32).t().contiguous()
        b1 = None if self.conv.bias is None else self.conv.bias.detach().to(f32).contiguous()
        b2 = torch.cat([self.conv1x1_skip.bias.detach(), self.conv1x1_out.bias.detach()]).to(f32).contiguous()
        s = torch.empty((x.shape[0], self.conv1x1_skip.out_channels, x.shape[2]), device=x.device, dtype=f32)
        x = ops.wavenet_block_f32(x, c.to(f32).contiguous(), w1t, b1, w2t, b2, s, ksize=k, dilation=self.dilation, first=True)
        return x, s

    @torch.no_grad()
    def incremental_forward(self, x, c):
        """One autoregressive step, (B, 1, C) tensors (modules.py:76-122 with is_incremental=True)."""
        residual = x
        x = self.conv.incremental_forward(x)
        a, b = x.split(x.size(-1) // 2, dim=-1)
        cc = self.conv1x1c.incremental_forward(c)
        ca, cb = cc.split(cc.size(-1) // 2, dim=-1)
        x = torch.tanh(a + ca) * torch.sigmoid(b + cb)
        s = self.conv1x1_skip.incremental_forward(x)
        x = self.conv1x1_out.incremental_forward(x)
        return x + residual, s

    def clear_buffer(self):
        for c in (self.conv, self.conv1x1_out, self.conv1x1_skip, self.conv1x1c):
            c.clear_buffer()
