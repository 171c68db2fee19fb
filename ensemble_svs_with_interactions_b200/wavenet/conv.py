"""``Conv1d`` parameter holder with the incremental (one-sample) evaluation API of ``nnsvs.wavenet.conv``
(nnsvs/wavenet/conv.py:9-69).  Used by ``WaveNet.incremental_logits`` and by the host loop of
``WaveNet.inference`` for CPU tensors and shapes the device sampler (svsk_wavenet_ar_f32) does not cover."""
import torch
from torch import nn
from torch.nn import functional as F


class Conv1d(nn.Conv1d):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.clear_buffer()
        self._linearized_weight = None

    def _current_weight(self):
        if hasattr(self, "weight_g"):
            return torch._weight_norm(self.weight_v, self.weight_g, 0)
        return self.weight

    def incremental_forward(self, input):
        """input (B, 1, C): push one frame, return the conv output for it (B, 1, Cout)."""
        if self.training:
            raise RuntimeError("incremental_forward only supports eval mode")
        kw, dil = self.kernel_size[0], self.dilation[0]
        bsz = input.size(0)
        w = self._current_weight().detach()
        w_lin = w.transpose(1, 2).reshape(self.out_channels, -1)  # (Cout, kw*Cin), tap-major like the ring buffer
        if kw > 1:
            span = kw + (kw - 1) * (dil - 1)
            if self.input_buffer is None:
                self.input_buffer = input.new_zeros(bsz, span, input.size(2))
            else:
                self.input_buffer = torch.roll(self.input_buffer, -1, dims=1)
            self.input_buffer[:, -1, :] = input[:, -1, :]
            input = self.input_buffer[:, 0::dil, :] if dil > 1 else self.input_buffer
        with torch.no_grad():
            out = F.linear(input.reshape(bsz, -1), w_lin, self.bias)
        return out.view(bsz, 1, -1)

    def clear_buffer(self):
        self.input_buffer = None
