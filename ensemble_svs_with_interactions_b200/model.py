"""FFConvLSTM encoder — drop-in for ``nnsvs.model.FFConvLSTM`` / ``MultiSpeakerFFConvLSTM`` (nnsvs/model.py:779-1015).

SURVEY.md §8(f) row 1: the step right in front of the denoiser.  In the multi-track recipe it is the ``encoder`` of both
``GaussianDiffusion`` streams (conf/train_acoustic/model/multitrack_acoustic_nnsvs_world_multi_ar_f0_diff_mgcbap.yaml:
104-116,146-158) and runs once per track; its output is the ``cond`` tensor of every denoiser call.

Same constructor kwargs, ``forward`` / ``inference`` signatures and ``state_dict`` keys and order as the reference
(``emb``, ``fc_in``, ``ff.{0,2,4}``, ``conv.{1,2,5,6,9,10}``, ``lstm.*``, ``fc``); the ``nn`` sub-modules only hold
parameters, their ``forward`` never runs.  Eval-mode forward only (BatchNorm running statistics, no dropout):

* ``precision="fp32"``: svsk_conv1d_f32 for every Linear (k = 1) and for the reflect-padded k = 7 convolutions with the
  BatchNorm folded into weights and bias, svsk_lstm_f32 for the recurrences — the reference's fp32 arithmetic.
* ``precision="bf16"``: svsk_tapgemm_bf16 (tcgen05) for every matrix product on frame-major bf16 activations, the
  recurrence itself stays fp32 (svsk_lstm_f32 with W_hh in registers).
* ``precision="auto"`` (default): bf16 when every width is a multiple of 16, fp32 otherwise.

``use_mdn=True`` puts a dimension-wise mixture-density head (``MDNLayer``, nnsvs/mdn.py:6-74) in place of the output
Linear: ``forward`` returns (log_pi, log_sigma, mu) [B, T, G, D], ``inference`` the (mu, sigma) of the most probable
component (svsk_mdn_head_f32).  Training mode (module.train()): the FORWARD is built for dropout = 0 — what the diffusion
recipe's encoders use — i.e. BatchNorm1d with the batch statistics of the padded batch and the running-buffer update
(svsk_bn_batch_stats_f32 / svsk_bn_apply_f32; fp32 kernels whatever ``precision`` says, since the statistics are taken
on the convolution's own output).

``backward_kernels=True`` makes the module trainable on the device: in training mode with grad enabled, when ``x``,
``spk_embs`` or a parameter requires grad, ``forward`` is one autograd Function (encoder_training.py) and
``loss.backward()`` fills every parameter's ``.grad`` (and those of ``x`` / ``spk_embs``); output and BatchNorm buffers are
those of the no-grad training forward, bit for bit.  Eval mode and ``torch.no_grad()`` record no graph, as for WaveNet.
With the default ``backward_kernels=False`` a call that needs gradients raises (the MDN head has no backward either way).
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import nn

from . import encoder_training, ops
from .base import BaseModel, PredictionType

__all__ = ["FFConvLSTM", "MultiSpeakerFFConvLSTM", "MDNLayer", "init_weights"]


def init_weights(net: nn.Module, init_type: str = "normal", init_gain: float = 0.02) -> None:
    """nnsvs/util.py:31-67: (re)initialise Conv*/Linear weights, zero their biases; ``"none"`` leaves torch's defaults."""
    if init_type == "none":
        return
    inits = {
        "normal": lambda w: nn.init.normal_(w, 0.0, init_gain),
        "xavier_normal": lambda w: nn.init.xavier_normal_(w, gain=init_gain),
        "kaiming_normal": lambda w: nn.init.kaiming_normal_(w, a=0, mode="fan_in"),
        "orthogonal": lambda w: nn.init.orthogonal_(w, gain=init_gain),
    }
    if init_type not in inits:
        raise NotImplementedError("initialization method [%s] is not implemented" % init_type)

    def visit(m):
        name = type(m).__name__
        if hasattr(m, "weight") and ("Conv" in name or "Linear" in name):
            inits[init_type](m.weight.data)
            if getattr(m, "bias", None) is not None:
                nn.init.constant_(m.bias.data, 0.0)
        elif "BatchNorm2d" in name:
            nn.init.normal_(m.weight.data, 1.0, init_gain)
            nn.init.constant_(m.bias.data, 0.0)

    net.apply(visit)


class MDNLayer(nn.Module):
    """Parameter holder with the reference's layout (nnsvs/mdn.py:32-43): ``log_pi``, ``log_sigma``, ``mu`` Linears.  Only
    the dimension-wise form (one 1-D mixture per output dimension) is built — the one FFConvLSTM uses (model.py:872)."""

    def __init__(self, in_dim, out_dim, num_gaussians=30, dim_wise=False):
        super().__init__()
        if not dim_wise:
            raise NotImplementedError("MDNLayer(dim_wise=False) is not built in this package")
        self.in_dim, self.out_dim, self.num_gaussians, self.dim_wise = in_dim, out_dim, num_gaussians, dim_wise
        self.log_pi = nn.Linear(in_dim, out_dim * num_gaussians)
        self.log_sigma = nn.Linear(in_dim, out_dim * num_gaussians)
        self.mu = nn.Linear(in_dim, out_dim * num_gaussians)


def _padded_hidden(H: int) -> int:
    """Smallest hidden size >= H that svsk_lstm_f32 has a layout for (H itself when it has one; 0 if none up to 256).
    Padded units get zero weights: their gates see 0, the cell stays 0 and they emit h = 0 at every step."""
    for hp in range(H, 257):
        if ops.lstm_supported(hp):
            return hp
    return 0


def _pad_gate_rows(w, H, Hp):
    """[4H, ...] (torch gate blocks i, f, g, o) -> [4Hp, ...] with zero rows appended to every gate block."""
    if Hp == H:
        return w
    w4 = w.reshape(4, H, *w.shape[1:])
    out = w4.new_zeros((4, Hp) + tuple(w.shape[1:]))
    out[:, :H] = w4
    return out.reshape(4 * Hp, *w.shape[1:])


def _pad_bidir_cols(w, H, Hp):
    """[..., 2H] (forward | backward outputs of a BiLSTM layer) -> [..., 2Hp]: each half zero-padded to Hp columns."""
    if Hp == H:
        return w
    out = w.new_zeros(tuple(w.shape[:-1]) + (2 * Hp,))
    out[..., :H] = w[..., :H]
    out[..., Hp:Hp + H] = w[..., H:]
    return out


class _Plan:
    """Weights in the layouts the kernels read, built once per parameter version."""

    def __init__(self, m: "FFConvLSTM", precision: str):
        with torch.no_grad():
            self.precision = precision
            f = lambda t: t.detach().float().contiguous()
            # front: emb(argmax(onehot)) + fc_in(rest) == [fc_in | emb^T] applied to the input with an exact one-hot block
            if m.embed_dim is not None:
                s, V = m.in_ph_start_idx, m.num_vocab
                wc = torch.empty((m.embed_dim, m.in_dim), device=m.fc_in.weight.device, dtype=torch.float32)
                wc[:, :s] = m.fc_in.weight[:, :s]
                wc[:, s:s + V] = m.emb.weight.t()
                wc[:, s + V:] = m.fc_in.weight[:, s:]
                front = [(wc, f(m.fc_in.bias))]
            else:
                front = []
            ff = [(f(m.ff[i].weight), f(m.ff[i].bias)) for i in (0, 2, 4)]
            conv = []
            for i in (1, 5, 9):
                bn = m.conv[i + 1]
                scale = bn.weight.float() / torch.sqrt(bn.running_var.float() + bn.eps)
                bias = (m.conv[i].bias.float() - bn.running_mean.float()) * scale + bn.bias.float()
                conv.append((f(m.conv[i].weight), scale.contiguous(), bias.contiguous()))
            # hidden sizes without a cluster layout (the recipe's bap stream has 62 units) run zero-padded to the next one
            H, Hp = m.lstm_hidden_dim, m.padded_hidden
            self.Hp = Hp
            lstm = []
            for l in range(m.lstm.num_layers):
                g = lambda n: getattr(m.lstm, n.format(l)).float()
                parts = []
                for suf in ("", "_reverse"):
                    w_ih = g("weight_ih_l{}" + suf)
                    if l > 0:
                        w_ih = _pad_bidir_cols(w_ih, H, Hp)
                    parts.append((_pad_gate_rows(w_ih, H, Hp), _pad_gate_rows(g("bias_ih_l{}" + suf) + g("bias_hh_l{}" + suf), H, Hp),
                                  _pad_gate_rows(g("weight_hh_l{}" + suf), H, Hp)))
                w_ih = torch.cat([parts[0][0], parts[1][0]], 0).contiguous()
                b = torch.cat([parts[0][1], parts[1][1]], 0).contiguous()
                w_hh = torch.stack([torch.nn.functional.pad(parts[0][2], (0, Hp - H)), torch.nn.functional.pad(parts[1][2], (0, Hp - H))], 0).contiguous()
                lstm.append((w_ih, b, w_hh))
            if m.use_mdn:   # the three Linears of the head as one product: columns [log_pi | log_sigma | mu]
                fc = (torch.cat([f(m.fc.log_pi.weight), f(m.fc.log_sigma.weight), f(m.fc.mu.weight)], 0).contiguous(),
                      torch.cat([f(m.fc.log_pi.bias), f(m.fc.log_sigma.bias), f(m.fc.mu.bias)], 0).contiguous())
            else:
                fc = (f(m.fc.weight), f(m.fc.bias))
            if fc[0].shape[1] == 2 * H:
                fc = (_pad_bidir_cols(fc[0], H, Hp).contiguous(), fc[1])
            n_out = fc[0].shape[0]

            if precision == "fp32":
                k1 = lambda w: w.unsqueeze(-1).contiguous()
                self.front = [(k1(w), b) for w, b in front]
                self.ff = [(k1(w), b) for w, b in ff]
                self.conv = [((w * s[:, None, None]).contiguous(), b) for w, s, b in conv]
                self.lstm = [(k1(w), b, whh) for w, b, whh in lstm]
                self.fc = (k1(fc[0]), fc[1])
            else:
                self.front = [(ops.tapgemm_pack_bf16(w), b) for w, b in front]
                self.ff = [(ops.tapgemm_pack_bf16(w), b) for w, b in ff]
                self.conv = [(ops.tapgemm_pack_bf16(w, s), b) for w, s, b in conv]
                self.lstm = [(ops.tapgemm_pack_bf16(w), b, whh) for w, b, whh in lstm]
                out_p = -(-n_out // 16) * 16         # the GEMM writes 16 output channels at a time
                wf = torch.zeros((out_p, fc[0].shape[1]), device=fc[0].device, dtype=torch.float32)
                wf[:n_out] = fc[0]
                bf = torch.zeros(out_p, device=fc[0].device, dtype=torch.float32)
                bf[:n_out] = fc[1]
                self.fc = (ops.tapgemm_pack_bf16(wf), bf)
                self.out_p = out_p


class FFConvLSTM(BaseModel):
    """nnsvs/model.py:779-926.  ``precision``: "auto" | "bf16" | "fp32" (see the module docstring)."""

    def __init__(self, in_dim, ff_hidden_dim=2048, conv_hidden_dim=1024, lstm_hidden_dim=256, out_dim=67, dropout=0.0,
                 num_lstm_layers=2, bidirectional=True, init_type="none", use_mdn=False, dim_wise=True, num_gaussians=4,
                 in_ph_start_idx: int = 1, in_ph_end_idx: int = 50, embed_dim=None, precision="auto", backward_kernels=False):
        super().__init__()
        self.in_dim, self.out_dim = in_dim, out_dim
        self.num_gaussians = num_gaussians
        self.in_ph_start_idx, self.in_ph_end_idx = in_ph_start_idx, in_ph_end_idx
        self.num_vocab = in_ph_end_idx - in_ph_start_idx
        self.embed_dim = embed_dim
        self.use_mdn = use_mdn
        self.precision = precision
        self.backward_kernels = bool(backward_kernels)
        self.ff_hidden_dim, self.conv_hidden_dim, self.lstm_hidden_dim = ff_hidden_dim, conv_hidden_dim, lstm_hidden_dim
        self._padded_hidden = None

        if embed_dim is not None:
            assert in_dim > self.num_vocab
            self.emb = nn.Embedding(self.num_vocab, embed_dim)
            self.fc_in = nn.Linear(in_dim - self.num_vocab, embed_dim)
            ff_in_dim = embed_dim
        else:
            ff_in_dim = in_dim
        self.ff = nn.Sequential(nn.Linear(ff_in_dim, ff_hidden_dim), nn.ReLU(), nn.Linear(ff_hidden_dim, ff_hidden_dim), nn.ReLU(),
                                nn.Linear(ff_hidden_dim, ff_hidden_dim), nn.ReLU())
        layers, c_in = [], ff_hidden_dim
        for _ in range(3):
            layers += [nn.ReflectionPad1d(3), nn.Conv1d(c_in, conv_hidden_dim, kernel_size=7, padding=0),
                       nn.BatchNorm1d(conv_hidden_dim), nn.ReLU()]
            c_in = conv_hidden_dim
        self.conv = nn.Sequential(*layers)
        # the reference builds the LSTM bidirectional whatever `bidirectional` says (model.py:861-868)
        self.lstm = nn.LSTM(conv_hidden_dim, lstm_hidden_dim, num_lstm_layers, bidirectional=True, batch_first=True, dropout=dropout)
        last_in_dim = (2 if bidirectional else 1) * lstm_hidden_dim
        if use_mdn:
            assert dim_wise
            self.fc = MDNLayer(in_dim=last_in_dim, out_dim=out_dim, num_gaussians=num_gaussians, dim_wise=dim_wise)
        else:
            self.fc = nn.Linear(last_in_dim, out_dim)
        init_weights(self, init_type)
        self._plan: Optional[_Plan] = None
        self._plan_key = None

    def prediction_type(self):
        return PredictionType.PROBABILISTIC if self.use_mdn else PredictionType.DETERMINISTIC

    @property
    def padded_hidden(self) -> int:
        """Hidden size the recurrence kernel runs with (>= lstm_hidden_dim; the extra units are inert zeros)."""
        if self._padded_hidden is None:
            self._padded_hidden = _padded_hidden(self.lstm_hidden_dim)
        return self._padded_hidden

    # ------------------------------------------------------------------ precision / plan
    def resolved_precision(self) -> str:
        widths = [self.ff_hidden_dim, self.conv_hidden_dim] + ([self.embed_dim] if self.embed_dim else [])
        ok = all(w % 16 == 0 for w in widths)
        if self.precision == "auto":
            return "bf16" if ok else "fp32"
        if self.precision == "bf16" and not ok:
            raise RuntimeError(f"FFConvLSTM precision='bf16' needs every layer width to be a multiple of 16, got {widths}")
        if self.precision not in ("bf16", "fp32"):
            raise RuntimeError(f"unknown precision {self.precision!r}")
        return self.precision

    def plan(self) -> _Plan:
        prec = self.resolved_precision()
        key = (prec,) + tuple((p.data_ptr(), p._version) for p in list(self.parameters()) + list(self.buffers()))
        if self._plan is None or self._plan_key != key:
            self._plan, self._plan_key = _Plan(self, prec), key
        return self._plan

    # ------------------------------------------------------------------ forward
    def _records_grad(self, x, spk_embs):
        """True when forward runs as the autograd Function: backward_kernels, training mode, grad enabled and something
        that requires grad."""
        return (self.backward_kernels and self.training and torch.is_grad_enabled()
                and (x.requires_grad or (spk_embs is not None and spk_embs.requires_grad)
                     or any(p.requires_grad for p in self.parameters())))

    def _check(self, x, lengths, spk_embs=None):
        if self.training:
            if self.lstm.dropout > 0 and self.lstm.num_layers > 1:
                raise RuntimeError("FFConvLSTM: the training-mode forward is built for dropout = 0 only (the diffusion recipe's "
                                   f"encoders); got dropout = {self.lstm.dropout}.  Call .eval() for inference")
            if not self.backward_kernels:
                if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
                    raise RuntimeError("FFConvLSTM has no backward kernels: the training-mode forward (BatchNorm batch statistics, "
                                       "running-buffer update) runs under torch.no_grad() or with frozen parameters only; "
                                       "construct with backward_kernels=True to train it on the device")
            elif self.use_mdn and self._records_grad(x, spk_embs):
                raise RuntimeError("FFConvLSTM(backward_kernels=True): the MDN head (use_mdn=True) has no backward kernels; "
                                   "train it with use_mdn=False or run the training forward under torch.no_grad()")
        if not x.is_cuda:
            raise RuntimeError("FFConvLSTM: input must be a CUDA tensor (libsvsk has no CPU path)")
        if x.dim() != 3 or x.shape[-1] != self.in_dim:
            raise RuntimeError(f"FFConvLSTM: expected input [B, T, {self.in_dim}], got {tuple(x.shape)}")
        if x.shape[1] < 4:
            raise RuntimeError("FFConvLSTM: ReflectionPad1d(3) needs at least 4 frames")
        if not self.padded_hidden:
            raise RuntimeError(f"FFConvLSTM: lstm_hidden_dim={self.lstm_hidden_dim} has no layout in svsk_lstm_f32 (at most 256 units)")
        B, T = x.shape[0], x.shape[1]
        if lengths is None:
            lens = [T] * B
        else:
            lens = [int(n) for n in (lengths.tolist() if isinstance(lengths, torch.Tensor) else lengths)]
            if len(lens) != B or max(lens) > T or min(lens) < 1:
                raise RuntimeError(f"FFConvLSTM: lengths {lens} do not fit a batch of {B} x {T} frames")
        return lens

    def _raw(self, x, lengths, spk_embs):
        """Output of the last product, [B, max(lengths), >= n_out] fp32 (a view when the GEMM padded its columns)."""
        lens = self._check(x, lengths)
        x = x.detach().float().contiguous()
        lens_dev = torch.tensor(lens, dtype=torch.int32, device=x.device)
        if spk_embs is not None:
            spk_embs = spk_embs.detach().float().expand(x.shape[0], x.shape[1], spk_embs.shape[-1]).contiguous()
        if self.training:
            # BatchNorm1d with batch statistics (model.py:839-852 under module.train()): the fp32 kernels, the convolutions'
            # own weights (nothing folded), the running buffers updated in place -> the cached eval plan is stale afterwards
            plan = self._train_plan()
            with torch.no_grad():
                out = self._forward_fp32(x, lens_dev, spk_embs, plan, train=True)
            self._plan = None
            return out[:, :max(lens)]
        plan = self.plan()
        out = self._forward_fp32(x, lens_dev, spk_embs, plan) if plan.precision == "fp32" else self._forward_bf16(x, lens_dev, spk_embs, plan)
        return out[:, :max(lens)]

    def _train_plan(self) -> _Plan:
        """fp32 weights of the training forward, rebuilt when a parameter changes."""
        key = tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self.__dict__.get("_plan_train_key") != key:
            self.__dict__["_plan_train"], self.__dict__["_plan_train_key"] = _Plan(self, "fp32"), key
        return self.__dict__["_plan_train"]

    def forward(self, x, lengths=None, y=None, spk_embs=None):
        if self._records_grad(x, spk_embs):
            lens = self._check(x, lengths, spk_embs)
            return encoder_training.ffconvlstm_forward_with_grad(self, x, lens, spk_embs)
        raw = self._raw(x, lengths, spk_embs)
        if self.use_mdn:     # (log_pi, log_sigma, mu), each [B, T, G, D]  (mdn.py:45-74)
            return ops.mdn_head_f32(raw.contiguous(), self.num_gaussians, self.out_dim)[0]
        return raw[:, :, :self.out_dim].contiguous()

    def inference(self, x, lengths=None, spk_embs=None):
        if self.use_mdn:     # (mu, sigma) of the most probable component (model.py:925-928; no speaker embedding there)
            raw = self._raw(x, lengths, None)
            sigma, mu = ops.mdn_head_f32(raw.contiguous(), self.num_gaussians, self.out_dim, want_params=False, want_best=True)[1]
            return mu, sigma
        return self(x, lengths, spk_embs=spk_embs)

    def _forward_fp32(self, x, lens_dev, spk, plan, train=False, keep=None):
        """keep (training only): a dict that receives what encoder_training's backward needs; the BatchNorm is then applied
        out of place and the recurrences also store their gates and cells — the same kernels and the same output bits."""
        B, T, _ = x.shape
        H = plan.Hp
        if self.embed_dim is not None:
            xf = torch.empty((B * T, self.in_dim), device=x.device, dtype=torch.float32)
            ops.encoder_front(x.view(B * T, self.in_dim), self.in_ph_start_idx, self.num_vocab, y_f32=xf)
            h = ops.ntc_to_nct_f32(xf.view(B, T, self.in_dim), self.in_dim)
            if keep is not None:
                keep["front_in"] = h
            h = ops.conv1d_f32(h, plan.front[0][0], plan.front[0][1])
        else:
            h = ops.ntc_to_nct_f32(x, self.in_dim)
        if spk is not None:
            h = ops.lincomb_f32([h, ops.ntc_to_nct_f32(spk, spk.shape[-1])], [1.0, 1.0])
        ff = [h]
        for w, b in plan.ff:
            h = ops.conv1d_f32(h, w, b, act=ops.ACT_RELU)
            ff.append(h)
        if keep is not None:
            keep.update(ff=ff, conv=[], lstm=[])
        for k, (w, b) in enumerate(plan.conv):
            if train:
                conv, bn = self.conv[4 * k + 1], self.conv[4 * k + 2]
                if bn.momentum is None or not bn.track_running_stats:
                    raise RuntimeError("FFConvLSTM: BatchNorm1d(momentum=None / track_running_stats=False) is not built")
                a_in = h
                h = ops.conv1d_f32(h, conv.weight.detach().float().contiguous(), conv.bias.detach().float().contiguous(),
                                   pad_mode=ops.PAD_REFLECT)
                z = h
                stats = None if keep is None else (torch.empty_like(h[0, :, 0]), torch.empty_like(h[0, :, 0]))
                h = ops.batchnorm_train_f32(z, bn.weight.detach().float().contiguous(), bn.bias.detach().float().contiguous(),
                                            bn.running_mean, bn.running_var, eps=bn.eps, momentum=bn.momentum, relu=True,
                                            out=None if keep is None else torch.empty_like(z), stats=stats)
                bn.num_batches_tracked += 1
                if keep is not None:
                    keep["conv"].append((z, stats, h, a_in))
            else:
                h = ops.conv1d_f32(h, w, b, pad_mode=ops.PAD_REFLECT, act=ops.ACT_RELU)
        for w_ih, b, w_hh in plan.lstm:
            pre = ops.conv1d_f32(h, w_ih, b)                                   # [B, 8H, T]
            h_in, h = h, torch.empty((B, 2 * H, T), device=x.device, dtype=torch.float32)
            if keep is None:
                ops.lstm_f32(pre, w_hh, lens_dev, H, pre_layout="nct", h_f32=h)
            else:
                gates, cell = torch.empty_like(pre), torch.empty_like(h)
                ops.lstm_train_f32(pre, w_hh, lens_dev, H, h_f32=h, gates=gates, cell=cell)
                keep["lstm"].append((h_in, h, gates, cell))
        y = ops.conv1d_f32(h, plan.fc[0], plan.fc[1])                          # [B, n_out, T]
        return ops.nct_to_ntc(y, want_bf16=False, want_f32=True)[1]

    def _forward_bf16(self, x, lens_dev, spk, plan):
        B, T, _ = x.shape
        dev, H, bf = x.device, plan.Hp, torch.bfloat16
        ld0 = -(-self.in_dim // 8) * 8
        if spk is not None and self.embed_dim is None:
            x = ops.lincomb_f32([x, spk], [1.0, 1.0])
        h = torch.empty((B, T, ld0), device=dev, dtype=bf)
        ops.encoder_front(x.view(B * T, self.in_dim), self.in_ph_start_idx, self.num_vocab if self.embed_dim is not None else 0,
                          y_bf16=h.view(B * T, ld0))
        c_in = self.in_dim
        if self.embed_dim is not None:
            E = self.embed_dim
            if spk is None:
                e = torch.empty((B, T, E), device=dev, dtype=bf)
                ops.tapgemm_bf16(h, plan.front[0][0], plan.front[0][1], c_in, T=T, y_bf16=e)
            else:
                e32 = torch.empty((B, T, E), device=dev, dtype=torch.float32)
                ops.tapgemm_bf16(h, plan.front[0][0], plan.front[0][1], c_in, T=T, y_f32=e32)
                e = ops.cast_scale_bf16(ops.lincomb_f32([e32, spk], [1.0, 1.0]))
            h, c_in = e, E
        # ff: the last layer writes into the time-padded input buffer of the first convolution
        F_, Cc = self.ff_hidden_dim, self.conv_hidden_dim
        for i, (w, b) in enumerate(plan.ff):
            last = i == len(plan.ff) - 1
            y = torch.empty((B, T + 6 if last else T, F_), device=dev, dtype=bf)
            ops.tapgemm_bf16(h, w, b, c_in, T=T, act=ops.ACT_RELU, y_bf16=y, y_row0=3 if last else 0)
            h, c_in = y, F_
        for i, (w, b) in enumerate(plan.conv):
            ops.reflect_pad_rows_bf16(h, T, 3)
            last = i == len(plan.conv) - 1
            y = torch.empty((B, T if last else T + 6, Cc), device=dev, dtype=bf)
            ops.tapgemm_bf16(h, w, b, c_in, T=T, act=ops.ACT_RELU, y_bf16=y, y_row0=0 if last else 3)
            h, c_in = y, Cc
        for w_ih, b, w_hh in plan.lstm:
            pre = torch.empty((B, T, 8 * H), device=dev, dtype=torch.float32)
            ops.tapgemm_bf16(h, w_ih, b, c_in, T=T, y_f32=pre)
            h = torch.empty((B, T, 2 * H), device=dev, dtype=bf)
            ops.lstm_f32(pre, w_hh, lens_dev, H, pre_layout="ntc", h_bf16=h)
            c_in = 2 * H
        y = torch.empty((B, T, plan.out_p), device=dev, dtype=torch.float32)
        ops.tapgemm_bf16(h, plan.fc[0], plan.fc[1], c_in, T=T, y_f32=y)
        return y


class MultiSpeakerFFConvLSTM(FFConvLSTM):
    """nnsvs/model.py:929-1015: the speaker embedding of ``spks`` is broadcast over time and added in front of ``ff``."""

    def __init__(self, in_dim, speaker_embedding, ff_hidden_dim=2048, conv_hidden_dim=1024, lstm_hidden_dim=256, out_dim=67,
                 dropout=0.0, num_lstm_layers=2, bidirectional=True, init_type="none", use_mdn=False, dim_wise=True,
                 num_gaussians=4, in_ph_start_idx: int = 1, in_ph_end_idx: int = 50, embed_dim=None, precision="auto",
                 backward_kernels=False):
        super().__init__(in_dim, ff_hidden_dim, conv_hidden_dim, lstm_hidden_dim, out_dim, dropout, num_lstm_layers, bidirectional,
                         init_type, use_mdn, dim_wise, num_gaussians, in_ph_start_idx, in_ph_end_idx, embed_dim, precision,
                         backward_kernels)
        self.speaker_embedding = speaker_embedding

    def forward(self, x, spks, lengths=None, y=None):
        spk_embs = self.speaker_embedding(spks)
        return super().forward(x, lengths, spk_embs=spk_embs.expand(spk_embs.shape[0], x.shape[1], spk_embs.shape[-1]))

    def inference(self, x, spks, lengths=None):
        return self(x, spks, lengths)
