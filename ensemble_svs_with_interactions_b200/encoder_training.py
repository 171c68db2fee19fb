"""Training-time FFConvLSTM forward AND backward on libsvsk kernels: ``FFConvLSTM.forward`` under autograd
(nnsvs/model.py:893-922 with dropout = 0), trained through ``loss.backward()`` like the reference.  Used when the module
is built with ``backward_kernels=True``.

The whole encoder is ONE ``torch.autograd.Function`` over its parameters (reference names and shapes; the kernel layouts
— the [fc_in | emb^T] front, hidden sizes zero-padded to a cluster layout — are rebuilt on every forward):

forward (FFConvLSTM._forward_fp32(train=True), the kernels and order of the no-grad training forward, same bits)
    front / ff: svsk_conv1d_f32 (+ReLU);  conv_k: svsk_conv1d_f32 (reflect) -> svsk_bn_batch_stats_f32 ->
    svsk_bn_apply_f32 out of place (the BatchNorm input is kept);  LSTM layer l: svsk_conv1d_f32 (W_ih) ->
    svsk_lstm_train_f32 (keeps gates and c_t);  fc: svsk_conv1d_f32
backward (gy = upstream gradient, [B, out_dim, T], zero past max(lengths))
    fc:       dW, db = svsk_wgrad_f32(gy, h_L);  dh_L = fc^T gy                                   svsk_conv1d_f32
    LSTM l:   dpre = svsk_lstm_bwd_f32(dh_l);  dW_ih, db = svsk_wgrad_f32(dpre, h_{l-1});
              dW_hh[d] = svsk_wgrad_f32(dpre[d], h_l[d], shift -1 / +1);  dh_{l-1} = W_ih^T dpre
    conv k:   dz, dgamma, dbeta = svsk_bn_relu_bwd_f32;  dW, db = svsk_wgrad_f32(dz, a_{k-1}, k = 7, reflect);
              da_{k-1} = conv(dz, W flipped^T) + svsk_reflect_fold_f32
    ff i:     dz = svsk_relu_mask_f32;  dW, db = svsk_wgrad_f32(dz, a_{i-1});  da_{i-1} = W^T dz
    front:    d[fc_in | emb^T], dfc_in.bias = svsk_wgrad_f32(de, one-hot input);  dx = [fc_in | 0]^T de
dspk_embs is the gradient at the sum in front of ``ff``.  The one-hot columns of x only feed argmax: their gradient is 0.

Numerics: fp32 on the CUDA cores throughout, like the training forward; no atomics, so gradients are bit-reproducible.
"""
from __future__ import annotations

import torch

from . import ops

f32 = torch.float32


def _params(m):
    """[(name, parameter)] of the encoder itself (a MultiSpeakerFFConvLSTM's speaker embedding trains through torch)."""
    return [(n, p) for n, p in m.named_parameters() if not n.startswith("speaker_embedding.")]


def _t1(w):
    """[Cout, Cin, 1] -> [Cin, Cout, 1]: the weights of the transposed 1x1 product."""
    return w.squeeze(-1).t().contiguous().unsqueeze(-1)


def _forward(m, x, lens, spk):
    """Training forward of module m -> (output [B, max(lens), out_dim], what the backward keeps)."""
    B, T, _ = x.shape
    lens_dev = torch.tensor(lens, dtype=torch.int32, device=x.device)
    if spk is not None:
        spk = spk.float().expand(B, T, spk.shape[-1]).contiguous()
    plan = m._train_plan()
    keep = {}
    out = m._forward_fp32(x.float().contiguous(), lens_dev, spk, plan, train=True, keep=keep)
    m._plan = None
    keep.update(plan=plan, lens_dev=lens_dev, T=T)
    return out[:, :max(lens), :m.out_dim].contiguous(), keep


def _backward(m, keep, g):
    """Backward kernels -> (dx [B, in_dim, T] or frame-major input gradient, dspk [B, S, T] or None, {name: gradient in
    the kernels' padded layouts})."""
    plan, lens_dev, T = keep["plan"], keep["lens_dev"], keep["T"]
    B, Tm, n_out = g.shape
    gy = torch.zeros((B, n_out, T), device=g.device, dtype=f32)
    gy[:, :, :Tm] = g.transpose(1, 2)
    grads = {}
    # output Linear
    h = keep["lstm"][-1][1]
    grads["fc.weight"], grads["fc.bias"] = ops.wgrad_f32(gy, h)
    dh = ops.conv1d_f32(gy, _t1(plan.fc[0]))
    # LSTM layers, last first
    Hp = plan.Hp
    for l in range(len(plan.lstm) - 1, -1, -1):
        w_ih, _, w_hh = plan.lstm[l]
        hin, hout, gates, cell = keep["lstm"][l]
        dpre = ops.lstm_bwd_f32(dh, gates, cell, w_hh, lens_dev, Hp)
        grads[f"lstm.w_ih{l}"], grads[f"lstm.b{l}"] = ops.wgrad_f32(dpre, hin)
        grads[f"lstm.w_hh{l}"] = [ops.wgrad_f32(dpre[:, d * 4 * Hp:(d + 1) * 4 * Hp], hout[:, d * Hp:(d + 1) * Hp],
                                                origin=1 if d == 0 else -1, bias=False)[0] for d in range(2)]
        dh = ops.conv1d_f32(dpre, _t1(w_ih))
    # conv layers, last first: dh is the gradient of the last conv layer's ReLU output
    for k in range(2, -1, -1):
        conv, bn = m.conv[4 * k + 1], m.conv[4 * k + 2]
        z, (mean, var), y, a_in = keep["conv"][k]
        gamma = bn.weight.detach().float().contiguous()
        dz, grads[f"conv.{4 * k + 2}.weight"], grads[f"conv.{4 * k + 2}.bias"] = ops.bn_relu_bwd_f32(dh, y, z, mean, var, gamma, eps=bn.eps)
        w = conv.weight.detach().float().contiguous()
        grads[f"conv.{4 * k + 1}.weight"], grads[f"conv.{4 * k + 1}.bias"] = ops.wgrad_f32(dz, a_in, ksize=7, origin=3,
                                                                                      pad_mode=ops.PAD_REFLECT)
        dh = ops.conv1d_f32(dz, w.flip(-1).transpose(0, 1).contiguous())
        ops.reflect_fold_f32(dh, dz, w)
    # ff: dh is the gradient of ff[4]'s ReLU output
    for i in range(2, -1, -1):
        a_in, a_out = keep["ff"][i], keep["ff"][i + 1]
        dz = ops.relu_mask_f32(dh, a_out)
        grads[f"ff.{2 * i}.weight"], grads[f"ff.{2 * i}.bias"] = ops.wgrad_f32(dz, a_in)
        dh = ops.conv1d_f32(dz, _t1(plan.ff[i][0]))
    dspk = dh if keep["has_spk"] else None
    if m.embed_dim is not None:
        grads["front"], grads["fc_in.bias"] = ops.wgrad_f32(dh, keep["front_in"])
        s, V = m.in_ph_start_idx, m.num_vocab
        wT = _t1(plan.front[0][0])
        wT[s:s + V] = 0           # the one-hot block only feeds argmax
        dx = ops.conv1d_f32(dh, wT)
    else:
        dx = dh
    return dx, dspk, grads


def _scatter(m, grads):
    """Kernel-layout gradients -> {parameter name: gradient in the reference shape}; the padding of hidden sizes without a
    cluster layout (it provably carries zero gradient) is dropped here."""
    H, Hp = m.lstm_hidden_dim, grads["fc.weight"].shape[1] // 2
    unpad_rows = lambda t: t.reshape(4, Hp, *t.shape[1:])[:, :H].reshape(4 * H, *t.shape[1:])
    unpad_cols = lambda t: torch.cat([t[..., :H], t[..., Hp:Hp + H]], dim=-1)
    out = {"fc.weight": unpad_cols(grads["fc.weight"].squeeze(-1)), "fc.bias": grads["fc.bias"]}
    for l in range(m.lstm.num_layers):
        w_ih, b = grads[f"lstm.w_ih{l}"].squeeze(-1), grads[f"lstm.b{l}"]
        if l > 0:
            w_ih = unpad_cols(w_ih)
        for d, suf in enumerate(("", "_reverse")):
            rows = slice(d * 4 * Hp, (d + 1) * 4 * Hp)
            out[f"lstm.weight_ih_l{l}{suf}"] = unpad_rows(w_ih[rows])
            out[f"lstm.bias_ih_l{l}{suf}"] = out[f"lstm.bias_hh_l{l}{suf}"] = unpad_rows(b[rows])
            out[f"lstm.weight_hh_l{l}{suf}"] = unpad_rows(grads[f"lstm.w_hh{l}"][d].squeeze(-1))[:, :H]
    for k in (1, 2, 5, 6, 9, 10):
        out[f"conv.{k}.weight"], out[f"conv.{k}.bias"] = grads[f"conv.{k}.weight"], grads[f"conv.{k}.bias"]
    for i in (0, 2, 4):
        out[f"ff.{i}.weight"], out[f"ff.{i}.bias"] = grads[f"ff.{i}.weight"].squeeze(-1), grads[f"ff.{i}.bias"]
    if m.embed_dim is not None:
        s, V = m.in_ph_start_idx, m.num_vocab
        wc = grads["front"].squeeze(-1)
        out["emb.weight"] = wc[:, s:s + V].t()
        out["fc_in.weight"] = torch.cat([wc[:, :s], wc[:, s + V:]], dim=1)
        out["fc_in.bias"] = grads["fc_in.bias"]
    return out


class _EncoderFn(torch.autograd.Function):
    """out (B, max(lens), out_dim) = FFConvLSTM(x (B, T, in_dim), spk_embs (B, T, S) or None) in training mode."""

    @staticmethod
    def forward(ctx, m, lens, names, x, spk, *params):
        out, keep = _forward(m, x, lens, spk)
        keep["has_spk"] = spk is not None
        ctx.m, ctx.names, ctx.keep = m, names, keep
        ctx.shapes = tuple(p.shape for p in params)
        ctx.x_dtype = x.dtype
        ctx.spk_dtype = None if spk is None else spk.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        m = ctx.m
        dx, dspk, grads = _backward(m, ctx.keep, g.to(f32).contiguous())
        ctx.keep = None
        full = _scatter(m, grads)
        dx = dx.transpose(1, 2).to(ctx.x_dtype) if ctx.needs_input_grad[3] else None
        dspk = dspk.transpose(1, 2).to(ctx.spk_dtype) if dspk is not None and ctx.needs_input_grad[4] else None
        pg = tuple(full[n].reshape(p_shape).contiguous() if need else None
                   for n, p_shape, need in zip(ctx.names, ctx.shapes, ctx.needs_input_grad[5:]))
        return (None, None, None, dx, dspk) + pg


def ffconvlstm_forward_with_grad(m, x, lens, spk_embs):
    """FFConvLSTM.forward under autograd (module.train(), backward_kernels=True): [B, max(lens), out_dim] with a grad_fn;
    output and BatchNorm buffers are those of the no-grad training forward, bit for bit."""
    if not x.is_cuda:
        raise RuntimeError("FFConvLSTM: input must be a CUDA tensor (libsvsk has no CPU path)")
    items = _params(m)
    names = tuple(n for n, _ in items)
    if spk_embs is not None:
        spk_embs = spk_embs.expand(x.shape[0], x.shape[1], spk_embs.shape[-1])
    return _EncoderFn.apply(m, tuple(lens), names, x, spk_embs, *[p for _, p in items])
