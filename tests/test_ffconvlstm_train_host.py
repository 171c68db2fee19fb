"""CPU-only: the FFConvLSTM training entries (svsk_lstm_train_f32, svsk_lstm_bwd_f32, svsk_wgrad_f32,
svsk_bn_relu_bwd_f32, svsk_reflect_fold_f32) reject bad arguments before any launch, their wrappers check shapes first,
and the opt-in training path of FFConvLSTM refuses what it does not build before launching anything."""
import ctypes as C
import inspect

import pytest
import torch

from ensemble_svs_with_interactions_b200 import _lib, ops
from ensemble_svs_with_interactions_b200.model import FFConvLSTM, MultiSpeakerFFConvLSTM

NEW = ("svsk_lstm_train_f32", "svsk_lstm_bwd_f32", "svsk_wgrad_f32", "svsk_bn_relu_bwd_f32", "svsk_reflect_fold_f32")


def test_new_symbols_are_exported():
    for n in NEW:
        assert n in _lib.EXPORTED_SYMBOLS
        assert hasattr(_lib.lib(), n)


def test_null_and_bad_arguments_are_rejected():
    l = _lib.lib()
    assert l.svsk_lstm_train_f32(None, None, None, None) == -1
    assert b"null params" in l.svsk_last_error()
    p = _lib.LstmParams()
    p.pre = p.w_hh = p.h_f32 = 256
    p.B, p.T, p.H, p.ndir = 2, 10, 16, 2
    assert l.svsk_lstm_train_f32(C.byref(p), None, None, None) == -1
    assert b"gates / cell" in l.svsk_last_error()
    p.H = 300
    assert l.svsk_lstm_train_f32(C.byref(p), 256, 256, None) == -1
    assert b"no cluster layout" in l.svsk_last_error()

    assert l.svsk_lstm_bwd_f32(None, None) == -1
    q = _lib.LstmBwdParams()
    q.dh = q.gates = q.cell = q.w_hh = 256
    q.B, q.T, q.H, q.ndir = 2, 10, 16, 2
    assert l.svsk_lstm_bwd_f32(C.byref(q), None) == -1                      # dpre missing
    assert b"null tensor" in l.svsk_last_error()
    q.dpre, q.H = 256, 62
    assert l.svsk_lstm_bwd_f32(C.byref(q), None) == -1
    assert b"no cluster layout" in l.svsk_last_error()
    q.H, q.ndir = 64, 3
    assert l.svsk_lstm_bwd_f32(C.byref(q), None) == -1

    assert l.svsk_wgrad_f32(None, None) == -1
    w = _lib.WgradF32Params()
    w.dy = w.x = w.dw = 256
    w.B, w.N, w.K, w.T, w.ksize, w.origin, w.pad_mode, w.splits = 2, 8, 8, 10, 7, 3, ops.PAD_REFLECT, 1
    w.dy_batch_stride, w.x_batch_stride = 80, 80
    w.splits = 2
    assert l.svsk_wgrad_f32(C.byref(w), None) == -1
    assert b"workspace" in l.svsk_last_error()
    w.splits, w.T, w.dy_batch_stride, w.x_batch_stride = 1, 3, 24, 24      # reflect reach 3 needs T > 3
    assert l.svsk_wgrad_f32(C.byref(w), None) == -1
    assert b"reflect" in l.svsk_last_error()
    w.T, w.pad_mode = 10, ops.PAD_REPLICATE
    assert l.svsk_wgrad_f32(C.byref(w), None) == -1
    w.pad_mode, w.dy_batch_stride = ops.PAD_ZEROS, 10                       # batch stride below N T
    assert l.svsk_wgrad_f32(C.byref(w), None) == -1
    assert b"batch strides" in l.svsk_last_error()

    assert l.svsk_bn_relu_bwd_f32(None, 256, 256, 256, 256, 256, 1e-5, 256, 256, 256, 2, 4, 8, None) == -1
    assert l.svsk_bn_relu_bwd_f32(256, 256, 256, 256, 256, 256, 0.0, 256, 256, 256, 2, 4, 8, None) == -1
    assert l.svsk_reflect_fold_f32(None, 256, 256, 2, 4, 4, 8, 3, None) == -1
    assert l.svsk_reflect_fold_f32(256, 256, 256, 2, 4, 4, 3, 3, None) == -1
    assert b"needs T > 3" in l.svsk_last_error()
    assert l.svsk_reflect_fold_f32(256, 256, 256, 2, 4, 4, 30, 5, None) == -1


def test_wrappers_reject_mismatched_shapes():
    B, H, T = 2, 16, 10
    with pytest.raises(ValueError, match="gates"):
        ops.lstm_train_f32(torch.zeros(B, 8 * H, T), torch.zeros(2, 4 * H, H), None, H, h_f32=torch.zeros(B, 2 * H, T),
                           gates=torch.zeros(B, 8 * H, T + 1), cell=torch.zeros(B, 2 * H, T))
    with pytest.raises(ValueError, match="cell"):
        ops.lstm_bwd_f32(torch.zeros(B, 2 * H, T), torch.zeros(B, 8 * H, T), torch.zeros(B, H, T), torch.zeros(2, 4 * H, H), None, H)
    with pytest.raises(ValueError, match="lengths"):
        ops.lstm_bwd_f32(torch.zeros(B, 2 * H, T), torch.zeros(B, 8 * H, T), torch.zeros(B, 2 * H, T), torch.zeros(2, 4 * H, H),
                         torch.zeros(B + 1, dtype=torch.int32), H)
    with pytest.raises(ValueError, match="x must be"):
        ops.wgrad_f32(torch.zeros(B, 8, T), torch.zeros(B, 4, T + 1))
    with pytest.raises(ValueError, match="contiguous frames"):
        ops.wgrad_f32(torch.zeros(B, T, 8).transpose(1, 2), torch.zeros(B, 4, T))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.wgrad_f32(torch.zeros(B, 8, T), torch.zeros(B, 4, T))
    with pytest.raises(ValueError, match="gamma"):
        ops.bn_relu_bwd_f32(torch.zeros(B, 4, T), torch.zeros(B, 4, T), torch.zeros(B, 4, T), torch.zeros(4), torch.zeros(4),
                            torch.zeros(5), eps=1e-5)
    with pytest.raises(ValueError, match="odd k"):
        ops.reflect_fold_f32(torch.zeros(B, 4, T), torch.zeros(B, 6, T), torch.zeros(6, 4, 6))
    with pytest.raises(ValueError, match="dy"):
        ops.reflect_fold_f32(torch.zeros(B, 4, T), torch.zeros(B, 5, T), torch.zeros(6, 4, 7))
    with pytest.raises(ValueError, match="out"):
        ops.batchnorm_train_f32(torch.zeros(B, 4, T), None, None, None, None, eps=1e-5, momentum=0.1, out=torch.zeros(B, 4, T + 1))


def test_keyword_is_last_and_off_by_default():
    for cls in (FFConvLSTM, MultiSpeakerFFConvLSTM):
        names = list(inspect.signature(cls.__init__).parameters)
        assert names[-1] == "backward_kernels" and names[-2] == "precision"
        assert inspect.signature(cls.__init__).parameters["backward_kernels"].default is False
    assert FFConvLSTM(16, 32, 16, 8, 4).backward_kernels is False


def _small(**kw):
    return FFConvLSTM(87, ff_hidden_dim=64, conv_hidden_dim=32, lstm_hidden_dim=16, out_dim=32, in_ph_start_idx=3, in_ph_end_idx=50,
                      embed_dim=32, **kw)


def test_default_keeps_refusing_with_a_hint():
    with pytest.raises(RuntimeError, match="no backward kernels.*backward_kernels=True"):
        _small()(torch.zeros(1, 8, 87))


def test_opt_in_refuses_what_it_does_not_build_before_launch():
    x = torch.zeros(1, 8, 87)
    with pytest.raises(RuntimeError, match="CUDA"):                        # CPU tensors
        _small(backward_kernels=True)(x)
    with pytest.raises(RuntimeError, match="CUDA"):
        _small(backward_kernels=True)(x.clone().requires_grad_(True))
    mdn = FFConvLSTM(16, 32, 16, 8, 4, use_mdn=True, backward_kernels=True)
    with pytest.raises(RuntimeError, match="MDN head"):
        mdn(torch.zeros(1, 8, 16))
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):        # no grad: the plain training forward, still CUDA
        mdn(torch.zeros(1, 8, 16))
    drop = FFConvLSTM(16, 32, 16, 8, 4, dropout=0.1, backward_kernels=True)
    with pytest.raises(RuntimeError, match="dropout = 0 only"):
        drop(torch.zeros(1, 8, 16))


def test_eval_mode_with_grad_takes_the_inference_path():
    m = _small(backward_kernels=True).eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 8, 87))
    assert not m._records_grad(torch.zeros(1, 8, 87), None)
    m.train()
    assert m._records_grad(torch.zeros(1, 8, 87), None)
    with torch.no_grad():
        assert not m._records_grad(torch.zeros(1, 8, 87), None)
    for p in m.parameters():
        p.requires_grad_(False)
    assert not m._records_grad(torch.zeros(1, 8, 87), None)
    assert m._records_grad(torch.zeros(1, 8, 87), torch.zeros(1, 8, 32, requires_grad=True))
