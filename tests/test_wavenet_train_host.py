"""CPU-only: argument checks of the WaveNet training entries (svsk_wavenet_*train*, dgrad, wgrad, wnorm_grad,
svsk_relu_mask_f32), all decided before any launch, the pack / gradient layouts, and the CPU error of the training path."""
import ctypes as C

import pytest
import torch

from ensemble_svs_with_interactions_b200 import _lib, ops
from ensemble_svs_with_interactions_b200.wavenet import WaveNet

# (out_dim, R, G, S, cin, layers, ksize)
REFERENCE_DEFAULT = (206, 64, 128, 64, 334, 10, 3)
GOLDEN = (12, 16, 32, 16, 10, 6, 3)
ODD = (30, 6, 20, 10, 20, 5, 2)            # R and G / 2 not multiples of 4: padded columns in the pack


def test_null_params_are_rejected():
    l = _lib.lib()
    assert l.svsk_wavenet_block_train_f32(None, None) == -1
    assert b"null" in l.svsk_last_error()
    assert l.svsk_wavenet_dgrad_f32(None, None) == -1
    assert b"null" in l.svsk_last_error()
    assert l.svsk_wavenet_wgrad_f32(None, None) == -1
    assert b"null" in l.svsk_last_error()
    assert l.svsk_wavenet_train_pack_f32(None, None, None) == -1
    assert l.svsk_wavenet_wnorm_grad_f32(None, None, None, None) == -1
    assert l.svsk_relu_mask_f32(None, None, None, 4, None) == -1
    p = _lib.WavenetBlockTrainParams()
    p.blk.x = p.blk.c = p.blk.w1t = p.blk.w2t = p.blk.b2 = p.blk.x_out = p.blk.skips = 256
    p.blk.B, p.blk.T, p.blk.R, p.blk.G, p.blk.S, p.blk.Cc, p.blk.ksize, p.blk.dilation = 1, 8, 16, 32, 16, 10, 3, 1
    assert l.svsk_wavenet_block_train_f32(C.byref(p), None) == -1            # y missing
    assert b"null tensor y" in l.svsk_last_error()


def test_bad_sizes_are_rejected():
    l = _lib.lib()
    a, b = C.c_longlong(), C.c_longlong()
    for bad in [(12, 16, 30, 16, 10, 6, 3),        # G not a multiple of 4
                (12, 15, 32, 16, 10, 6, 3),        # S + R not a multiple of 4
                (12, 16, 512, 16, 10, 6, 3),       # G > 256
                (12, 16, 32, 16, 10, 0, 3),        # no layers
                (12, 16, 32, 16, 10, 6, 0)]:       # kernel size
        assert l.svsk_wavenet_train_sizes(*bad, C.byref(a), C.byref(b)) == -1
    with pytest.raises(RuntimeError, match="multiples of 4"):
        ops.wavenet_train_sizes(12, 15, 32, 16, 10, 6, 3)
    d = _lib.WavenetDgradParams()
    d.g_out = d.dS = d.dy_in = d.wT = 256
    d.B, d.T, d.R, d.G, d.S, d.ksize, d.dilation, d.dy_bstride = 2, 10, 16, 30, 16, 3, 1, 300
    assert l.svsk_wavenet_dgrad_f32(C.byref(d), None) == -1
    assert b"multiples of 4" in l.svsk_last_error()
    d.G, d.dy_bstride = 32, 100                                                 # batch stride below G T
    assert l.svsk_wavenet_dgrad_f32(C.byref(d), None) == -1
    assert b"dy_bstride" in l.svsk_last_error()
    w = _lib.WavenetWgradParams()
    for n in ("x_in", "c", "xs", "ys", "gs", "dy", "dS", "skips", "h1", "dh1", "glog", "dilations", "dW"):
        setattr(w, n, 256)
    w.B, w.T, w.out_dim, w.R, w.G, w.S, w.cin, w.layers, w.ksize, w.splits = 2, 10, 12, 16, 32, 16, 10, 6, 3, 2
    assert l.svsk_wavenet_wgrad_f32(C.byref(w), None) == -1                     # splits > 1 without workspace
    assert b"workspace" in l.svsk_last_error()
    assert l.svsk_relu_mask_f32(256, 256, 256, 0, None) == -1


@pytest.mark.parametrize("cfg", [REFERENCE_DEFAULT, GOLDEN, ODD])
def test_layouts_agree_with_the_library(cfg):
    pack, grad = ops.wavenet_train_layout(*cfg)
    out_dim, R, G, S, cin, L, k = cfg
    assert grad["conv"][1] == (L, G, R, k) and grad["last3_b"][1] == (out_dim,)
    assert pack["wT"][1] == (L, k * G, (R + 3) // 4 * 4) and pack["wB"][1] == (L, R + S, (G // 2 + 3) // 4 * 4)


def test_wrappers_reject_mismatched_shapes():
    out_dim, R, G, S, cin, L, k = GOLDEN
    G2 = G // 2
    w = dict(first_v=torch.zeros(R, out_dim, 1), conv_v=torch.zeros(L, G, R, k), cond_v=torch.zeros(L, G, cin, 1),
             skip_v=torch.zeros(L, S, G2, 1), out_v=torch.zeros(L, R, G2, 1), last1_v=torch.zeros(S, S, 1),
             last3_v=torch.zeros(out_dim, S, 1))
    dims = dict(out_dim=out_dim, R=R, G=G, S=S, cin=cin, layers=L, ksize=k)
    with pytest.raises(ValueError, match="conv_v"):
        ops.wavenet_train_pack_f32(dict(w, conv_v=torch.zeros(L, G, R, k + 1)), **dims)
    with pytest.raises(ValueError, match="gains"):
        ops.wavenet_train_pack_f32(dict(w, conv_g=torch.zeros(L, G - 1, 1, 1)), **dims)
    with pytest.raises(ValueError, match="dW"):
        ops.wavenet_wnorm_grad_f32(w, torch.zeros(5), **dims)
    with pytest.raises(ValueError, match="relu_mask"):
        ops.relu_mask_f32(torch.zeros(4), torch.zeros(5))
    B, T = 2, 10
    with pytest.raises(ValueError, match="dS"):
        ops.wavenet_dgrad_f32(dy_in=None, wT=None, g_next=None, g_out=torch.zeros(B, R, T), dS=torch.zeros(B, S, T + 1),
                              y_prev=torch.zeros(B, G, T), wB=torch.zeros(R + S, G2), dy_out=torch.zeros(B, G, T), ksize=k,
                              dilation=1)
    with pytest.raises(ValueError, match="wB"):
        ops.wavenet_dgrad_f32(dy_in=None, wT=None, g_next=None, g_out=torch.zeros(B, R, T), dS=torch.zeros(B, S, T),
                              y_prev=torch.zeros(B, G, T), wB=torch.zeros(R + S, G2 + 4), dy_out=torch.zeros(B, G, T), ksize=k,
                              dilation=1)
    t = dict(x_in=torch.zeros(B, out_dim, T), c=torch.zeros(B, cin, T), xs=torch.zeros(L, B, R, T), ys=torch.zeros(L, B, G, T),
             gs=torch.zeros(L + 1, B, R, T), dy=torch.zeros(B, L, G, T), dS=torch.zeros(B, S, T), skips=torch.zeros(B, S, T),
             h1=torch.zeros(B, S, T), dh1=torch.zeros(B, S, T), glog=torch.zeros(B, out_dim, T),
             dilations=torch.ones(L, dtype=torch.int32))
    with pytest.raises(ValueError, match="gs"):
        ops.wavenet_wgrad_f32(**dict(t, gs=torch.zeros(L, B, R, T)), ksize=k)
    with pytest.raises(ValueError, match="dy"):
        ops.wavenet_wgrad_f32(**dict(t, dy=torch.zeros(L, B, G, T)), ksize=k)


def test_cpu_module_in_training_mode_raises():
    torch.manual_seed(0)
    m = WaveNet(in_dim=10, out_dim=12, layers=2, residual_channels=16, gate_channels=32, skip_out_channels=16).train()
    c, x = torch.randn(2, 8, 10), torch.randn(2, 8, 12)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(c, x)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(c.requires_grad_(True), x)
    m.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m(c, x)
