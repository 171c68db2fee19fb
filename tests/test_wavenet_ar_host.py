"""CPU-only: shape coverage and argument checks of the device WaveNet sampler (svsk_wavenet_ar_*), all decided before
any launch."""
import ctypes as C

import pytest

from ensemble_svs_with_interactions_b200 import _lib, ops

# (out_dim, R, G, S, layers, stacks, ksize)
REFERENCE_DEFAULT = (206, 64, 128, 64, 10, 1, 3)
REFERENCE_TEST_SHAPE = (206, 64, 128, 64, 2, 1, 3)
GOLDEN = (12, 16, 32, 16, 6, 2, 3)


@pytest.mark.parametrize("cfg", [REFERENCE_DEFAULT, REFERENCE_TEST_SHAPE, GOLDEN])
def test_reference_configs_supported(cfg):
    assert ops.wavenet_ar_supported(*cfg)
    npack, nhist = ops.wavenet_ar_sizes(*cfg)
    out_dim, R, G, S, L, stacks, k = cfg
    per_layer = G * k * R + G + (S + R) * (G // 2) + S + R
    assert npack == out_dim * R + R + L * per_layer + S * S + S + out_dim * S + out_dim
    assert nhist == sum(((k - 1) * 2 ** (l % (L // stacks)) + 1) * R for l in range(L))


@pytest.mark.parametrize("cfg", [(300, 64, 128, 64, 10, 1, 3),     # out_dim > 256
                                 (206, 64, 256, 64, 10, 1, 3),     # G / 2 > 64
                                 (206, 128, 128, 64, 10, 1, 3),    # k R > 256
                                 (206, 64, 128, 64, 10, 3, 3)])    # layers not a multiple of stacks
def test_unsupported_configs(cfg):
    assert not ops.wavenet_ar_supported(*cfg)
    with pytest.raises(RuntimeError, match="unsupported"):
        ops.wavenet_ar_sizes(*cfg)


def test_argument_errors_before_launch():
    l = _lib.lib()
    assert l.svsk_wavenet_ar_f32(None, None) == -1
    assert b"null" in l.svsk_last_error()
    assert l.svsk_wavenet_ar_pack_f32(None, None, None, None) == -1
    p = _lib.WavenetArParams()
    p.wpack = p.cproj = p.u = p.y = p.hist = 256           # never dereferenced: the checks come first
    p.B, p.T, p.steps = 2, 10, 11
    p.out_dim, p.R, p.G, p.S, p.layers, p.stacks, p.ksize = GOLDEN
    assert l.svsk_wavenet_ar_f32(C.byref(p), None) == -1
    assert b"exceeds" in l.svsk_last_error()
    p.steps, p.out_dim = 10, 300
    assert l.svsk_wavenet_ar_f32(C.byref(p), None) == -1
    assert b"unsupported" in l.svsk_last_error()
