"""WaveNet training on the device (wavenet/training.py): gradients of WaveNet.forward against float64 autograd through
the oracle (oracle.wavenet_forward is built from differentiable torch ops, weight norm included), the forward against
the eval path bit for bit, the weight packs against torch's weight-norm fold bit for bit, ResSkipBlock on its own,
determinism, and a short SGD run against the same run driven by oracle gradients."""
import pytest
import torch
import torch.nn.functional as F

from ensemble_svs_with_interactions_b200 import _lib
from ensemble_svs_with_interactions_b200.wavenet import WaveNet
from oracle import svs_oracle as O
from tests.golden_util import Golden

pytestmark = pytest.mark.gpu
DEV = "cuda"
# measured on a B200 over every config below: worst rel-L2 1.2e-6, worst max-abs / max(1, |ref|) 2.0e-6 (DESIGN.md §5);
# fp32 sums over up to 2 x 1100 frames, against float64
REL_L2 = 1e-5
MAX_ABS = 1e-5


def _model(name):
    """(module on the GPU in training mode, config) for 'golden' (6 layers in 2 stacks), 'test_shape' (2 layers, in
    300, out 206), 'default' (the reference default, seeded as in test_gpu_wavenet_ar) and 'k2' (kernel size 2, channel
    counts that are not multiples of 4: R 6, S 10, G / 2 = 10)."""
    if name == "default":
        torch.manual_seed(1234)
        cfg = dict(in_dim=334, out_dim=206, layers=10, stacks=1)
        m = WaveNet(**cfg)
        with torch.no_grad():
            m.last_conv_layers[3].weight_g.mul_(10.0)
    elif name == "k2":
        torch.manual_seed(77)
        cfg = dict(in_dim=20, out_dim=30, layers=5, stacks=1, residual_channels=6, gate_channels=20, skip_out_channels=10,
                   kernel_size=2)
        m = WaveNet(**cfg)
    else:
        g = Golden({"golden": "wavenet_incremental", "test_shape": "wavenet_test_shape"}[name])
        cfg = dict(g.cfg)
        m = WaveNet(**cfg)
        m.load_state_dict(g.sd, strict=True)
    cfg = dict(cfg, stacks=cfg.get("stacks", 1))
    return m.to(DEV).train(), cfg


def _inputs(cfg, B, T, seed):
    gen = torch.Generator().manual_seed(seed)
    c = torch.randn(B, T, cfg["in_dim"], generator=gen)
    x = torch.randn(B, T, cfg["out_dim"], generator=gen)
    gup = torch.randn(B, T, cfg["out_dim"], generator=gen)
    return c, x, gup


def _oracle_grads(m, cfg, c, x, gup):
    sd = {k: v.detach().cpu().double().requires_grad_(True) for k, v in m.named_parameters()}
    c64 = c.double().requires_grad_(True)
    x64 = x.double().requires_grad_(True)
    out = O.wavenet_forward(sd, c64, x64, cfg["layers"], cfg["stacks"])
    (out * gup.double()).sum().backward()
    # the last block's conv1x1_out feeds nothing (only the skips reach the output): no gradient, i.e. zeros
    return {k: torch.zeros_like(v) if v.grad is None else v.grad for k, v in sd.items()}, c64.grad, x64.grad


def _device_grads(m, c, x, gup):
    m.zero_grad(set_to_none=True)
    cd = c.to(DEV).requires_grad_(True)
    xd = x.to(DEV).requires_grad_(True)
    out = m(cd, xd)
    assert out.grad_fn is not None
    out.backward(gup.to(DEV))
    return {k: v.grad.detach().cpu().double() for k, v in m.named_parameters()}, cd.grad.cpu().double(), xd.grad.cpu().double()


def _compare(name, got, ref, worst):
    assert got.shape == ref.shape, name
    nref = ref.norm().item()
    if nref == 0:
        assert torch.count_nonzero(got) == 0, name
        return
    rel = (got - ref).norm().item() / nref
    mab = (got - ref).abs().max().item() / max(1.0, ref.abs().max().item())
    worst["rel"] = max(worst["rel"], (rel, name))
    worst["abs"] = max(worst["abs"], (mab, name))
    assert rel <= REL_L2, f"{name}: rel-L2 {rel:.2e}"
    assert mab <= MAX_ABS, f"{name}: max-abs / max(1, |ref|) {mab:.2e}"


def _check(m, cfg, B, T, seed):
    c, x, gup = _inputs(cfg, B, T, seed)
    ref, rc, rx = _oracle_grads(m, cfg, c, x, gup)
    got, gc, gx = _device_grads(m, c, x, gup)
    assert set(got) == set(ref)
    worst = {"rel": (0.0, ""), "abs": (0.0, "")}
    for k in ref:
        _compare(k, got[k], ref[k], worst)
    _compare("c", gc, rc, worst)
    _compare("x", gx, rx, worst)
    print(f"\n  B={B} T={T}: worst rel-L2 {worst['rel'][0]:.2e} ({worst['rel'][1]}), worst max-abs / max(1, |ref|) "
          f"{worst['abs'][0]:.2e} ({worst['abs'][1]})")


@pytest.mark.parametrize("T", [200, 1100])
@pytest.mark.parametrize("name", ["golden", "test_shape", "default", "k2"])
def test_gradients_match_float64_autograd(name, T):
    m, cfg = _model(name)
    _check(m, cfg, 2, T, seed=T + len(name))


@pytest.mark.parametrize("name", ["golden", "k2"])
def test_gradients_without_weight_norm(name):
    m, cfg = _model(name)
    m.remove_weight_norm_()
    assert not any(k.endswith("weight_g") for k, _ in m.named_parameters())
    _check(m, cfg, 2, 1100, seed=3)


@pytest.mark.parametrize("name", ["golden", "test_shape", "default", "k2"])
def test_training_forward_equals_eval_forward(name):
    m, cfg = _model(name)
    c, x, _ = _inputs(cfg, 3, 333, seed=1)
    c, x = c.to(DEV), x.to(DEV)
    y_train = m(c, x)
    assert y_train.grad_fn is not None
    m.eval()
    y_eval = m(c, x)
    assert y_eval.grad_fn is None and not y_eval.requires_grad          # eval mode with grad enabled: today's path
    assert torch.equal(y_train.detach(), y_eval)


def _fold(mod):
    """torch's weight-norm fold on CUDA; the weight itself after remove_weight_norm_()."""
    if hasattr(mod, "weight_g"):
        return torch._weight_norm(mod.weight_v, mod.weight_g, 0).detach()
    return mod.weight.detach()


@pytest.mark.parametrize("weight_norm", [True, False])
@pytest.mark.parametrize("name", ["golden", "test_shape", "default", "k2"])
def test_packs_equal_torch_weight_norm(name, weight_norm):
    """The one fold of the library gives torch._weight_norm's bits, in the forward's pack and in the sampler's."""
    m, _ = _model(name)
    if not weight_norm:
        m.remove_weight_norm_()
    blocks, l1, l3 = m.main_conv_layers, m.last_conv_layers[1], m.last_conv_layers[3]
    _, _, pk, _ = m._packed()
    for l, f in enumerate(blocks):
        k, R = f.kernel_size, f.conv.in_channels
        w1t = torch.cat([_fold(f.conv).permute(2, 1, 0).reshape(k * R, -1), _fold(f.conv1x1c)[:, :, 0].t()])
        w2t = torch.cat([_fold(f.conv1x1_skip), _fold(f.conv1x1_out)])[:, :, 0].t()
        assert torch.equal(pk["w1t"][l], w1t) and torch.equal(pk["w2t"][l], w2t), l
    for key, mod in (("first", m.first_conv), ("last1", l1), ("last3", l3)):
        assert torch.equal(pk[key], _fold(mod)), key
    # the sampler's ArLayout (include/svsk.h, svsk_wavenet_ar_f32): WfT, bf; per layer Wg, bg, Wso, bso; W3, b3, W4, b4
    conf = m._ar_config()
    assert conf is not None
    wpack, wcond = m._ar_packed(conf)
    bias = lambda mod: mod.bias.detach() if mod.bias is not None else torch.zeros(mod.out_channels, device=DEV)
    parts = [_fold(m.first_conv)[:, :, 0].t(), bias(m.first_conv)]
    for f in blocks:
        G = f.conv.out_channels
        parts += [_fold(f.conv).permute(0, 2, 1).reshape(G, -1), bias(f.conv),
                  torch.cat([_fold(f.conv1x1_skip), _fold(f.conv1x1_out)]), torch.cat([bias(f.conv1x1_skip), bias(f.conv1x1_out)])]
    parts += [_fold(l1), bias(l1), _fold(l3), bias(l3)]
    assert torch.equal(wpack, torch.cat([p.flatten() for p in parts]))
    assert torch.equal(wcond, torch.cat([_fold(f.conv1x1c) for f in blocks]))


@pytest.mark.parametrize("weight_norm", [True, False])
@pytest.mark.parametrize("name", ["golden", "test_shape", "default", "k2"])
def test_res_skip_block_standalone_matches_oracle(name, weight_norm):
    """ResSkipBlock.forward on its own (WaveNet runs its blocks from the shared pack) against oracle.wavenet_block."""
    m, cfg = _model(name)
    if not weight_norm:
        m.remove_weight_norm_()
    sd = {k: v.detach().cpu().double() for k, v in m.state_dict().items()}
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(2, m.first_conv.out_channels, 300, generator=gen)
    c = torch.randn(2, cfg["in_dim"], 300, generator=gen)
    worst = {"rel": (0.0, ""), "abs": (0.0, "")}
    for i, f in enumerate(m.main_conv_layers):
        xo, s = f(x.to(DEV), c.to(DEV))
        rx, rs = O.wavenet_block(sd, i, x.double(), c.double(), f.dilation)
        _compare(f"block {i} x_out", xo.cpu().double(), rx, worst)
        _compare(f"block {i} skips", s.cpu().double(), rs, worst)


def test_no_grad_in_training_mode_takes_the_inference_path():
    m, cfg = _model("golden")
    c, x, _ = _inputs(cfg, 2, 50, seed=2)
    with torch.no_grad():
        y = m(c.to(DEV), x.to(DEV))
    assert y.grad_fn is None
    for p in m.parameters():
        p.requires_grad_(False)
    y = m(c.to(DEV), x.to(DEV))                                           # nothing requires grad
    assert y.grad_fn is None


def test_gradients_are_bit_reproducible():
    m, cfg = _model("default")
    c, x, gup = _inputs(cfg, 4, 1000, seed=9)
    a = _device_grads(m, c, x, gup)
    b = _device_grads(m, c, x, gup)
    for k in a[0]:
        assert torch.equal(a[0][k], b[0][k]), k
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


def test_only_requested_input_gradients_and_launch_count():
    m, cfg = _model("golden")
    c, x, gup = _inputs(cfg, 2, 64, seed=4)
    n0 = _lib.launch_count
    out = m(c.to(DEV), x.to(DEV))
    out.backward(gup.to(DEV))
    L = cfg["layers"]
    # forward: pack + first conv + L blocks + 2 head convs; backward: 2 convs + 2 masks + L + 1 dgrad + wgrad (1 or 2)
    # + weight-norm gradient; no dc / dx convs since neither c nor x requires grad
    assert _lib.launch_count - n0 in (3 + L + 1 + 4 + L + 1 + 1 + 1, 3 + L + 1 + 4 + L + 1 + 2 + 1)
    assert all(p.grad is not None for p in m.parameters())


def test_sgd_trajectory_tracks_oracle_gradients():
    m, cfg = _model("test_shape")
    B, T, lr = 2, 200, 0.05
    gen = torch.Generator().manual_seed(21)
    c = torch.randn(B, T, cfg["in_dim"], generator=gen)
    x = torch.randn(B, T, cfg["out_dim"], generator=gen)
    target = torch.randint(0, cfg["out_dim"], (B, T), generator=gen)
    ref = {k: v.detach().cpu().double().clone() for k, v in m.named_parameters()}
    cd, xd, td = c.to(DEV), x.to(DEV), target.to(DEV)
    losses = []
    for _ in range(10):
        m.zero_grad(set_to_none=True)
        loss = F.cross_entropy(m(cd, xd).reshape(-1, cfg["out_dim"]), td.reshape(-1))
        loss.backward()
        losses.append(loss.item())
        with torch.no_grad():
            for p in m.parameters():
                p.sub_(lr * p.grad)
        sd = {k: v.requires_grad_(True) for k, v in ref.items()}
        out = O.wavenet_forward(sd, c.double(), x.double(), cfg["layers"], cfg["stacks"])
        F.cross_entropy(out.reshape(-1, cfg["out_dim"]), target.reshape(-1)).backward()
        ref = {k: (v if v.grad is None else v - lr * v.grad).detach() for k, v in sd.items()}
    print(f"\n  loss {losses[0]:.4f} -> {losses[-1]:.4f}")
    assert losses[-1] < losses[0]
    worst = 0.0
    for k, p in m.named_parameters():
        r = ref[k]
        rel = (p.detach().cpu().double() - r).norm().item() / max(r.norm().item(), 1e-30)
        worst = max(worst, rel)
        assert rel <= 1e-4, f"{k}: {rel:.2e}"
    print(f"  worst parameter deviation after 10 steps: {worst:.2e} relative")
