"""WaveNet.inference on the device (svsk_wavenet_ar_f32): the whole sampled chain against the oracle's parallel forward.

Causality makes the teacher-forced parallel forward on the shifted samples, oracle.wavenet_forward(sd, c, shift(y)),
equal the logits of every autoregressive step, so one oracle call checks the chain.  Each draw is then checked against
the inverse CDF of the float64 softmax of the kernel's own logits at the injected uniform.
"""
import numpy as np
import pytest
import torch
from scipy import stats

from ensemble_svs_with_interactions_b200 import _lib, ops
from ensemble_svs_with_interactions_b200.wavenet import WaveNet
from oracle import svs_oracle as O
from tests.golden_util import Golden

pytestmark = pytest.mark.gpu
DEV = "cuda"
CDF_EPS = 1e-6


def _model(name):
    """(module on the GPU, float64 state dict, config) for 'golden' (R 16, G 32, S 16, out 12, 6 layers in 2 stacks),
    'test_shape' (in 300, out 206, 2 layers) or 'default' (the reference default, seeded, last conv gain x 10 so that
    the softmax is neither flat nor one-hot)."""
    if name == "default":
        torch.manual_seed(1234)
        cfg = dict(in_dim=334, out_dim=206, layers=10, stacks=1)
        m = WaveNet(**cfg)
        with torch.no_grad():
            m.last_conv_layers[3].weight_g.mul_(10.0)
        sd = m.state_dict()
    else:
        g = Golden({"golden": "wavenet_incremental", "test_shape": "wavenet_test_shape"}[name])
        cfg, sd = g.cfg, g.sd
        m = WaveNet(**cfg)
        m.load_state_dict(sd, strict=True)
    cfg = dict(cfg, stacks=cfg.get("stacks", 1))
    return m.to(DEV).eval(), {k: v.detach().cpu().double() for k, v in sd.items()}, cfg


def _shift(y):
    s = torch.zeros_like(y)
    s[:, 1:] = y[:, :-1]
    return s


def _check_chain(m, sd, cfg, B, steps, seed=0):
    gen = torch.Generator().manual_seed(seed)
    c = torch.randn(B, steps, cfg["in_dim"], generator=gen)
    u = torch.rand(B, steps, generator=gen)
    lg = torch.empty(B, steps, cfg["out_dim"], device=DEV)
    y = m.inference(c.to(DEV), num_time_steps=steps, u=u.to(DEV), logits=lg)
    assert m.first_conv.input_buffer is None
    y, lg = y.cpu(), lg.cpu()
    assert y.shape == (B, steps, cfg["out_dim"]) and y.dtype == torch.float32
    assert torch.equal(y.sum(-1), torch.ones(B, steps)) and torch.equal(y, (y == 1).float())
    # the whole chain: logits of step t are the network's output on the samples drawn before t
    ref = O.wavenet_forward(sd, c.double(), _shift(y).double(), cfg["layers"], cfg["stacks"])
    err = ((lg.double() - ref).abs() / ref.abs().clamp_min(1.0)).max().item()
    # the draw: inverse CDF of the float64 softmax of the kernel's logits
    p = torch.softmax(lg.double(), -1)
    cdf = torch.cumsum(p, -1)
    u64 = u.double()
    want = (u64[..., None] >= cdf).sum(-1)                      # smallest k with u < P_k
    last = (torch.arange(p.shape[-1]) * (p > 0)).argmax(-1)     # largest k with p_k > 0
    want = torch.where(want >= p.shape[-1], last, want)
    near = ((u64[..., None] - cdf).abs() < CDF_EPS).any(-1)
    got = y.argmax(-1)
    bad = (got != want) & ~near
    print(f"\n  B={B} steps={steps}: max |logit err| / max(1, |ref|) = {err:.2e}; "
          f"{int(near.sum())} of {B * steps} draws within {CDF_EPS:g} of a CDF boundary; {len(set(got.flatten().tolist()))} classes drawn")
    assert err <= 1e-5
    assert not bad.any(), f"{int(bad.sum())} draws differ from the inverse CDF"


@pytest.mark.parametrize("steps", [1, 37, 300])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("name", ["golden", "test_shape", "default"])
def test_chain_parity(name, B, steps):
    m, sd, cfg = _model(name)
    _check_chain(m, sd, cfg, B, steps, seed=B * 1000 + steps)


def test_long_sequence_wraps_the_tap_history():
    """2000 steps > twice the largest dilation (512): every ring buffer wraps."""
    m, sd, cfg = _model("default")
    _check_chain(m, sd, cfg, 2, 2000, seed=7)


def test_reproducible():
    m, _, cfg = _model("default")
    c = torch.randn(3, 120, cfg["in_dim"], device=DEV)
    u = torch.rand(3, 120, device=DEV)
    runs = []
    for _ in range(2):
        lg = torch.empty(3, 120, cfg["out_dim"], device=DEV)
        runs.append((m.inference(c, 120, u=u, logits=lg), lg))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    torch.manual_seed(5)
    a = m.inference(c, 120)
    torch.manual_seed(5)
    b = m.inference(c, 120)
    assert torch.equal(a, b)


def test_first_step_distribution():
    """512 tracks with the same conditioning share the logits of step 0; their draws (u from the module) follow the
    softmax of those logits."""
    m, _, cfg = _model("golden")
    B = 512
    c = torch.randn(1, 4, cfg["in_dim"], device=DEV).expand(B, -1, -1)
    lg = torch.empty(B, 4, cfg["out_dim"], device=DEV)
    torch.manual_seed(11)
    y = m.inference(c, 4, logits=lg)
    assert torch.equal(lg[:, 0], lg[:1, 0].expand(B, -1))
    p = torch.softmax(lg[0, 0].double(), -1).cpu().numpy()
    counts = y[:, 0].sum(0).double().cpu().numpy()
    exp = p * B
    keep = exp >= 5                                             # pool the rare classes into one cell
    f_obs = np.append(counts[keep], counts[~keep].sum())
    f_exp = np.append(exp[keep], exp[~keep].sum())
    if f_exp[-1] == 0:
        f_obs, f_exp = f_obs[:-1], f_exp[:-1]
    res = stats.chisquare(f_obs, f_exp)
    print(f"\n  chi-square over {len(f_obs)} cells: statistic {res.statistic:.2f}, p = {res.pvalue:.3f}")
    assert len(f_obs) >= 3 and res.pvalue > 1e-3


def test_configs_of_the_reference_are_supported():
    for name in ("golden", "test_shape", "default"):
        m, _, _ = _model(name)
        assert m._ar_config() is not None, name


def test_unsupported_shape_and_cpu_run_the_host_loop():
    torch.manual_seed(0)
    big = WaveNet(in_dim=8, out_dim=300, layers=2, residual_channels=8, gate_channels=16, skip_out_channels=8).eval()
    assert not ops.wavenet_ar_supported(300, 8, 16, 8, 2, 1, 3)
    m, _, cfg = _model("golden")
    for net, c in ((big.to(DEV), torch.randn(2, 6, 8, device=DEV)), (m.cpu(), torch.randn(2, 6, cfg["in_dim"]))):
        n0 = _lib.launch_count
        y = net.inference(c, num_time_steps=6, tqdm=None)
        assert _lib.launch_count == n0
        assert y.shape == (2, 6, net.out_dim) and torch.equal(y.sum(-1), torch.ones(2, 6, device=y.device))
        with pytest.raises(ValueError, match="device sampler"):
            net.inference(c, num_time_steps=6, u=torch.rand(2, 6, device=c.device))


def test_bad_arguments_are_rejected_before_launch():
    m, _, cfg = _model("golden")
    conf = m._ar_config()
    out_dim, R, G, S, layers, stacks, k = conf
    wpack, wcond = m._ar_packed(conf)
    B, T = 2, 10
    cproj = ops.conv1d_f32(torch.randn(B, cfg["in_dim"], T, device=DEV), wcond)
    u = torch.rand(B, T, device=DEV)
    kw = dict(out_dim=out_dim, R=R, G=G, S=S, layers=layers, stacks=stacks, ksize=k)
    n0 = _lib.launch_count
    bad = [
        dict(u=torch.rand(B, T + 1, device=DEV)),                       # steps > T
        dict(u=u[0]),                                                   # u not [B, steps]
        dict(u=u.double()),                                             # dtype
        dict(u=u.cpu()),                                                # host tensor
        dict(cproj=cproj[:, 1:].contiguous()),                          # layers * G rows
        dict(cproj=cproj[:1]),                                          # batch
        dict(cproj=cproj.to(torch.float16)),                            # dtype
        dict(wpack=wpack[1:]),                                          # packed size
        dict(logits=torch.empty(B, T, out_dim + 1, device=DEV)),        # logits shape
        dict(logits=torch.empty(B, T, out_dim, device=DEV, dtype=torch.float64)),
    ]
    for change in bad:
        args = dict(wpack=wpack, cproj=cproj, u=u, logits=None)
        args.update(change)
        with pytest.raises((ValueError, RuntimeError)):
            ops.wavenet_ar_f32(args["wpack"], args["cproj"], args["u"], logits=args["logits"], **kw)
    assert _lib.launch_count == n0
    with pytest.raises(RuntimeError, match="unsupported"):
        ops.wavenet_ar_f32(wpack, cproj, u, **dict(kw, out_dim=300))
    y = ops.wavenet_ar_f32(wpack, cproj, u, **kw)
    assert _lib.launch_count == n0 + 1 and torch.equal(y.sum(-1), torch.ones(B, T, device=DEV))
