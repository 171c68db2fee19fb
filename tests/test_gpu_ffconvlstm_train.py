"""FFConvLSTM training on the device (backward_kernels=True): each new kernel against float64 on the same inputs, every
gradient of the module against float64 autograd through oracle.ffconvlstm_forward(train=True), and the behaviour of the
opt-in path (bit-identical forward, reproducible backward, SGD, no graph in eval / no_grad, end-to-end in
GaussianDiffusion)."""
import copy

import pytest
import torch
import torch.nn.functional as F

from ensemble_svs_with_interactions_b200 import encoder_training, ops
from ensemble_svs_with_interactions_b200.model import FFConvLSTM, MultiSpeakerFFConvLSTM
from oracle import svs_oracle as O
from tests.golden_util import Golden

pytestmark = pytest.mark.gpu
DEV = "cuda"
f64 = torch.float64


def _check(name, got, ref, errs=None):
    """max-abs <= 2e-4 max(1, max|ref|); rel-L2 <= 1e-4 where ||ref|| >= 1e-3."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    ma = (got - ref).abs().max().item() / max(1.0, ref.abs().max().item())
    nr = ref.norm().item()
    rl = (got - ref).norm().item() / nr if nr >= 1e-3 else 0.0
    if errs is not None:
        errs[name] = (ma, rl)
    assert ma <= 2e-4, f"{name}: max-abs {ma:.3g}"
    assert rl <= 1e-4, f"{name}: rel-L2 {rl:.3g}"


# ---------------------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("H,T,lens", [(16, 50, [50, 4, 31]), (32, 50, [17, 50, 4]), (64, 60, [4, 60, 33]),
                                      (128, 50, [29, 4, 50]), (256, 40, [40, 4, 23]), (128, 1000, [1000, 613])])
def test_lstm_backward_matches_float64(H, T, lens):
    g = torch.Generator().manual_seed(H + T)
    B = len(lens)
    pre = torch.randn(B, 8 * H, T, generator=g)
    w_hh = torch.randn(2, 4 * H, H, generator=g) / H ** 0.5
    dH = torch.randn(B, 2 * H, T, generator=g)
    lens_dev = torch.tensor(lens, dtype=torch.int32, device=DEV)
    pre_d, w_d = pre.to(DEV), w_hh.to(DEV)
    h = torch.empty(B, 2 * H, T, device=DEV)
    gates, cell = torch.empty_like(pre_d), torch.empty(B, 2 * H, T, device=DEV)
    ops.lstm_train_f32(pre_d, w_d, lens_dev, H, h_f32=h, gates=gates, cell=cell)
    h_inf = torch.empty_like(h)
    ops.lstm_f32(pre_d, w_d, lens_dev, H, pre_layout="nct", h_f32=h_inf)
    assert torch.equal(h, h_inf)                                   # the kept-state variant computes the same bits
    dpre = ops.lstm_bwd_f32(dH.to(DEV), gates, cell, w_d, lens_dev, H)
    pr = pre.double().requires_grad_(True)
    loss = 0
    for b in range(B):
        for d in range(2):
            out = O.lstm_direction(pr[b, d * 4 * H:(d + 1) * 4 * H].t(), w_hh[d].double(), lens[b], d == 1)
            loss = loss + (out * dH[b, d * H:(d + 1) * H].t().double()).sum()
    loss.backward()
    _check("dpre", dpre, pr.grad)
    for b in range(B):
        assert torch.count_nonzero(dpre[b, :, lens[b]:]) == 0


@pytest.mark.parametrize("ksize,origin,pad", [(1, 1, ops.PAD_ZEROS), (1, 0, ops.PAD_ZEROS), (1, -1, ops.PAD_ZEROS),
                                              (7, 3, ops.PAD_REFLECT)])
def test_wgrad_matches_float64(ksize, origin, pad):
    g = torch.Generator().manual_seed(ksize * 10 + origin)
    B, N, K, T = 3, 70, 45, 203
    dy, x = torch.randn(B, N + 5, T, generator=g), torch.randn(B, K, T, generator=g)
    dw, db = ops.wgrad_f32(dy.to(DEV)[:, 2:2 + N], x.to(DEV), ksize=ksize, origin=origin, pad_mode=pad)
    dyd, xd = dy[:, 2:2 + N].double(), x.double()
    cols = []
    for j in range(ksize):
        u = torch.arange(T) + j - origin
        if pad == ops.PAD_REFLECT:
            u = torch.where(u < 0, -u, u)
            u = torch.where(u >= T, 2 * (T - 1) - u, u)
        valid = (u >= 0) & (u < T)
        xs = xd[:, :, u.clamp(0, T - 1)] * valid.double()
        cols.append(torch.einsum("bnt,bkt->nk", dyd, xs))
    ref = torch.stack(cols, -1)
    _check("dw", dw, ref)
    _check("db", db, dyd.sum((0, 2)))


def test_bn_relu_backward_matches_float64():
    g = torch.Generator().manual_seed(7)
    B, C, T = 3, 24, 77
    x = torch.randn(B, C, T, generator=g) * 2 + 0.5
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.3
    dy = torch.randn(B, C, T, generator=g)
    xd = x.to(DEV)
    rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    mean, var = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    y = ops.batchnorm_train_f32(xd, gamma.to(DEV), beta.to(DEV), rm, rv, eps=1e-5, momentum=0.1, out=torch.empty_like(xd),
                                stats=(mean, var))
    dx, dgam, dbet = ops.bn_relu_bwd_f32(dy.to(DEV), y, xd, mean, var, gamma.to(DEV), eps=1e-5)
    xr, gr, br = x.double().requires_grad_(), gamma.double().requires_grad_(), beta.double().requires_grad_()
    out = torch.relu(F.batch_norm(xr, None, None, gr, br, training=True, eps=1e-5))
    (out * dy.double()).sum().backward()
    _check("dx", dx, xr.grad)
    _check("dgamma", dgam, gr.grad)
    _check("dbeta", dbet, br.grad)


@pytest.mark.parametrize("T", [4, 5, 9, 64])
def test_reflect_fold_matches_float64(T):
    g = torch.Generator().manual_seed(T)
    B, Cin, Cout = 2, 19, 37
    w, dy = torch.randn(Cout, Cin, 7, generator=g) / 10, torch.randn(B, Cout, T, generator=g)
    wd, dyd = w.to(DEV), dy.to(DEV)
    dx = ops.conv1d_f32(dyd, wd.flip(-1).transpose(0, 1).contiguous())
    ops.reflect_fold_f32(dx, dyd, wd)
    xr = torch.zeros(B, Cin, T, dtype=f64, requires_grad=True)
    (F.conv1d(F.pad(xr, (3, 3), mode="reflect"), w.double()) * dy.double()).sum().backward()
    _check("dx", dx, xr.grad)


# ---------------------------------------------------------------------------------------------------------- module level
RECIPE = dict(in_dim=87, ff_hidden_dim=512, conv_hidden_dim=256, lstm_hidden_dim=128, out_dim=256, in_ph_start_idx=3,
              in_ph_end_idx=50, embed_dim=256)
BAP = dict(RECIPE, ff_hidden_dim=256, conv_hidden_dim=128, lstm_hidden_dim=64, out_dim=128)
SMALL = dict(in_dim=40, ff_hidden_dim=48, conv_hidden_dim=32, lstm_hidden_dim=32, out_dim=12, in_ph_start_idx=2,
             in_ph_end_idx=20, embed_dim=24)
CONFIGS = {
    "golden": None,
    "recipe": RECIPE,
    "bap": BAP,
    "h62": dict(SMALL, lstm_hidden_dim=62),
    "no_embed": dict(SMALL, embed_dim=None),
    "layers1": dict(SMALL, num_lstm_layers=1),
    "layers3": dict(SMALL, num_lstm_layers=3, lstm_hidden_dim=16),
    "multispeaker": dict(SMALL),
}


def _build(name, seed=0):
    torch.manual_seed(seed)
    if name == "golden":
        gd = Golden("ffconvlstm_train")
        m = FFConvLSTM(**gd.cfg, backward_kernels=True)
        m.load_state_dict(gd.sd, strict=True)
    elif name == "multispeaker":
        m = MultiSpeakerFFConvLSTM(speaker_embedding=torch.nn.Embedding(4, 24), **CONFIGS[name], backward_kernels=True)
    else:
        m = FFConvLSTM(**CONFIGS[name], backward_kernels=True)
    with torch.no_grad():                          # non-trivial BatchNorm affine and running statistics
        for k in (2, 6, 10):
            bn = m.conv[k]
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.normal_(0, 0.2)
            bn.running_mean.normal_(0, 0.1)
            bn.running_var.uniform_(0.5, 1.5)
    return m.to(DEV).train()


def _inputs(m, B, T, lens, seed=1):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, m.in_dim, generator=g)
    return x.to(DEV), lens


def _ref_grads(m, x, lens, R, spk=None):
    """float64 autograd through oracle.ffconvlstm_forward(train=True) on the CPU -> (out, {name: grad}, dx, dspk)."""
    sd = {k: v.detach().double().cpu().clone() for k, v in m.state_dict().items()}
    names = [n for n, _ in encoder_training._params(m)]
    for n in names:
        sd[n].requires_grad_(True)
    xr = x.detach().double().cpu().requires_grad_(True)
    sr = None if spk is None else spk.detach().double().cpu().requires_grad_(True)
    out = O.ffconvlstm_forward(sd, xr, lens, in_ph_start_idx=m.in_ph_start_idx, in_ph_end_idx=m.in_ph_end_idx,
                               embed_dim=m.embed_dim, num_lstm_layers=m.lstm.num_layers, spk_embs=sr, train=True)
    (out * R.double().cpu()).sum().backward()
    return out, {n: sd[n].grad for n in names}, xr.grad, None if sr is None else sr.grad


@pytest.mark.parametrize("name", list(CONFIGS))
def test_module_gradients_match_float64(name):
    m = _build(name)
    B, T = (3, 50) if name == "golden" else (3, 200) if name not in ("recipe", "bap") else (2, 120)
    lens = [T, T - 9, 4] if B == 3 else [T - 17, T]
    if name == "golden":
        gd = Golden("ffconvlstm_train")
        x, lens = gd.inp["x1"].to(DEV), gd.inp["lengths"].tolist()
    else:
        x, lens = _inputs(m, B, T, lens)
    x = x.clone().requires_grad_(True)
    R = torch.randn(B, max(lens), m.out_dim, generator=torch.Generator().manual_seed(5))
    spk = None
    if name == "multispeaker":
        spks = torch.tensor([[1], [3], [0]], device=DEV)
        out = m(x, spks, lens)
        spk = m.speaker_embedding(spks).expand(B, x.shape[1], 24)
    else:
        out = m(x, lens)
    assert out.grad_fn is not None
    (out * R.to(DEV)).sum().backward()
    ref_out, ref, dx_ref, dspk_ref = _ref_grads(m, x, lens, R, spk)
    _check("out", out, ref_out)
    errs = {}
    for n, p in encoder_training._params(m):
        assert p.grad is not None, n
        _check(n, p.grad, ref[n], errs)
    _check("x", x.grad, dx_ref, errs)
    if m.embed_dim is not None:
        s, e = m.in_ph_start_idx, m.in_ph_end_idx
        assert torch.count_nonzero(x.grad[..., s:e]) == 0           # the one-hot block only feeds argmax
    if name == "multispeaker":
        emb = m.speaker_embedding.weight.grad
        ref_emb = torch.zeros(4, 24, dtype=f64)
        for b, sidx in enumerate((1, 3, 0)):
            ref_emb[sidx] += dspk_ref[b].sum(0)
        _check("speaker_embedding", emb, ref_emb, errs)
    worst = max(errs.items(), key=lambda kv: kv[1][0])
    print(f"{name}: worst max-abs {worst[0]} {worst[1][0]:.3g}; worst rel-L2 "
          f"{max(errs.items(), key=lambda kv: kv[1][1])[0]} {max(v[1] for v in errs.values()):.3g}")


def test_padded_hidden_units_carry_zero_gradient():
    m = _build("h62")
    assert m.padded_hidden == 64
    x, lens = _inputs(m, 3, 60, [60, 7, 33])
    with torch.no_grad():
        out, keep = encoder_training._forward(m, x, lens, None)
        keep["has_spk"] = False
        _, _, grads = encoder_training._backward(m, keep, torch.randn_like(out))
    H, Hp = 62, 64
    pad_rows = lambda t: t.reshape(-1, 4, Hp, *t.shape[1:])[:, :, H:]
    assert torch.count_nonzero(grads["fc.weight"][:, H:Hp]) == 0 and torch.count_nonzero(grads["fc.weight"][:, Hp + H:]) == 0
    for l in range(2):
        assert torch.count_nonzero(pad_rows(grads[f"lstm.w_ih{l}"])) == 0
        assert torch.count_nonzero(pad_rows(grads[f"lstm.b{l}"].unsqueeze(-1))) == 0
        for d in range(2):
            w = grads[f"lstm.w_hh{l}"][d]
            assert torch.count_nonzero(pad_rows(w)) == 0 and torch.count_nonzero(w[:, H:]) == 0
        if l > 0:
            w = grads[f"lstm.w_ih{l}"]
            assert torch.count_nonzero(w[:, H:Hp]) == 0 and torch.count_nonzero(w[:, Hp + H:]) == 0
    for l in range(2):                                          # padded units emit h = 0
        hout = keep["lstm"][l][1]
        assert torch.count_nonzero(hout[:, H:Hp]) == 0 and torch.count_nonzero(hout[:, Hp + H:]) == 0


# ------------------------------------------------------------------------------------------------------------- behaviour
def test_grad_forward_equals_no_grad_training_forward_bitwise():
    a = _build("recipe")
    b = copy.deepcopy(a)
    x, lens = _inputs(a, 3, 150, [150, 61, 4])
    ya = a(x, lens)
    assert ya.grad_fn is not None
    with torch.no_grad():
        yb = b(x, lens)
    assert torch.equal(ya.detach(), yb)
    for (n, ba), bb in zip(a.named_buffers(), b.buffers()):
        assert torch.equal(ba, bb), n
    assert int(a.conv[2].num_batches_tracked) == 1


def test_two_backward_passes_are_bitwise_identical():
    m = _build("bap")
    x, lens = _inputs(m, 3, 120, [120, 40, 77])
    R = torch.randn(3, 120, m.out_dim, device=DEV)
    gs = []
    for _ in range(2):
        mm = copy.deepcopy(m)
        (mm(x, lens) * R).sum().backward()
        gs.append([p.grad.clone() for _, p in encoder_training._params(mm)])
    for a, b in zip(*gs):
        assert torch.equal(a, b)


def test_sgd_steps_match_oracle_driven_steps():
    """Five SGD steps on a mean loss: all parameters together within 1e-6 relative (L2 over the concatenation) of the same
    steps driven by float64 oracle gradients."""
    m = _build("no_embed")
    ref = copy.deepcopy(m)
    x, lens = _inputs(m, 2, 80, [80, 51])
    R = torch.randn(2, 80, m.out_dim, generator=torch.Generator().manual_seed(3))
    R = R / R.numel()                               # the gradient of a mean loss
    lr = 0.1
    for _ in range(5):
        m.zero_grad()
        (m(x, lens) * R.to(DEV)).sum().backward()
        _, grads, _, _ = _ref_grads(ref, x, lens, R)
        with torch.no_grad():
            for n, p in encoder_training._params(m):
                p -= lr * p.grad
            for n, p in encoder_training._params(ref):
                p -= lr * grads[n].to(DEV, torch.float32)
    ours = torch.cat([p.detach().flatten() for _, p in encoder_training._params(m)])
    theirs = torch.cat([p.detach().flatten() for _, p in encoder_training._params(ref)])
    rel = ((ours - theirs).norm() / theirs.norm()).item()
    worst = max(((p - q).norm().item() / max(q.norm().item(), 1e-3), n)
                for (n, p), (_, q) in zip(encoder_training._params(m), encoder_training._params(ref)))
    print(f"sgd: all parameters {rel:.3g} relative; worst tensor {worst[1]} {worst[0]:.3g}")
    assert rel <= 1e-6


def test_eval_and_no_grad_record_no_graph():
    m = _build("layers1")
    x, lens = _inputs(m, 2, 40, [40, 22])
    with torch.no_grad():
        assert m(x, lens).grad_fn is None
    m.eval()
    assert m(x.clone().requires_grad_(True), lens).grad_fn is None


def test_unsupported_configurations_raise_before_launch():
    mdn = FFConvLSTM(16, 32, 16, 8, 4, use_mdn=True, backward_kernels=True).to(DEV).train()
    with pytest.raises(RuntimeError, match="MDN head"):
        mdn(torch.zeros(1, 8, 16, device=DEV))
    big = FFConvLSTM(16, 32, 16, 300, 4, backward_kernels=True).to(DEV).train()
    with pytest.raises(RuntimeError, match="at most 256 units"):
        big(torch.zeros(1, 8, 16, device=DEV))
    drop = FFConvLSTM(16, 32, 16, 8, 4, dropout=0.1, backward_kernels=True).to(DEV).train()
    with pytest.raises(RuntimeError, match="dropout = 0 only"):
        drop(torch.zeros(1, 8, 16, device=DEV))


def test_gaussian_diffusion_step_fills_encoder_gradients():
    from ensemble_svs_with_interactions_b200.diffsinger import DiffNet, GaussianDiffusion
    torch.manual_seed(11)
    enc = FFConvLSTM(**RECIPE, backward_kernels=True)
    model = GaussianDiffusion(87, 60, DiffNet(60, 256, 20, 256, 4), encoder=enc, K_step=100).to(DEV).train()
    before = copy.deepcopy(model.encoder)
    B, T = 2, 200
    g = torch.Generator().manual_seed(12)
    cond, y = torch.randn(B, T, 87, generator=g).to(DEV), torch.randn(B, T, 60, generator=g).to(DEV)
    t = torch.randint(0, 100, (B,), generator=g).to(DEV)
    noise = torch.randn(B, 1, 60, T, generator=g).to(DEV)
    captured = {}
    def keep_grad(mod, inp, out):
        out.register_hook(lambda gr: captured.setdefault("g", gr.clone()))     # returns None: the output is unchanged

    h = model.encoder.register_forward_hook(keep_grad)
    n, eps = model(cond, [T, T - 30], y, t=t, noise=noise)
    (n - eps).abs().mean().backward()
    h.remove()
    for name, p in encoder_training._params(model.encoder):
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
    out = before(cond, [T, T - 30])
    out.backward(captured["g"])
    for (name, p), (_, q) in zip(encoder_training._params(model.encoder), encoder_training._params(before)):
        assert torch.equal(p.grad, q.grad), name
