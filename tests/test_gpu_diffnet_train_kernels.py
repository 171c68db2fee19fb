"""The DiffNet training kernels (csrc/diffnet_train_sm100.cu) one launch at a time against float64, and the gradients of
DiffNet in training mode against a float64 restatement of diffsinger/training.py that rounds to bf16 exactly where the
kernels store bf16.

Per launch: the inputs are seeded bf16 tensors, and the reference is the same formula evaluated in float64 on the same
bf16 values (torch on the device).  Every element is checked against
    |got - ref| <= C_ACC * (|A| @ |B| + |every added term|)        (+ 2^-8 |ref| for bf16 outputs)
i.e. fp32 accumulation error scaled by the float64 sum of absolute terms (so cancellation cannot loosen the bound), plus
the bf16 rounding of the stored value.  The gate modes add C_ACT times the size of the activation's factor for
tanh.approx.f32 (and sigmoid through it).  Segment
columns beyond kx, time columns beyond T and output columns beyond N hold NaN or a sentinel: they must be neither read
nor written.  The transpose and the weight pack are checked bit for bit.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from ensemble_svs_with_interactions_b200 import ops
from ensemble_svs_with_interactions_b200.diffsinger import training as TR

pytestmark = pytest.mark.gpu
DEV = "cuda"
bf16, f32, f64 = torch.bfloat16, torch.float32, torch.float64

# Bound constants; DESIGN.md §5 records the worst measured value of each on a B200.
C_ACC = 1.5 * 2.0 ** -20    # fp32 accumulation, relative to the float64 sum of absolute terms
C_BF16 = 2.0 ** -8          # bf16 round-to-nearest of a stored output (the exact bound, not a fitted constant)
C_ACT = 2.0 ** -18          # tanh.approx.f32 beyond the rounding bound (absolute, on values in [-1, 1])
REL_L2_BF16 = 3e-3          # rel-L2 of a bf16 output of one launch
REL_L2_F32 = 1e-5           # rel-L2 of an fp32 output of one launch
GRAD_REL_L2 = 1e-2          # end-to-end gradients vs the bf16-faithful float64 reference
MASK_FLIPS = 2.5e-3         # share of the tail ReLU's decisions the kernels and the reference may take differently
MASK_NEAR = 2e-2            # ... each at an input within this fraction of the inputs' rms
SENTINEL = -4096.0          # exactly representable in bf16 and fp32
RS2 = 1.0 / math.sqrt(2.0)


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _randn_bf16(shape, g, scale=1.0):
    return (torch.randn(shape, generator=g, device=DEV) * scale).to(bf16)


def _padded(x, ld, fill=float("nan")):
    """[..., k] -> [..., ld] with the columns beyond k set to `fill` (a pitch larger than the data)."""
    out = torch.full(x.shape[:-1] + (ld,), fill, device=DEV, dtype=x.dtype)
    out[..., :x.shape[-1]] = x
    return out


def _shift(x, s):
    """x [B, T, K] -> x[:, t + s] with zeros outside [0, T) (the conv's zero padding)."""
    T = x.shape[1]
    out = torch.zeros_like(x)
    if s >= 0 and s < T:
        out[:, :T - s] = x[:, s:]
    elif s < 0 and -s < T:
        out[:, -s:] = x[:, :T + s]
    return out


def _check(name, got, ref, absref, *, is_bf16, act=None):
    """Every element within the bound; also the rel-L2.  Returns the worst fraction of the bound used."""
    got = got.to(f64)
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    err = (got - ref).abs()
    bound = C_ACC * absref
    if is_bf16:
        bound = bound + C_BF16 * ref.abs()
    if act is not None:
        bound = bound + C_ACT * act
    frac = (err / bound.clamp_min(1e-300)).max().item() if err.numel() else 0.0
    r = ((got - ref).norm() / ref.norm().clamp_min(1e-300)).item()
    need = ""
    if act is not None:        # the smallest C_ACT that would still hold
        rest = (err - C_ACC * absref - (C_BF16 * ref.abs() if is_bf16 else 0)).clamp_min(0)
        need = f", C_ACT >= {(rest / act.clamp_min(1e-300)).max().item():.2e}"
    print(f"  {name:10s} worst {frac:.3f} of bound, rel-L2 {r:.2e}{need}")
    bad = (err > bound).nonzero()
    assert bad.numel() == 0, f"{name}: {bad.shape[0]} elements outside the bound, first at {bad[0].tolist()}: " \
                             f"got {got[tuple(bad[0])].item()!r} ref {ref[tuple(bad[0])].item()!r}"
    assert r <= (REL_L2_BF16 if is_bf16 else REL_L2_F32) or ref.norm().item() == 0.0, f"{name}: rel-L2 {r:.3e}"
    return frac


def _untouched(name, t, cols):
    """The spare columns [cols, ld) of an output still hold the sentinel."""
    if t.shape[-1] > cols:
        assert (t[..., cols:].float() == SENTINEL).all(), f"{name}: columns beyond {cols} were written"


def _segments(B, T, spec, g):
    """spec: list of (kx, ld, shift, key).  Segments with the same key share one tensor.  Returns (kernel segments,
    [(x float64 [B, T, kx], shift)])."""
    tensors, segs, refs = {}, [], []
    for kx, ld, shift, key in spec:
        if key not in tensors:
            tensors[key] = _padded(_randn_bf16((B, T, kx), g), ld)
        x = tensors[key]
        segs.append((x, kx, shift))
        refs.append((x[..., :kx].to(f64), shift))
    return segs, refs


def _gemm_ref(refs, w):
    """D and |A| @ |B| in float64: D[b, t, n] = sum_s x_s[b, t + shift_s] . w[n, koff_s:]."""
    w = w.to(f64)
    D, A, koff = 0, 0, 0
    for x, s in refs:
        xs, ws = _shift(x, s), w[:, koff:koff + x.shape[2]]
        D = D + xs @ ws.t()
        A = A + xs.abs() @ ws.abs().t()
        koff += x.shape[2]
    return D, A


# ------------------------------------------------------------------------------------------------ seggemm: PLAIN, ADD_SCALE
# (B, T, segments [(kx, ld, shift, key)], Nrows, bias, act, alpha, in0, mask, out0 / out1 / outf, accumulate, out pitch pad)
PLAIN_CASES = [
    (1, 1, [(64, 64, 0, 0)], 16, True, ops.ACT_RELU, 1.0, False, False, "o", False, 0),
    (3, 129, [(128, 136, 0, 0)], 80, True, ops.ACT_NONE, 0.5, False, True, "o", False, 8),
    (6, 1000, [(256, 256, 0, 0)], 272, True, ops.ACT_RELU, 1.0, False, False, "o1f", True, 16),
    (3, 128, [(64, 128, 8, 0), (128, 128, -8, 1)], 512, False, ops.ACT_RELU, -0.75, False, True, "f", False, 8),
    (3, 7, [(64, 64, 9, 0), (64, 64, 0, 0)], 64, True, ops.ACT_NONE, 2.0, True, False, "of", True, 0),
    (1, 127, [(192, 200, 0, 0)], 256, True, ops.ACT_RELU, 0.25, True, True, "o1", False, 8),
    (6, 1000, [(64, 64, 0, 0)], 256, True, ops.ACT_RELU, 1.0, False, False, "o1", False, 0),   # the head's shape
]


@pytest.mark.parametrize("B,T,spec,Nrows,bias,act,alpha,in0,mask,outs,accumulate,pad", PLAIN_CASES)
def test_seggemm_plain(B, T, spec, Nrows, bias, act, alpha, in0, mask, outs, accumulate, pad):
    """PLAIN: act(D + bias + in0) * alpha, then zero where mask <= 0; out1 adds a per-track vector; outf (+)= fp32."""
    g = _gen(B * 7 + T + Nrows)
    segs, refs = _segments(B, T, spec, g)
    K = sum(k for k, _, _, _ in spec)
    w = _randn_bf16((Nrows, K), g, 1.0 / math.sqrt(K))
    b = torch.randn(Nrows, generator=g, device=DEV) * 0.5 if bias else None
    x_in = _padded(_randn_bf16((B, T, Nrows), g), Nrows + pad) if in0 else None
    m = _padded(torch.relu(_randn_bf16((B, T, Nrows), g)), Nrows + pad) if mask else None   # exact zeros: a ReLU output
    dp = torch.randn((B, Nrows), generator=g, device=DEV) if "1" in outs else None
    o0 = torch.full((B, T, Nrows + pad), SENTINEL, device=DEV, dtype=bf16) if "o" in outs else None
    o1 = torch.full((B, T, Nrows + pad), SENTINEL, device=DEV, dtype=bf16) if "1" in outs else None
    prev = torch.randn((B, T, Nrows), generator=g, device=DEV)
    of = _padded(prev, Nrows + pad, SENTINEL) if "f" in outs else None
    ops.seggemm_bf16(segs, w, mode=ops.SEG_PLAIN, bias=b, in0=x_in, mask=m, dp_next=dp, out0=o0, out1=o1, outf=of,
                     alpha=alpha, act=act, accumulate=accumulate)
    D, A = _gemm_ref(refs, w)
    if b is not None:
        D, A = D + b.to(f64), A + b.abs().to(f64)
    if x_in is not None:
        D, A = D + x_in[..., :Nrows].to(f64), A + x_in[..., :Nrows].abs().to(f64)
    v = torch.relu(D) if act == ops.ACT_RELU else D
    v, A = v * alpha, A * abs(alpha)
    if m is not None:
        keep = m[..., :Nrows] > 0
        v, A = torch.where(keep, v, 0.0), torch.where(keep, A, 0.0)
    if o0 is not None:
        _check("out0", o0[..., :Nrows], v, A, is_bf16=True)
        _untouched("out0", o0, Nrows)
    if o1 is not None:
        dpv = dp.to(f64)[:, None]
        _check("out1", o1[..., :Nrows], v + dpv, A + dpv.abs(), is_bf16=True)
        _untouched("out1", o1, Nrows)
    if of is not None:
        ref, absref = (v + prev.to(f64), A + prev.abs().to(f64)) if accumulate else (v, A)
        _check("outf", of[..., :Nrows], ref, absref, is_bf16=False)
        _untouched("outf", of, Nrows)


# (B, T, C, d, alpha, mask, ld pad of dy, out pitch pad)
ADD_SCALE_CASES = [
    (6, 1000, 256, 8, RS2, False, 0, 0),       # config 5's dgrad: K = 3 * 2C = 1536
    (3, 129, 128, 2, 1.0, True, 0, 8),         # the first block: mask = x0
    (3, 7, 128, 8, 1.0, True, 64, 0),          # a tap shift larger than T
    (1, 1, 256, 1, RS2, False, 0, 0),
    (6, 128, 128, 4, RS2, False, 64, 8),
    (3, 127, 256, 1, 1.0, True, 0, 0),
]


@pytest.mark.parametrize("B,T,C,d,alpha,mask,ldpad,pad", ADD_SCALE_CASES)
def test_seggemm_add_scale_dgrad(B, T, C, d, alpha, mask, ldpad, pad):
    """ADD_SCALE as the transposed conv uses it: u = ([dy(t+d) | dy(t) | dy(t-d)] . w1T + u_next) * alpha [* (x0 > 0)]."""
    g = _gen(B * 11 + T + C + d)
    C2 = 2 * C
    segs, refs = _segments(B, T, [(C2, C2 + ldpad, d, 0), (C2, C2 + ldpad, 0, 0), (C2, C2 + ldpad, -d, 0)], g)
    w = _randn_bf16((C, 3 * C2), g, 1.0 / math.sqrt(3 * C2))
    u_next = _padded(_randn_bf16((B, T, C), g), C + pad)
    x0 = _padded(torch.relu(_randn_bf16((B, T, C), g)), C + pad) if mask else None
    out = torch.full((B, T, C + pad), SENTINEL, device=DEV, dtype=bf16)
    ops.seggemm_bf16(segs, w, mode=ops.SEG_ADD_SCALE, in0=u_next, alpha=alpha, mask=x0, out0=out)
    D, A = _gemm_ref(refs, w)
    un = u_next[..., :C].to(f64)
    v, A = (D + un) * alpha, (A + un.abs()) * alpha
    if x0 is not None:
        keep = x0[..., :C] > 0
        v, A = torch.where(keep, v, 0.0), torch.where(keep, A, 0.0)
    _check("u", out[..., :C], v, A, is_bf16=True)
    _untouched("u", out, C)


# ------------------------------------------------------------------------------------------------ seggemm: GATE_FWD
# (B, T, C, H, d, segment ld pad, out pitch pad)
GATE_FWD_CASES = [
    (6, 1000, 256, 256, 8, 0, 0),              # config 5
    (3, 129, 128, 64, 1, 0, 0),
    (3, 7, 128, 64, 8, 64, 8),                 # d > T
    (1, 127, 256, 64, 2, 64, 16),
    (3, 128, 128, 256, 4, 0, 8),
    (1, 1, 128, 64, 1, 0, 0),
]


@pytest.mark.parametrize("B,T,C,H,d,ldpad,pad", GATE_FWD_CASES)
def test_seggemm_gate_fwd(B, T, C, H, d, ldpad, pad):
    """GATE_FWD: y = [xd(t-d) | xd | xd(t+d) | cond] . W1p + b1 in the packed row order of ops.diffnet_packed_rows;
    ypre = bf16(y), z = sigmoid(y_gate) * tanh(y_filter) from the unrounded fp32 y."""
    g = _gen(B * 13 + T + C + H + d)
    C2 = 2 * C
    segs, refs = _segments(B, T, [(C, C + ldpad, -d, 0), (C, C + ldpad, 0, 0), (C, C + ldpad, d, 0), (H, H + ldpad, 0, 1)], g)
    K = 3 * C + H
    w_ref = _randn_bf16((C2, K), g, 1.5 / math.sqrt(K))         # reference row order: gate rows [0, C), filter [C, 2C)
    b_ref = torch.randn(C2, generator=g, device=DEV) * 0.5
    perm = ops.diffnet_packed_rows(C).to(DEV)
    wp = torch.empty_like(w_ref)
    wp[perm] = w_ref
    bp = torch.empty_like(b_ref)
    bp[perm] = b_ref
    ypre = torch.full((B, T, C2 + pad), SENTINEL, device=DEV, dtype=bf16)
    z = torch.full((B, T, C + pad), SENTINEL, device=DEV, dtype=bf16)
    ops.seggemm_bf16(segs, wp, mode=ops.SEG_GATE_FWD, bias=bp, out0=ypre, out1=z)
    y, A = _gemm_ref(refs, w_ref)
    y, A = y + b_ref.to(f64), A + b_ref.abs().to(f64)
    _check("ypre", ypre[..., :C2][..., perm], y, A, is_bf16=True)
    s, th = torch.sigmoid(y[..., :C]), torch.tanh(y[..., C:])
    # |dz| <= |d sigmoid| + |d tanh| <= dy_gate + dy_filter; tanh.approx: absolute, plus its share through sigmoid
    _check("z", z[..., :C], s * th, A[..., :C] + A[..., C:], is_bf16=True, act=1.0 + th.abs())
    _untouched("ypre", ypre, C2)
    _untouched("z", z, C)


# ------------------------------------------------------------------------------------------------ seggemm: GATE_BWD
# (B, T, C, ypre pitch pad, out pitch pad)
GATE_BWD_CASES = [
    (6, 1000, 256, 0, 0),
    (3, 129, 128, 0, 0),
    (1, 1, 128, 0, 0),
    (3, 7, 256, 64, 16),
    (3, 128, 128, 8, 8),
]


@pytest.mark.parametrize("B,T,C,ypad,pad", GATE_BWD_CASES)
def test_seggemm_gate_bwd(B, T, C, ypad, pad):
    """GATE_BWD: dz = [u | dS] . Wout; dy_gate = dz tanh(f) s (1 - s), dy_filter = dz s (1 - tanh^2 f), s = sigmoid(g),
    evaluated at the stored bf16 ypre (packed columns)."""
    g = _gen(B * 17 + T + C)
    C2 = 2 * C
    segs, refs = _segments(B, T, [(C, C, 0, 0), (C, C, 0, 1)], g)
    wT = _randn_bf16((C, C2), g, 1.0 / math.sqrt(C2))
    ypre = _padded(_randn_bf16((B, T, C2), g, 2.0), C2 + ypad)
    dy = torch.full((B, T, C2 + pad), SENTINEL, device=DEV, dtype=bf16)
    ops.seggemm_bf16(segs, wT, mode=ops.SEG_GATE_BWD, in0=ypre, out0=dy)
    dz, A = _gemm_ref(refs, wT)                                  # [B, T, C], channel c = 128 p + i
    yp = ypre[..., :C2].to(f64).reshape(B, T, C // 128, 2, 128)
    s, th = torch.sigmoid(yp[:, :, :, 0]), torch.tanh(yp[:, :, :, 1])
    dzp, Ap = dz.reshape(B, T, C // 128, 128), A.reshape(B, T, C // 128, 128)
    dg, df = s * (1 - s) * th, s * (1 - th * th)
    ref = torch.stack([dzp * dg, dzp * df], dim=3).reshape(B, T, C2)
    absref = torch.stack([Ap * dg.abs(), Ap * df.abs()], dim=3).reshape(B, T, C2)
    act = 2.0 * torch.stack([dzp.abs(), dzp.abs()], dim=3).reshape(B, T, C2)
    _check("dy", dy[..., :C2], ref, absref, is_bf16=True, act=act)
    _untouched("dy", dy, C2)


# ------------------------------------------------------------------------------------------------ seggemm: RES_SKIP
# (B, T, C, init, write x' / xd', in0 pitch pad, out pitch pad)
RES_SKIP_CASES = [
    (6, 1000, 256, True, True, 0, 0),
    (3, 129, 128, False, True, 8, 8),
    (3, 7, 128, False, False, 0, 0),           # the last block: no x' / xd'
    (1, 1, 256, True, True, 0, 16),
    (3, 128, 256, False, False, 64, 4),
    (6, 127, 128, True, False, 0, 0),
]


@pytest.mark.parametrize("B,T,C,init,write_x,inpad,pad", RES_SKIP_CASES)
def test_seggemm_res_skip(B, T, C, init, write_x, inpad, pad):
    """RES_SKIP: o = z . Wout + bout; x' = (x + o[:C]) / sqrt 2, xd' = x' + dp_next, skip = (init ? 0 : skip) + o[C:]."""
    g = _gen(B * 19 + T + C + int(init))
    C2 = 2 * C
    segs, refs = _segments(B, T, [(C, C, 0, 0)], g)
    w = _randn_bf16((C2, C), g, 1.0 / math.sqrt(C))
    b = torch.randn(C2, generator=g, device=DEV) * 0.5
    x = _padded(_randn_bf16((B, T, C), g), C + inpad)
    dp = torch.randn((B, C), generator=g, device=DEV)
    xo = torch.full((B, T, C + pad), SENTINEL, device=DEV, dtype=bf16) if write_x else None
    xdo = torch.full((B, T, C + pad), SENTINEL, device=DEV, dtype=bf16) if write_x else None
    prev = torch.randn((B, T, C), generator=g, device=DEV)
    skip = _padded(torch.full_like(prev, float("nan")) if init else prev, C + pad, SENTINEL)
    ops.seggemm_bf16(segs, w, mode=ops.SEG_RES_SKIP, bias=b, in0=x, out0=xo, out1=xdo, dp_next=dp if write_x else None,
                     outf=skip, init=init)
    o, A = _gemm_ref(refs, w)
    o, A = o + b.to(f64), A + b.abs().to(f64)
    xv = x[..., :C].to(f64)
    xn, An = (xv + o[..., :C]) * RS2, (xv.abs() + A[..., :C]) * RS2
    if write_x:
        _check("x'", xo[..., :C], xn, An, is_bf16=True)
        dpv = dp.to(f64)[:, None]
        _check("xd'", xdo[..., :C], xn + dpv, An + dpv.abs(), is_bf16=True)
        _untouched("x'", xo, C)
        _untouched("xd'", xdo, C)
    ref, absref = (o[..., C:], A[..., C:]) if init else (o[..., C:] + prev.to(f64), A[..., C:] + prev.abs().to(f64))
    _check("skip", skip[..., :C], ref, absref, is_bf16=False)
    _untouched("skip", skip, C)


# ------------------------------------------------------------------------------------------------ wgrad
def _nct(B, rows, T, Tp, g):
    """[B, rows, Tp] bf16 operand with NaN in the time columns [T, Tp): frames the kernel must not read."""
    x = torch.full((B, rows, Tp), float("nan"), device=DEV, dtype=bf16)
    x[:, :, :T] = _randn_bf16((B, rows, T), g)
    return x


def _wgrad_ref(p, qs, T):
    """dW[n, koff_s + k] = sum_b sum_{t < T} p[b, n, t] q_s[b, k, t + shift_s] (q zero outside [0, T)), and the sum of
    absolute terms."""
    P = p[:, :, :T].to(f64)
    D, A = [], []
    for q, s in qs:
        Q = _shift(q[:, :, :T].to(f64).transpose(1, 2), s).transpose(1, 2)      # shift along time
        D.append(torch.einsum("bnt,bkt->nk", P, Q))
        A.append(torch.einsum("bnt,bkt->nk", P.abs(), Q.abs()))
    return torch.cat(D, 1), torch.cat(A, 1)


# (B, T, Prows, [(rows, shift)], accumulate, ldw pad)
WGRAD_CASES = [
    (1, 1, 64, [(16, 0)], False, 0),
    (3, 63, 128, [(64, 8), (144, -8)], False, 4),
    (2, 1000, 256, [(128, 0), (768, 64), (384, -64), (16, 8), (64, -8)], False, 0),
    (3, 65, 512, [(144, -64)], True, 12),
    (3, 64, 128, [(768, 0), (16, 64)], True, 0),
    (6, 1000, 64, [(128, -8), (16, 0)], False, 0),
]


@pytest.mark.parametrize("B,T,Prows,qspec,accumulate,ldpad", WGRAD_CASES)
def test_wgrad(B, T, Prows, qspec, accumulate, ldpad):
    g = _gen(B * 23 + T + Prows + len(qspec))
    Tp = (T + 7) // 8 * 8 + (8 if T % 8 == 0 else 0)     # always some padding columns to fill with NaN
    p = _nct(B, Prows, T, Tp, g)
    qs = [(_nct(B, rows, T, Tp, g), s) for rows, s in qspec]
    K = sum(rows for rows, _ in qspec)
    prev = torch.randn((Prows, K), generator=g, device=DEV)
    dW = _padded(prev, K + ldpad, SENTINEL)
    ops.wgrad_bf16(p, qs, dW, T=T, accumulate=accumulate)
    D, A = _wgrad_ref(p, qs, T)
    if accumulate:
        D, A = D + prev.to(f64), A + prev.abs().to(f64)
    _check("dW", dW[:, :K], D, A, is_bf16=False)
    _untouched("dW", dW, K)


# (B, T, d, splits): config 5 selects 3 and 6 at B 6; uneven groups at B 5; empty groups at 8 > B
@pytest.mark.parametrize("B,T,d,splits", [(6, 1000, 8, 3), (6, 1000, 1, 6), (5, 517, 2, 2), (5, 517, 4, 3), (5, 129, 8, 8)])
def test_wgrad_track_groups_with_indicator_rows(B, T, d, splits):
    """The dW1 launch of a block: P = dy^T [B, 2C, Tp], Q = [xd taps (3C) | cond (H) | indicator rows (R)], track groups
    through the 3-D dW.  Each group's partial result, their sum against splits = 1, and a repeated launch bit for bit."""
    C, H = 256, 256
    g = _gen(B * 29 + T + d + splits)
    Tp = (T + 7) // 8 * 8
    p = _nct(B, 2 * C, T, Tp, g)
    xdT = _nct(B, 3 * C, T, Tp, g)
    condT = _nct(B, H, T, Tp, g)
    ind = TR._indicator_rows(B, T, Tp, d, DEV)
    assert ind.shape[1] == (3 * B + 15) // 16 * 16
    qs = [(xdT, 0), (condT, 0), (ind, 0)]
    K = 3 * C + H + ind.shape[1]
    one = torch.full((2 * C, K + 8), SENTINEL, device=DEV)
    ops.wgrad_bf16(p, qs, one, T=T)
    parts = torch.full((splits, 2 * C, K + 8), float("nan"), device=DEV)
    parts[..., K:] = SENTINEL
    ops.wgrad_bf16(p, qs, parts, T=T)
    again = torch.full_like(parts, float("nan"))
    ops.wgrad_bf16(p, qs, again, T=T)
    D, A = _wgrad_ref(p, qs, T)
    _check("splits=1", one[:, :K], D, A, is_bf16=False)
    _untouched("splits=1", one, K)
    for z in range(splits):                  # group z sums tracks [B z / S, B (z + 1) / S): possibly none -> zeros
        b0, b1 = B * z // splits, B * (z + 1) // splits
        if b1 == b0:
            assert (parts[z, :, :K] == 0).all(), f"empty group {z} must write zeros"
        else:
            Dz, Az = _wgrad_ref(p[b0:b1], [(q[b0:b1], s) for q, s in qs], T)
            _check(f"group {z}", parts[z, :, :K], Dz, Az, is_bf16=False)
        _untouched(f"group {z}", parts[z], K)
    _check("sum", parts[:, :, :K].sum(0), one[:, :K].to(f64), A, is_bf16=False)
    assert torch.equal(parts[..., :K], again[..., :K]), "a repeated launch must be bit-identical"
    # the indicator columns are the per-track sums of P over all / the first d / the last d frames
    P = p[:, :, :T].to(f64)
    cs = one[:, 3 * C + H:3 * C + H + 3 * B].reshape(2 * C, B, 3).permute(1, 2, 0).to(f64)
    ref = torch.stack([P.sum(2), P[:, :, :min(d, T)].sum(2), P[:, :, max(T - d, 0):].sum(2)], dim=1)
    absref = torch.stack([P.abs().sum(2), P[:, :, :min(d, T)].abs().sum(2), P[:, :, max(T - d, 0):].abs().sum(2)], dim=1)
    _check("ind sums", cs, ref, absref, is_bf16=False)


# ------------------------------------------------------------------------------------------------ ntc_to_nct_bf16
# (B, T, N, ldx, shifts, row0, spare rows after the copies)
NTC_CASES = [
    (3, 1, 8, 8, (0,), 0, 0),
    (3, 7, 72, 80, (-8, 0, 8), 8, 16),
    (2, 129, 256, 264, (-2, 0, 2), 256, 0),
    (6, 1000, 256, 256, (0,), 0, 0),
    (3, 64, 72, 72, (-64, 64), 72, 8),
    (1, 1000, 8, 16, (-1000, 1, 999), 24, 8),
    (3, 127, 72, 72, (5, -3), 0, 0),
]


@pytest.mark.parametrize("B,T,N,ldx,shifts,row0,spare", NTC_CASES)
def test_ntc_to_nct_bf16(B, T, N, ldx, shifts, row0, spare):
    """out[b, row0 + j N + n, t] = x[b, t + shift_j, n] where that frame exists, else 0, bit for bit, for every t < Tp:
    the columns [T, Tp) are written by the same rule (no consumer reads them).  Rows outside the copies are untouched."""
    g = _gen(B * 31 + T + N + row0)
    x = _padded(_randn_bf16((B, T, N), g), ldx)
    Tp = (T + 7) // 8 * 8
    rows = row0 + len(shifts) * N + spare
    out = torch.full((B, rows, Tp), SENTINEL, device=DEV, dtype=bf16)
    ops.ntc_to_nct_bf16(x, N=N, out=out, row0=row0, shifts=shifts)
    for j, s in enumerate(shifts):
        ref = torch.zeros((B, Tp, N), device=DEV, dtype=bf16)
        lo, hi = max(0, -s), min(Tp, T - s)                    # frames t with 0 <= t + s < T
        if lo < hi:
            ref[:, lo:hi] = x[:, lo + s:hi + s, :N]
        got = out[:, row0 + j * N:row0 + (j + 1) * N]
        assert torch.equal(got, ref.transpose(1, 2)), f"shift {s}: {(got != ref.transpose(1, 2)).sum().item()} elements differ"
    assert (out[:, :row0] == SENTINEL).all() and (out[:, row0 + len(shifts) * N:] == SENTINEL).all(), "rows outside written"


# ------------------------------------------------------------------------------------------------ diffnet_train_pack
@pytest.mark.parametrize("C,H,L", [(128, 64, 1), (256, 192, 3), (128, 192, 3), (256, 64, 1)])
def test_diffnet_train_pack_bit_exact(C, H, L):
    g = _gen(C + H + L)
    C2 = 2 * C
    wd = torch.randn((L, C2, C, 3), generator=g, device=DEV) * 0.1
    wc = torch.randn((L, C2, H), generator=g, device=DEV) * 0.1
    wo = torch.randn((L, C2, C), generator=g, device=DEV) * 0.1
    pk = ops.diffnet_train_pack(wd, wc, wo)
    perm = ops.diffnet_packed_rows(C).to(DEV)
    taps = wd.permute(0, 1, 3, 2).reshape(L, C2, 3 * C).to(bf16)            # [l, r, j C + ci]
    w1p = torch.empty((L, C2, 3 * C + H), device=DEV, dtype=bf16)
    w1p[:, perm] = torch.cat([taps, wc.to(bf16)], dim=2)
    w1T = torch.empty((L, C, 3 * C2), device=DEV, dtype=bf16)
    wcT = torch.empty((L, H, C2), device=DEV, dtype=bf16)
    for j in range(3):
        w1T[:, :, j * C2 + perm] = wd[:, :, :, j].transpose(1, 2).to(bf16)
    wcT[:, :, perm] = wc.transpose(1, 2).to(bf16)
    want = dict(w1p=w1p, woutp=wo.to(bf16), woutT=wo.transpose(1, 2).to(bf16), w1T=w1T, wcT=wcT)
    for k, v in want.items():
        assert torch.equal(pk[k].view(torch.int16), v.view(torch.int16)), f"{k}: {(pk[k] != v).sum().item()} elements differ"


# ------------------------------------------------------------------------------------------------ end to end
def _bf(x):
    """Round to bf16 where a kernel stores bf16, keep computing in float64."""
    return x.to(bf16).to(f64)


def _mish(x):
    return x * torch.tanh(F.softplus(x))


def _rel_l2(got, ref):
    got, ref = got.to(f64), ref.to(f64).reshape(got.shape)
    return ((got - ref).norm() / ref.norm().clamp_min(1e-300)).item()


def _reference_grads(net, spec, t, cond, d_eps, h_mask=None):
    """float64 restatement of training._stack_forward / _stack_backward (activations [B, T, channels], reference row
    order), rounded to bf16 exactly where the kernels store bf16: forward specb, condb, x0, xd_l, ypre_l, z_l, x_{l+1},
    Sb, h; backward deb, dh, dS, dy_l, u_l, dpre0.  Sums and everything else in float64; weights enter the GEMMs as
    bf16, as packed.  The step-embedding MLP is float64 autograd.  h_mask: the tail ReLU's mask to use in the backward
    instead of h > 0 (the kernels' own, see the test).  Returns ({parameter name: gradient}, d spec, d cond,
    {'x0', 'h': the ReLU outputs, 'hpre': the tail ReLU's input})."""
    P = {k: v.detach().to(f64) for k, v in net.named_parameters()}
    layers = net.residual_layers
    L, C = len(layers), net.residual_channels
    dil = [int(ly.dilation) for ly in layers]
    pre = [f"residual_layers.{l}." for l in range(L)]
    # step embedding and per-layer projections dp [L, B, C], float64 autograd
    mlp = {k: P[k].clone().requires_grad_(True) for k in ("mlp.0.weight", "mlp.0.bias", "mlp.2.weight", "mlp.2.bias")}
    dpw = [P[p + "diffusion_projection.weight"].clone().requires_grad_(True) for p in pre]
    dpb = [P[p + "diffusion_projection.bias"].clone().requires_grad_(True) for p in pre]
    half = C // 2
    freq = torch.exp(torch.arange(half, device=DEV, dtype=f64) * -(math.log(10000) / (half - 1)))
    arg = t.to(f64)[:, None] * freq[None]
    e = torch.cat((arg.sin(), arg.cos()), dim=-1)
    e = F.linear(_mish(F.linear(e, mlp["mlp.0.weight"], mlp["mlp.0.bias"])), mlp["mlp.2.weight"], mlp["mlp.2.bias"])
    dp_t = torch.stack([F.linear(e, w, b) for w, b in zip(dpw, dpb)])                    # [L, B, C]
    dp = dp_t.detach()
    Wd = [P[p + "dilated_conv.weight"] for p in pre]                                     # [2C, C, 3] fp32 values
    Wdb = [_bf(w) for w in Wd]
    Wcb = [_bf(P[p + "conditioner_projection.weight"][:, :, 0]) for p in pre]          # [2C, H]
    Wob = [_bf(P[p + "output_projection.weight"][:, :, 0]) for p in pre]               # [2C, C]
    b1 = [P[p + "dilated_conv.bias"] + P[p + "conditioner_projection.bias"] for p in pre]
    bo = [P[p + "output_projection.bias"] for p in pre]
    Win, Wsk, Wout = (_bf(P[n + ".weight"][:, :, 0]) for n in ("input_projection", "skip_projection", "output_projection"))
    specb = _bf(spec[:, 0].to(f64).transpose(1, 2))                                      # [B, T, M]
    condb = _bf(cond.to(f64).transpose(1, 2))                                            # [B, T, H]
    # ---- forward
    h0 = torch.relu(specb @ Win.t() + P["input_projection.bias"])
    x = x0 = _bf(h0)
    xd = _bf(h0 + dp[0][:, None])
    xds, ypres, zs, skip = [], [], [], 0
    for l in range(L):
        d = dil[l]
        y = sum(_shift(xd, (j - 1) * d) @ Wdb[l][:, :, j].t() for j in range(3)) + condb @ Wcb[l].t() + b1[l]
        z = _bf(torch.sigmoid(y[..., :C]) * torch.tanh(y[..., C:]))
        o = z @ Wob[l].t() + bo[l]
        xn = (x + o[..., :C]) * RS2
        skip = skip + o[..., C:]
        xds.append(xd), ypres.append(_bf(y)), zs.append(z)
        if l < L - 1:
            x, xd = _bf(xn), _bf(xn + dp[l + 1][:, None])
    Sb = _bf(skip / math.sqrt(L))
    h = _bf(torch.relu(Sb @ Wsk.t() + P["skip_projection.bias"]))
    # ---- backward
    G = {}
    deb = _bf(d_eps[:, 0].to(f64).transpose(1, 2))                                       # [B, T, M]
    dh = _bf(torch.where(h > 0 if h_mask is None else h_mask, deb @ Wout, 0.0))
    dS = _bf(dh @ Wsk / math.sqrt(L))
    G["output_projection.weight"] = torch.einsum("btm,btc->mc", deb, h)[:, :, None]
    G["output_projection.bias"] = deb.sum((0, 1))
    G["skip_projection.weight"] = torch.einsum("btn,btc->nc", dh, Sb)[:, :, None]
    G["skip_projection.bias"] = dh.sum((0, 1))
    u = torch.zeros_like(x0)
    g_cond = 0
    g_dp = torch.empty_like(dp)
    for l in reversed(range(L)):
        d = dil[l]
        do = torch.cat([u, dS], dim=-1)
        dz = do @ Wob[l]
        s, th = torch.sigmoid(ypres[l][..., :C]), torch.tanh(ypres[l][..., C:])
        dy = _bf(torch.cat([dz * th * s * (1 - s), dz * s * (1 - th * th)], dim=-1))
        G[pre[l] + "dilated_conv.weight"] = torch.stack(
            [torch.einsum("btr,btc->rc", dy, _shift(xds[l], (j - 1) * d)) for j in range(3)], dim=2)
        G[pre[l] + "dilated_conv.bias"] = G[pre[l] + "conditioner_projection.bias"] = dy.sum((0, 1))
        G[pre[l] + "conditioner_projection.weight"] = torch.einsum("btr,btk->rk", dy, condb)[:, :, None]
        G[pre[l] + "output_projection.weight"] = torch.einsum("btr,btc->rc", do, zs[l])[:, :, None]
        G[pre[l] + "output_projection.bias"] = do.sum((0, 1))
        # dp_l is added to x_l before the zero padding: every tap that exists at a frame carries it (fp32 weights, as
        # training._stack_backward does)
        g_dp[l] = sum(_shift(dy, (1 - j) * d).sum(1) @ Wd[l][:, :, j] for j in range(3))
        g_cond = g_cond + dy @ Wcb[l]
        g = sum(_shift(dy, (1 - j) * d) @ Wdb[l][:, :, j] for j in range(3)) + u
        u = _bf(g * RS2) if l > 0 else _bf(torch.where(x0 > 0, g, 0.0))
    dpre0 = u
    G["input_projection.weight"] = torch.einsum("btc,btm->cm", dpre0, specb)[:, :, None]
    G["input_projection.bias"] = dpre0.sum((0, 1))
    g_spec = (dpre0 @ Win).transpose(1, 2)[:, None]
    leaves = list(mlp.values()) + dpw + dpb
    grads = torch.autograd.grad(dp_t, leaves, g_dp)
    names = list(mlp) + [p + "diffusion_projection.weight" for p in pre] + [p + "diffusion_projection.bias" for p in pre]
    G.update(zip(names, grads))
    return G, g_spec, g_cond.transpose(1, 2), dict(x0=x0, h=h, hpre=Sb @ Wsk.t() + P["skip_projection.bias"])


def _kernel_relu_outputs(net, spec, t, cond):
    """x0 and h as training._stack_forward stores them (for the mask comparison)."""
    with torch.no_grad():
        layers = net.residual_layers
        e = TR._step_embedding(net, t)
        dp = torch.einsum("bk,lck->lbc", e, torch.stack([ly.diffusion_projection.weight for ly in layers])) + \
            torch.stack([ly.diffusion_projection.bias for ly in layers])[:, None]
        st = lambda name, attr: torch.stack([getattr(getattr(ly, name), attr) for ly in layers])
        _, saved, _ = TR._stack_forward(
            tuple(int(ly.dilation) for ly in layers), spec, cond, dp, st("dilated_conv", "weight"), st("dilated_conv", "bias"),
            st("conditioner_projection", "weight"), st("conditioner_projection", "bias"), st("output_projection", "weight"),
            st("output_projection", "bias"), net.input_projection.weight, net.input_projection.bias,
            net.skip_projection.weight, net.skip_projection.bias, net.output_projection.weight, net.output_projection.bias)
    return saved[5], saved[7]


# (C, H, M, L, B, T, cycle): config 5 of bench.py; the bap stream's width and depth; dilation 8 > T
@pytest.mark.parametrize("C,H,M,L,B,T,cycle", [(256, 256, 60, 20, 6, 1000, 4), (128, 64, 5, 10, 3, 517, 4),
                                               (256, 128, 80, 4, 3, 7, 4)])
def test_diffnet_training_gradients_vs_bf16_faithful_reference(C, H, M, L, B, T, cycle):
    """Every parameter gradient and d spec, d cond of DiffNet in training mode (ordinary initialisation) against
    _reference_grads.

    The reference evaluates sigmoid and tanh exactly where the kernels use tanh.approx.f32, which flips the bf16 rounding
    of a few per cent of z.  Through 20 layers that moves the skip sum by about 1e-3 of its size, and ~0.1 % of the tail
    ReLU's inputs lie that close to zero: there the two forwards take different ReLU branches, and each such element is
    a full-size difference in dh that reaches every gradient (~5e-2 rel-L2 at config 5).  So the test (1) bounds how many
    mask decisions differ and checks that they sit at near-zero inputs, and (2) compares the gradients with the
    reference run on the kernels' own tail mask, which leaves fp32 vs float64 sums and the tanh.approx roundings."""
    from ensemble_svs_with_interactions_b200.diffsinger import DiffNet
    torch.manual_seed(C + L + T)
    m = DiffNet(in_dim=M, encoder_hidden_dim=H, residual_layers=L, residual_channels=C, dilation_cycle_length=cycle)
    with torch.no_grad():
        m.output_projection.weight.normal_(0, 0.05)          # the module's zero init would make every other gradient 0
    m = m.to(DEV).train()
    assert m.resolved_precision() == "bf16"
    g = _gen(T + M)
    spec = torch.randn((B, 1, M, T), generator=g, device=DEV)
    cond = torch.randn((B, H, T), generator=g, device=DEV)
    t = torch.randint(0, 100, (B,), generator=g, device=DEV)
    d_eps = torch.randn((B, 1, M, T), generator=g, device=DEV)
    spec_d, cond_d = spec.clone().requires_grad_(True), cond.clone().requires_grad_(True)
    (m(spec_d, t, cond_d) * d_eps).sum().backward()
    x0k, hk = _kernel_relu_outputs(m, spec, t, cond)

    def errors(h_mask):
        G, g_spec, g_cond, relu = _reference_grads(m, spec, t, cond, d_eps, h_mask)
        e = {n: _rel_l2(p.grad, G[n]) for n, p in m.named_parameters()}
        e["d spec"], e["d cond"] = _rel_l2(spec_d.grad, g_spec), _rel_l2(cond_d.grad, g_cond)
        assert len(e) == len(list(m.parameters())) + 2
        return sorted(e.items(), key=lambda kv: -kv[1]), relu

    own, relu = errors(None)
    ranked, _ = errors(hk > 0)
    flip_x0 = ((x0k > 0) != (relu["x0"] > 0)).sum().item()
    flip_h = (hk > 0) != (relu["h"] > 0)
    hpre = relu["hpre"]
    near = (hpre[flip_h].abs().max() / hpre.pow(2).mean().sqrt()).item() if flip_h.any() else 0.0
    print(f"gradients C={C} L={L} B={B} T={T}: ReLU masks differing: x0 {flip_x0} / {x0k.numel()}, h {flip_h.sum().item()} / "
          f"{hk.numel()} (largest |input| there {near:.2e} rms); with its own masks the reference is off by "
          f"{own[0][1]:.2e} worst, {own[len(own) // 2][1]:.2e} median; on the kernels' tail mask worst " +
          ", ".join(f"{k} {v:.2e}" for k, v in ranked[:4]) + f"; median {ranked[len(ranked) // 2][1]:.2e}")
    assert flip_x0 == 0
    assert flip_h.sum().item() <= MASK_FLIPS * hk.numel() and near <= MASK_NEAR
    assert ranked[0][1] <= GRAD_REL_L2, ranked[:8]
