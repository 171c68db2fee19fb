"""CPU-only: the argument checks of the DiffNet training entries (svsk_seggemm_bf16, svsk_wgrad_bf16,
svsk_ntc_to_nct_bf16, svsk_diffnet_train_pack), all decided before any launch.  The pointers are fake, so every
parameter set below breaks exactly one rule: a set that passed every check would launch on a GPU machine."""
import ctypes as C

import pytest

from ensemble_svs_with_interactions_b200 import _lib, ops

E_ARG, E_ALIGN = -1, -2


def _seg_params(mode=ops.SEG_PLAIN, **kw):
    """A PLAIN launch of 64 output rows over one 64-wide segment, or the given mode's usual operands; kw overrides."""
    p = _lib.SegGemmParams()
    p.nseg, p.x[0], p.ldx[0], p.kx[0], p.wp = 1, 0x10000, 64, 64, 0x20000
    p.Nrows, p.B, p.T, p.mode, p.C, p.init, p.alpha = 64, 1, 8, mode, 64, 1, 1.0
    if mode == ops.SEG_PLAIN or mode == ops.SEG_ADD_SCALE:
        p.out0, p.ld_out0 = 0x30000, 64
    elif mode == ops.SEG_GATE_FWD:
        p.Nrows, p.bias, p.out0, p.ld_out0, p.out1, p.ld_out1 = 256, 0x40000, 0x30000, 256, 0x50000, 128
    elif mode == ops.SEG_GATE_BWD:
        p.Nrows, p.in0, p.ld_in0, p.out0, p.ld_out0 = 128, 0x60000, 256, 0x30000, 256
    elif mode == ops.SEG_RES_SKIP:
        p.Nrows, p.C, p.bias, p.in0, p.ld_in0, p.outf, p.ld_outf = 256, 128, 0x40000, 0x60000, 128, 0x70000, 128
    for k, v in kw.items():
        if k in ("x", "ldx", "kx", "shift"):
            getattr(p, k)[0] = v
        else:
            setattr(p, k, v)
    return p


SEGGEMM_BAD = [
    ("nseg 0", {}, dict(nseg=0), E_ARG, "nseg=0"),
    ("nseg 5", {}, dict(nseg=5), E_ARG, "nseg=5"),
    ("Nrows % 16", {}, dict(Nrows=72), E_ARG, "Nrows=72"),
    ("kx % 64", {}, dict(kx=96, ldx=96), E_ARG, "K=96"),
    ("ldx < kx", {}, dict(ldx=32), E_ARG, "ld=32"),
    ("ldx % 8", {}, dict(ldx=68), E_ARG, "ld=68"),
    ("segment alignment", {}, dict(x=0x10008), E_ALIGN, "not 16-byte aligned"),
    ("GATE_FWD Nrows % 256", dict(mode=ops.SEG_GATE_FWD), dict(Nrows=384), E_ARG, "GATE_FWD"),
    ("GATE_FWD no z", dict(mode=ops.SEG_GATE_FWD), dict(out1=0), E_ARG, "GATE_FWD"),
    ("GATE_FWD no bias", dict(mode=ops.SEG_GATE_FWD), dict(bias=0), E_ARG, "GATE_FWD"),
    ("GATE_FWD ypre pitch", dict(mode=ops.SEG_GATE_FWD), dict(ld_out0=248), E_ARG, "GATE_FWD"),
    ("GATE_FWD z pitch", dict(mode=ops.SEG_GATE_FWD), dict(ld_out1=120), E_ARG, "GATE_FWD"),
    ("GATE_BWD Nrows % 128", dict(mode=ops.SEG_GATE_BWD), dict(Nrows=192), E_ARG, "GATE_BWD"),
    ("GATE_BWD ypre pitch", dict(mode=ops.SEG_GATE_BWD), dict(ld_in0=248), E_ARG, "GATE_BWD"),
    ("GATE_BWD dy pitch", dict(mode=ops.SEG_GATE_BWD), dict(ld_out0=248), E_ARG, "GATE_BWD"),
    ("GATE_BWD no ypre", dict(mode=ops.SEG_GATE_BWD), dict(in0=0), E_ARG, "GATE_BWD"),
    ("RES_SKIP C 64", dict(mode=ops.SEG_RES_SKIP), dict(Nrows=128, C=64), E_ARG, "RES_SKIP"),
    ("RES_SKIP C 192", dict(mode=ops.SEG_RES_SKIP), dict(Nrows=384, C=192), E_ARG, "RES_SKIP"),
    ("RES_SKIP C != Nrows / 2", dict(mode=ops.SEG_RES_SKIP), dict(C=256), E_ARG, "RES_SKIP"),
    ("RES_SKIP ld_outf % 4", dict(mode=ops.SEG_RES_SKIP), dict(ld_outf=130), E_ARG, "RES_SKIP"),
    ("RES_SKIP no skip", dict(mode=ops.SEG_RES_SKIP), dict(outf=0), E_ARG, "RES_SKIP"),
    ("RES_SKIP x pitch", dict(mode=ops.SEG_RES_SKIP), dict(ld_in0=120), E_ARG, "RES_SKIP"),
    ("PLAIN no output", {}, dict(out0=0), E_ARG, "no output"),
    ("ADD_SCALE no output", dict(mode=ops.SEG_ADD_SCALE), dict(out0=0), E_ARG, "no output"),
    ("PLAIN ld_outf % 4", {}, dict(outf=0x70000, ld_outf=66), E_ALIGN, "multiple of 4"),
    ("unknown mode", {}, dict(mode=7), E_ARG, "unknown mode 7"),
    ("out0 pitch % 8", {}, dict(ld_out0=68), E_ALIGN, "multiples of 8"),
    ("out1 pitch % 8", {}, dict(out1=0x50000, ld_out1=68), E_ALIGN, "multiples of 8"),
    ("in0 pitch % 8", {}, dict(in0=0x60000, ld_in0=68), E_ALIGN, "multiples of 8"),
    ("mask pitch % 8", {}, dict(mask=0x60000, ld_mask=68), E_ALIGN, "multiples of 8"),
    ("GATE_BWD dy pitch % 8", dict(mode=ops.SEG_GATE_BWD), dict(ld_out0=260), E_ALIGN, "multiples of 8"),
]


@pytest.mark.parametrize("what,base,bad,rc,msg", SEGGEMM_BAD, ids=[c[0] for c in SEGGEMM_BAD])
def test_seggemm_rejects_before_launch(what, base, bad, rc, msg):
    l = _lib.lib()
    assert l.svsk_seggemm_bf16(C.byref(_seg_params(**base, **bad)), None) == rc, what
    assert msg.encode() in l.svsk_last_error(), l.svsk_last_error()


def _wgrad_params(**kw):
    p = _lib.WgradParams()
    p.p, p.q[0], p.qrows[0], p.dW = 0x10000, 0x20000, 64, 0x30000
    p.nseg, p.Prows, p.B, p.T, p.Tp, p.ldw, p.splits = 1, 128, 1, 64, 64, 64, 1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


WGRAD_BAD = [
    ("nseg 0", dict(nseg=0), E_ARG, "nseg=0"),
    ("nseg 6", dict(nseg=6), E_ARG, "nseg=6"),
    ("Tp % 8", dict(Tp=68, T=64), E_ARG, "Tp=68"),
    ("Tp < T", dict(Tp=64, T=65), E_ARG, "Tp=64"),
    ("no P", dict(p=0), E_ARG, "wgrad_bf16"),
    ("ldw % 4", dict(ldw=66), E_ALIGN, "pitch"),
    ("dW alignment", dict(dW=0x30008), E_ALIGN, "16-byte aligned"),
]


@pytest.mark.parametrize("what,bad,rc,msg", WGRAD_BAD, ids=[c[0] for c in WGRAD_BAD])
def test_wgrad_rejects_before_launch(what, bad, rc, msg):
    l = _lib.lib()
    assert l.svsk_wgrad_bf16(C.byref(_wgrad_params(**bad)), None) == rc, what
    assert msg.encode() in l.svsk_last_error(), l.svsk_last_error()


def test_null_params_are_rejected():
    l = _lib.lib()
    assert l.svsk_seggemm_bf16(None, None) == E_ARG
    assert b"null params" in l.svsk_last_error()
    assert l.svsk_wgrad_bf16(None, None) == E_ARG
    assert b"null params" in l.svsk_last_error()


NTC_BAD = [  # (what, B, T, N, ldx, Tp, out_rows, row0, nshift, msg)
    ("N % 8", 1, 8, 12, 16, 8, 64, 0, 1, "multiples of 8"),
    ("ldx % 8", 1, 8, 16, 20, 8, 64, 0, 1, "multiples of 8"),
    ("ldx < N", 1, 8, 16, 8, 8, 64, 0, 1, "multiples of 8"),
    ("Tp % 8", 1, 12, 16, 16, 12, 64, 0, 1, "multiples of 8"),
    ("Tp < T", 1, 16, 16, 16, 8, 64, 0, 1, "multiples of 8"),
    ("nshift 0", 1, 8, 16, 16, 8, 64, 0, 0, "1..3 shifted copies"),
    ("nshift 4", 1, 8, 16, 16, 8, 64, 0, 4, "1..3 shifted copies"),
    ("rows do not fit", 1, 8, 16, 16, 8, 47, 0, 3, "1..3 shifted copies"),
    ("rows do not fit after row0", 1, 8, 16, 16, 8, 64, 17, 3, "1..3 shifted copies"),
    ("negative row0", 1, 8, 16, 16, 8, 64, -1, 1, "1..3 shifted copies"),
]


@pytest.mark.parametrize("what,B,T,N,ldx,Tp,out_rows,row0,nshift,msg", NTC_BAD, ids=[c[0] for c in NTC_BAD])
def test_ntc_to_nct_rejects_before_launch(what, B, T, N, ldx, Tp, out_rows, row0, nshift, msg):
    l = _lib.lib()
    shifts = (C.c_int * 4)(0, 0, 0, 0)
    assert l.svsk_ntc_to_nct_bf16(0x10000, 0x20000, B, T, N, ldx, Tp, out_rows, row0, nshift, shifts, None) == E_ARG, what
    assert msg.encode() in l.svsk_last_error(), l.svsk_last_error()


@pytest.mark.parametrize("L,Cc,H", [(1, 192, 64), (1, 64, 64), (1, 512, 64), (1, 128, 96), (1, 256, 0), (0, 128, 64)])
def test_diffnet_train_pack_rejects_before_launch(L, Cc, H):
    l = _lib.lib()
    ptrs = [0x10000 * (i + 1) for i in range(8)]
    assert l.svsk_diffnet_train_pack(*ptrs, L, Cc, H, None) == E_ARG
    assert b"need C in {128,256}, H % 64 == 0" in l.svsk_last_error(), l.svsk_last_error()
