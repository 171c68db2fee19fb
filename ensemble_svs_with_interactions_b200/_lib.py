"""ctypes binding of libsvsk.so (include/svsk.h).

There is no fallback: if the library is missing or a call fails, a RuntimeError is raised with the
library's own message (``svsk_last_error``).  PyTorch is only used for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# SVSK_LIB_PATH: A/B measurements of kernel variants on one box (tools/); the product path is the in-tree build
LIB_PATH = os.environ.get("SVSK_LIB_PATH") or os.path.join(_HERE, "csrc", "libsvsk.so")

_lib = None
_lock = threading.Lock()


class Conv1dF32Params(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("in_bias", C.c_void_p),
        ("residual", C.c_void_p), ("idx_past", C.c_void_p), ("idx_future", C.c_void_p), ("y", C.c_void_p),
        ("B", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32), ("T", C.c_int32),
        ("ksize", C.c_int32), ("dilation", C.c_int32), ("tap_origin", C.c_int32), ("pad_mode", C.c_int32),
        ("accumulate", C.c_int32), ("act", C.c_int32), ("in_relu", C.c_int32), ("out_scale", C.c_float),
    ]


class DiffnetBlockParams(C.Structure):
    _fields_ = [
        ("xb_in", C.c_void_p), ("xb_out", C.c_void_p), ("x32", C.c_void_p), ("skip32", C.c_void_p),
        ("cond", C.c_void_p), ("w1p", C.c_void_p), ("woutp", C.c_void_p), ("stepbias", C.c_void_p),
        ("bout", C.c_void_p),
        ("B", C.c_int32), ("T", C.c_int32), ("C", C.c_int32), ("H", C.c_int32),
        ("dilation", C.c_int32), ("stepbias_batch_stride", C.c_int32), ("init_skip", C.c_int32),
        ("write_x", C.c_int32), ("reserved0", C.c_int32),
    ]


class DiffnetStackParams(C.Structure):
    _fields_ = [
        ("xb_in", C.c_void_p), ("edge0", C.c_void_p), ("edge1", C.c_void_p), ("skip32", C.c_void_p),
        ("cond", C.c_void_p), ("w1p", C.c_void_p), ("woutp", C.c_void_p), ("stepbias", C.c_void_p),
        ("bout", C.c_void_p), ("flags", C.c_void_p), ("dilation", C.POINTER(C.c_int32)),
        ("B", C.c_int32), ("T", C.c_int32), ("C", C.c_int32), ("H", C.c_int32), ("L", C.c_int32),
        ("stepbias_batch_stride", C.c_int32), ("stepbias_layer_stride", C.c_int32), ("init_skip", C.c_int32),
        ("pcond_gate", C.c_void_p), ("pcond_filt", C.c_void_p),
    ]


class DiffnetStepParams(C.Structure):
    _fields_ = [
        ("skip32", C.c_void_p), ("x32s", C.c_void_p), ("z", C.c_void_p), ("eps_out", C.c_void_p), ("xb_out", C.c_void_p),
        ("w_skip", C.c_void_p), ("w_out", C.c_void_p), ("w_in", C.c_void_p),
        ("b_skip", C.c_void_p), ("b_out", C.c_void_p), ("b_in", C.c_void_p), ("t", C.c_void_p),
        ("sra", C.c_void_p), ("srm1", C.c_void_p), ("c1", C.c_void_p), ("c2", C.c_void_p), ("plv", C.c_void_p),
        ("skip_scale", C.c_float),
        ("B", C.c_int32), ("T", C.c_int32), ("C", C.c_int32), ("Mp", C.c_int32), ("clip_denoised", C.c_int32),
    ]


class LinearBf16Params(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("y_bf16", C.c_void_p), ("y_f32", C.c_void_p),
        ("N", C.c_int64), ("K", C.c_int32), ("Cout", C.c_int32),
        ("lda", C.c_int32), ("ldy_b", C.c_int32), ("ldy_f", C.c_int32), ("act", C.c_int32),
    ]


class LstmParams(C.Structure):
    _fields_ = [
        ("pre", C.c_void_p), ("w_hh", C.c_void_p), ("lengths", C.c_void_p), ("h_f32", C.c_void_p), ("h_bf16", C.c_void_p),
        ("pre_stride_b", C.c_int64), ("pre_stride_t", C.c_int64), ("pre_stride_r", C.c_int64),
        ("hf_stride_b", C.c_int64), ("hf_stride_t", C.c_int64), ("hf_stride_c", C.c_int64),
        ("hb_stride_b", C.c_int64), ("hb_stride_t", C.c_int64),
        ("B", C.c_int32), ("T", C.c_int32), ("H", C.c_int32), ("ndir", C.c_int32),
    ]


class LstmBwdParams(C.Structure):
    _fields_ = [
        ("dh", C.c_void_p), ("gates", C.c_void_p), ("cell", C.c_void_p), ("w_hh", C.c_void_p), ("lengths", C.c_void_p),
        ("dpre", C.c_void_p), ("B", C.c_int32), ("T", C.c_int32), ("H", C.c_int32), ("ndir", C.c_int32),
    ]


class WgradF32Params(C.Structure):
    _fields_ = [
        ("dy", C.c_void_p), ("x", C.c_void_p), ("dw", C.c_void_p), ("db", C.c_void_p), ("ws", C.c_void_p),
        ("dy_batch_stride", C.c_int64), ("x_batch_stride", C.c_int64),
        ("B", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("T", C.c_int32), ("ksize", C.c_int32), ("origin", C.c_int32),
        ("pad_mode", C.c_int32), ("splits", C.c_int32),
    ]


class TapGemmBf16Params(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("wp", C.c_void_p), ("bias", C.c_void_p), ("y_bf16", C.c_void_p), ("y_f32", C.c_void_p),
        ("B", C.c_int32), ("T", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32), ("ksize", C.c_int32),
        ("Tp_x", C.c_int32), ("ldx", C.c_int32),
        ("Tp_y", C.c_int32), ("y_row0", C.c_int32), ("ldy_b", C.c_int32), ("ldy_f", C.c_int32),
        ("act", C.c_int32),
    ]


class WavenetBlockParams(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("c", C.c_void_p), ("w1t", C.c_void_p), ("b1", C.c_void_p), ("w2t", C.c_void_p), ("b2", C.c_void_p),
        ("x_out", C.c_void_p), ("skips", C.c_void_p),
        ("B", C.c_int32), ("T", C.c_int32), ("R", C.c_int32), ("G", C.c_int32), ("S", C.c_int32), ("Cc", C.c_int32),
        ("ksize", C.c_int32), ("dilation", C.c_int32), ("first", C.c_int32),
    ]


class WavenetArParams(C.Structure):
    _fields_ = [
        ("wpack", C.c_void_p), ("cproj", C.c_void_p), ("u", C.c_void_p), ("y", C.c_void_p), ("logits", C.c_void_p),
        ("hist", C.c_void_p),
        ("B", C.c_int32), ("T", C.c_int32), ("steps", C.c_int32), ("out_dim", C.c_int32), ("R", C.c_int32), ("G", C.c_int32),
        ("S", C.c_int32), ("layers", C.c_int32), ("stacks", C.c_int32), ("ksize", C.c_int32),
    ]


class WavenetArWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "first_v", "first_g", "first_b", "conv_v", "conv_g", "conv_b", "cond_v", "cond_g", "skip_v", "skip_g", "skip_b",
        "out_v", "out_g", "out_b", "last1_v", "last1_g", "last1_b", "last3_v", "last3_g", "last3_b")] + [
        (n, C.c_int32) for n in ("out_dim", "R", "G", "S", "cin", "layers", "stacks", "ksize")]


class WavenetBlockTrainParams(C.Structure):
    _fields_ = [("blk", WavenetBlockParams), ("y", C.c_void_p)]


class WavenetDgradParams(C.Structure):
    _fields_ = [
        ("dy_in", C.c_void_p), ("wT", C.c_void_p), ("g_next", C.c_void_p), ("g_out", C.c_void_p), ("dS", C.c_void_p),
        ("y_prev", C.c_void_p), ("wB", C.c_void_p), ("dy_out", C.c_void_p), ("dy_bstride", C.c_int64),
        ("B", C.c_int32), ("T", C.c_int32), ("R", C.c_int32), ("G", C.c_int32), ("S", C.c_int32), ("ksize", C.c_int32),
        ("dilation", C.c_int32),
    ]


class WavenetWgradParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "x_in", "c", "xs", "ys", "gs", "dy", "dS", "skips", "h1", "dh1", "glog", "dilations", "dW", "ws")] + [
        (n, C.c_int32) for n in ("B", "T", "out_dim", "R", "G", "S", "cin", "layers", "ksize", "splits")]


class SegGemmParams(C.Structure):
    _fields_ = [
        ("x", C.c_void_p * 4), ("ldx", C.c_int32 * 4), ("kx", C.c_int32 * 4), ("shift", C.c_int32 * 4), ("nseg", C.c_int32),
        ("wp", C.c_void_p),
        ("Nrows", C.c_int32), ("B", C.c_int32), ("T", C.c_int32), ("mode", C.c_int32), ("C", C.c_int32), ("init", C.c_int32),
        ("act", C.c_int32), ("accumulate", C.c_int32),
        ("bias", C.c_void_p), ("in0", C.c_void_p), ("ld_in0", C.c_int32), ("mask", C.c_void_p), ("ld_mask", C.c_int32),
        ("dp_next", C.c_void_p), ("out0", C.c_void_p), ("ld_out0", C.c_int32), ("out1", C.c_void_p), ("ld_out1", C.c_int32),
        ("outf", C.c_void_p), ("ld_outf", C.c_int32), ("alpha", C.c_float),
    ]


class WgradParams(C.Structure):
    _fields_ = [
        ("p", C.c_void_p), ("q", C.c_void_p * 5), ("qrows", C.c_int32 * 5), ("shift", C.c_int32 * 5),
        ("nseg", C.c_int32), ("Prows", C.c_int32), ("B", C.c_int32), ("T", C.c_int32), ("Tp", C.c_int32), ("ldw", C.c_int32),
        ("accumulate", C.c_int32), ("splits", C.c_int32), ("split_stride", C.c_int64), ("dW", C.c_void_p),
    ]


class UsfganBlockParams(C.Structure):
    _fields_ = [
        ("xb_in", C.c_void_p), ("xb_out", C.c_void_p), ("aux", C.c_void_p),
        ("w1p", C.c_void_p), ("woutp", C.c_void_p), ("bias1", C.c_void_p), ("bout", C.c_void_p),
        ("idx_past", C.c_void_p), ("idx_future", C.c_void_p),
        ("B", C.c_int32), ("T", C.c_int32), ("A", C.c_int32),
        ("dilation", C.c_int32), ("adaptive", C.c_int32), ("out_scale", C.c_float), ("out_relu", C.c_int32),
        ("aux_u", C.c_void_p), ("aux_q", C.c_void_p), ("q_batch_stride", C.c_int64),
        ("q_ld", C.c_int32), ("q_fpad", C.c_int32), ("hop", C.c_int32), ("reach", C.c_int32),
    ]


class Conv1dBf16Params(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("wp", C.c_void_p), ("bias", C.c_void_p), ("y", C.c_void_p),
        ("B", C.c_int32), ("T", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32),
        ("ksize", C.c_int32), ("dilation", C.c_int32), ("tap_origin", C.c_int32), ("pad_mode", C.c_int32),
        ("act", C.c_int32),
    ]


# name -> argtypes (all return int except where noted)
_V, _I, _F, _Z = C.c_void_p, C.c_int, C.c_float, C.c_size_t
_SIGNATURES = {
    "svsk_version": [],
    "svsk_device_check": [_I],
    "svsk_conv1d_f32": [C.POINTER(Conv1dF32Params), _V],
    "svsk_linear_f32": [_V, _V, _V, _V, _I, _I, _I, _I, _V],
    "svsk_gated_act_f32": [_V, _V, _I, _I, _I, _I, _V],
    "svsk_diffnet_residual_skip_f32": [_V, _V, _V, _I, _I, _I, _I, _V],
    "svsk_scale_act_f32": [_V, _V, _Z, _F, _I, _V],
    "svsk_sinusoidal_embedding_f32": [_V, _V, _I, _I, _V],
    "svsk_ddpm_update_f32": [_V, _V, _V, _V, _V, _V, _V, _V, _V, _V, _I, _Z, _I, _V],
    "svsk_q_sample_f32": [_V, _V, _V, _V, _V, _V, _I, _Z, _V],
    "svsk_plms_transfer_f32": [_V, _V, _V, _V, _I, _V, _I, _Z, _V],
    "svsk_lincomb_f32": [C.POINTER(C.c_void_p), C.POINTER(C.c_float), _I, _V, _Z, _V],
    "svsk_pd_index": [_V, _V, _V, _I, _I, _I, _V],
    "svsk_upsample_smooth_f32": [_V, _V, _V, _I, _I, _I, _V],
    "svsk_periodic_mix_f32": [_V, _V, _V, _V, _V, _V, _Z, _V],
    "svsk_nct_to_ntc": [_V, _V, _V, _I, _I, _I, _I, _V],
    "svsk_ntc_to_nct_f32": [_V, _V, _I, _I, _I, _I, _F, _V],
    "svsk_cast_scale_bf16": [_V, _V, _Z, _F, _I, _V],
    "svsk_diffnet_block3_bf16": [C.POINTER(DiffnetBlockParams), _V],
    "svsk_diffnet_stack_bf16": [C.POINTER(DiffnetStackParams), _V],
    "svsk_diffnet_stack_fits": [C.c_int, C.c_int, C.c_int, C.c_int],
    "svsk_diffnet_stack_uses_pcond": [C.c_int, C.c_int, C.c_int, C.c_int],
    "svsk_diffnet_cond_project_bf16": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p],
    "svsk_diffnet_pcond_pack_bf16": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p],
    "svsk_diffnet_step_bf16": [C.POINTER(DiffnetStepParams), _V],
    "svsk_upsample_fused": [_V, _V, C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int, C.c_int, _V, _V, C.c_int, _V],
    "svsk_expand1_bf16": [_V, C.c_longlong, _V, _V, _V, C.c_int, C.c_int, C.c_int, _V],
    "svsk_diffnet_pack_block": [_V, _V, _V, _V, _V, _I, _I, _V],
    "svsk_wavenet_block_f32": [C.POINTER(WavenetBlockParams), _V],
    "svsk_wavenet_ar_f32": [C.POINTER(WavenetArParams), _V],
    "svsk_wavenet_ar_supported": [_I, _I, _I, _I, _I, _I, _I],
    "svsk_wavenet_ar_sizes": [_I, _I, _I, _I, _I, _I, _I, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)],
    "svsk_wavenet_ar_pack_f32": [C.POINTER(WavenetArWeights), _V, _V, _V],
    "svsk_wavenet_block_train_f32": [C.POINTER(WavenetBlockTrainParams), _V],
    "svsk_wavenet_train_sizes": [_I, _I, _I, _I, _I, _I, _I, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)],
    "svsk_wavenet_train_pack_f32": [C.POINTER(WavenetArWeights), _V, _V],
    "svsk_wavenet_dgrad_f32": [C.POINTER(WavenetDgradParams), _V],
    "svsk_wavenet_wgrad_f32": [C.POINTER(WavenetWgradParams), _V],
    "svsk_wavenet_wnorm_grad_f32": [C.POINTER(WavenetArWeights), _V, _V, _V],
    "svsk_relu_mask_f32": [_V, _V, _V, C.c_longlong, _V],
    "svsk_usfgan_source": [_V, _V, _V, C.c_longlong, _V, _V, _I, _I, _I, _I, _I, _F, _F, _V],
    "svsk_seggemm_bf16": [C.POINTER(SegGemmParams), _V],
    "svsk_wgrad_bf16": [C.POINTER(WgradParams), _V],
    "svsk_ntc_to_nct_bf16": [_V, _V, _I, _I, _I, _I, _I, _I, _I, _I, C.POINTER(C.c_int), _V],
    "svsk_diffnet_train_pack": [_V, _V, _V, _V, _V, _V, _V, _V, _I, _I, _I, _V],
    "svsk_diffnet_packed_row": [_I, _I],
    "svsk_linear_bf16": [C.POINTER(LinearBf16Params), _V],
    "svsk_usfgan_block_bf16": [C.POINTER(UsfganBlockParams), _V],
    "svsk_usfgan_pack_block": [_V, _V, _V, _V, _V, _I, _I, _I, _V],
    "svsk_usfgan_aux_frames": [_V, _V, _V, _I, _I, _I, _I, _I, _I, _V],
    "svsk_usfgan_aux_weights": [_V, _V, _I, _I, _I, _V],
    "svsk_upsample_frames_bf16": [_V, _V, _V, _I, _I, _I, _I, _I, _I, _I, _V],
    "svsk_usfgan_frame_base": [_I, _I, _I],
    "svsk_ntc_bf16_to_nct_f32": [_V, _V, _I, _I, _I, _I, _V],
    "svsk_conv1d_bf16": [C.POINTER(Conv1dBf16Params), _V],
    "svsk_conv1d_pack_bf16": [_V, _V, _I, _I, _I, _V],
    "svsk_periodic_mix_bf16": [_V, _V, _V, _V, _Z, _V],
    "svsk_dot_rows_bf16": [_V, _V, _F, _V, _Z, _I, _V],
    "svsk_lstm_f32": [C.POINTER(LstmParams), _V],
    "svsk_lstm_supported": [C.c_int],
    "svsk_tapgemm_bf16": [C.POINTER(TapGemmBf16Params), _V],
    "svsk_tapgemm_pack_bf16": [_V, _V, _V, _I, _I, _I, _V],
    "svsk_reflect_pad_rows_bf16": [_V, _I, _I, _I, _I, _I, _V],
    "svsk_bn_batch_stats_f32": [_V, _I, _I, _I, _V, _V, _V, _V, _F, _V],
    "svsk_bn_apply_f32": [_V, _V, _V, _V, _V, _V, _F, _I, _I, _I, _I, _V],
    "svsk_encoder_front": [_V, _V, _V, C.c_longlong, _I, _I, _I, _I, _I, _V],
    "svsk_lstm_train_f32": [C.POINTER(LstmParams), _V, _V, _V],
    "svsk_lstm_bwd_f32": [C.POINTER(LstmBwdParams), _V],
    "svsk_wgrad_f32": [C.POINTER(WgradF32Params), _V],
    "svsk_bn_relu_bwd_f32": [_V, _V, _V, _V, _V, _V, _F, _V, _V, _V, _I, _I, _I, _V],
    "svsk_reflect_fold_f32": [_V, _V, _V, _I, _I, _I, _I, _I, _V],
    "svsk_filtfilt_f32": [_V, _V, _V, _V, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), _I, _I, _I, _I, _I, _I, _V],
    "svsk_variance_scaling_f32": [_V, _V, _V, _V, _V, _I, _I, _I, _I, _V],
    "svsk_scale_features_f32": [_V, _V, _V, _V, _I, C.c_longlong, _I, _V],
    "svsk_mdn_head_f32": [_V, _V, _V, _V, _V, _V, C.c_longlong, _I, _I, _I, _V],
}
EXPORTED_SYMBOLS = ["svsk_last_error"] + list(_SIGNATURES)


def lib() -> C.CDLL:
    """Loads libsvsk.so (once).  Raises if it has not been built — there is no other code path."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} not found: build it with `python -m ensemble_svs_with_interactions_b200.csrc.build` "
                    "(or __graft_entry__.build()).  This package has no CPU or PyTorch fallback.")
            l = C.CDLL(LIB_PATH)
            l.svsk_last_error.restype = C.c_char_p
            l.svsk_last_error.argtypes = []
            for name, args in _SIGNATURES.items():
                fn = getattr(l, name)
                fn.argtypes = args
                fn.restype = C.c_int
            _lib = l
    return _lib


launch_count = 0  # successful libsvsk kernel enqueues of this process (bench.py's gpu_launches evidence)


def check(rc: int, what: str) -> None:
    global launch_count
    launch_count += 1
    if rc != 0:
        msg = lib().svsk_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libsvsk {what} failed (code {rc}): {msg}")


def stream_ptr() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t, dtype=None, name="tensor"):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: libsvsk has no CPU path")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous, got strides {t.stride()} for shape {tuple(t.shape)}")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"{name} must be {dtype}, got {t.dtype}")
    return C.c_void_p(t.data_ptr())
