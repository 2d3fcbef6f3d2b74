"""ctypes binding of liba2f_sm100.so (the C-ABI declared in include/a2f.h).

Only plain pointers, sizes and the CUDA stream handle cross this boundary; torch is used by the callers for device
memory and streams.  There is no fallback: if the library is missing, load() raises; on a non-sm_100 device every
compute entry point returns A2F_EARCH and check() raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liba2f_sm100.so")

A2F_OK, A2F_EINVAL, A2F_EARCH, A2F_ECUDA = 0, -1, -2, -3
F32, BF16, I16 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_GELU, ACT_TANH = 0, 1, 2, 3
SIMT_F32, TCGEN05 = 0, 1
RESID_ADD, RESID_DACT = 0, 1

c_void_p, c_int, c_ll, c_float, c_size_t = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_size_t


class A2FError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("M", c_int), ("N", c_int), ("K", c_int),
        ("A", c_void_p), ("a_dtype", c_int),
        ("a_row_stride", c_ll), ("a_batch_stride", c_ll), ("rows_per_batch", c_int),
        ("W", c_void_p), ("ldw", c_ll),
        ("bias", c_void_p), ("act", c_int),
        ("resid", c_void_p), ("resid_dtype", c_int), ("ldr", c_ll),
        ("tmpl", c_void_p), ("rows_per_tmpl", c_int),
        ("C", c_void_p), ("c_dtype", c_int), ("ldc", c_ll), ("c_batch_stride", c_ll),
        ("a_rows", c_int), ("n_seg", c_int), ("seg_row_off", c_int * 4), ("seg_col_off", c_int * 4),
        ("r_batch_stride", c_ll), ("resid_mode", c_int),
        ("C2", c_void_p), ("ldc2", c_ll),
    ]


class WgradArgs(C.Structure):
    _fields_ = [
        ("M", c_int), ("N", c_int), ("K", c_int), ("dtype", c_int),
        ("dY", c_void_p), ("dy_row_stride", c_ll), ("dy_batch_stride", c_ll),
        ("X", c_void_p), ("x_row_stride", c_ll), ("x_batch_stride", c_ll),
        ("rows_per_batch", c_int), ("x_rows", c_int), ("n_seg", c_int),
        ("x_row_off", c_int * 4), ("x_col_off", c_int * 4),
        ("dW", c_void_p), ("ldw", c_ll), ("x_row_step", c_int),
    ]


class CopyJob(C.Structure):
    """a2f_copy_job of include/a2f.h (one strided 2-D copy of an a2f_strided_copy_jobs launch)."""
    _fields_ = [
        ("src", c_void_p), ("dst", c_void_p), ("ld_r", c_ll), ("ld_c", c_ll), ("ldo_r", c_ll), ("ldo_c", c_ll),
        ("R", c_int), ("C", c_int), ("dst_dtype", c_int), ("tile0", c_int),
    ]


class EncoderBlockArgs(C.Structure):
    """a2f_encoder_block_args (include/a2f.h)"""
    _fields_ = [
        ("M", c_int), ("N", c_int), ("F", c_int),
        ("att", c_void_p), ("ld_att", c_ll), ("wo", c_void_p), ("ld_wo", c_ll), ("bo", c_void_p),
        ("h_in", c_void_p), ("ld_hin", c_ll), ("ln1_g", c_void_p), ("ln1_b", c_void_p),
        ("h1", c_void_p), ("ld_h1", c_ll),
        ("w1", c_void_p), ("ld_w1", c_ll), ("b1", c_void_p),
        ("f", c_void_p), ("ld_f", c_ll),
        ("w2", c_void_p), ("ld_w2", c_ll), ("b2", c_void_p),
        ("ln2_g", c_void_p), ("ln2_b", c_void_p),
        ("h_out", c_void_p), ("ld_hout", c_ll),
        ("wq", c_void_p), ("ld_wq", c_ll), ("bq", c_void_p), ("NQ", c_int),
        ("qkv", c_void_p), ("ld_qkv", c_ll),
        ("eps", c_float),
    ]


class DropoutArgs(C.Structure):
    """a2f_dropout_args (include/a2f.h): drop probability, site id, device pointer to {seed, offset} (int64 x 2)."""
    _fields_ = [("p", c_float), ("site", C.c_uint), ("seed_offset_dev", c_void_p)]


# site ids of the encoder dropout RNG contract (include/a2f.h): 8 * layer + kind, and the two pre-layer sites
DROP_ATTN_PROB, DROP_ATTN_OUT, DROP_FFN_ACT, DROP_FFN_OUT = 0, 1, 2, 3
DROP_FEAT_PROJ, DROP_ENC_IN = 96, 97


class DecoderWeights(C.Structure):
    _names = [
        "sa_in_w", "sa_in_b", "sa_out_w", "sa_out_b", "ca_in_w", "ca_in_b", "ca_out_w", "ca_out_b",
        "lin1_w", "lin1_b", "lin2_w", "lin2_b", "n1_w", "n1_b", "n2_w", "n2_b", "n3_w", "n3_b",
        "fb_w", "fb_b", "obj_w", "pe", "fold_w", "fold_pe",
    ]
    _fields_ = [(n, c_void_p) for n in _names]


class VocaWeights(C.Structure):
    _fields_ = [
        ("conv_w", c_void_p * 4), ("conv_b", c_void_p * 4),
        ("fc_w", c_void_p * 3), ("fc_b", c_void_p * 3),
    ]


_SIGNATURES = {
    # name: (restype, argtypes)
    "a2f_version": (c_int, []),
    "a2f_status_string": (C.c_char_p, [c_int]),
    "a2f_last_error": (C.c_char_p, []),
    "a2f_device_check": (c_int, []),
    "a2f_launch_count": (c_ll, []),
    "a2f_gemm": (c_int, [C.POINTER(GemmArgs), c_int, c_void_p]),
    "a2f_gemm_wgrad": (c_int, [C.POINTER(WgradArgs), c_int, c_void_p]),
    "a2f_gemm_ln": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_float, c_void_p, c_ll,
                            c_void_p, c_ll, c_int, c_int, c_int, c_void_p]),
    "a2f_encoder_block": (c_int, [C.POINTER(EncoderBlockArgs), c_void_p]),
    "a2f_posconv": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "a2f_pack_posconv_weight": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "a2f_pack_conv1d_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "a2f_cast_f32_to_bf16": (c_int, [c_void_p, c_void_p, c_ll, c_void_p]),
    "a2f_cast_bf16_to_f32": (c_int, [c_void_p, c_void_p, c_ll, c_void_p]),
    "a2f_split_bf16x3": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_void_p]),
    "a2f_audio_stats": (c_int, [c_void_p, c_int, c_ll, c_void_p, c_void_p]),
    "a2f_conv0_workspace_bytes": (c_size_t, [c_int, c_ll]),
    "a2f_conv0_gn_gelu": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_ll,
                                  c_void_p, c_size_t, c_void_p]),
    "a2f_conv0_auto_workspace_bytes": (c_size_t, [c_int, c_ll]),
    "a2f_conv0_gn_gelu_auto": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_ll,
                                       c_void_p, c_size_t, c_void_p]),
    "a2f_interp_ln": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_int, c_int,
                              c_int, c_void_p]),
    "a2f_layernorm": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_float, c_void_p, c_int, c_void_p, c_int, c_ll,
                              c_int, c_void_p]),
    "a2f_mha_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "a2f_mha_fwd_lse": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "a2f_mha_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float,
                            c_void_p, c_size_t, c_void_p]),
    "a2f_mha_fwd_train": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "a2f_mha_bwd_train": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                  c_float, c_void_p, c_size_t, c_void_p]),
    "a2f_mha_fwd_train_dropout": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float,
                                          C.POINTER(DropoutArgs), c_void_p]),
    "a2f_mha_bwd_train_dropout": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                          c_int, c_float, C.POINTER(DropoutArgs), c_void_p, c_size_t, c_void_p]),
    "a2f_decoder_workspace_bytes": (c_size_t, [c_int, c_int]),
    "a2f_decoder_rollout_ca": (c_int, [C.POINTER(DecoderWeights), c_void_p, c_void_p, c_int, c_int, c_void_p, c_int,
                                    c_int, c_void_p, c_size_t, c_void_p]),
    "a2f_decoder_rollout": (c_int, [C.POINTER(DecoderWeights), c_void_p, c_void_p, c_int, c_int, c_void_p, c_int,
                                    c_int, c_void_p, c_size_t, c_void_p]),
    "a2f_decoder_rollout_stream": (c_int, [C.POINTER(DecoderWeights), c_void_p, c_void_p, c_int, c_int, c_void_p, c_int,
                                           c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "a2f_vertex_head_stream_rows": (c_int, [c_int, c_int]),
    "a2f_vertex_head_stream": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                       c_int, c_void_p]),
    "a2f_decoder_save_offset": (c_int, [c_int]),
    "a2f_decoder_rollout_train": (c_int, [C.POINTER(DecoderWeights), c_void_p, c_void_p, c_int, c_int, c_void_p, c_int,
                                          c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "a2f_decoder_grad_offset": (c_int, [c_int]),
    "a2f_decoder_bwd_workspace_bytes": (c_size_t, [c_int, c_int]),
    "a2f_decoder_rollout_bwd": (c_int, [C.POINTER(DecoderWeights), c_void_p, c_void_p, c_int, c_void_p, c_int, c_int,
                                        c_void_p, c_size_t, c_void_p]),
    "a2f_ln64_param_grad": (c_int, [c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_void_p]),
    "a2f_pack_feedback": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "a2f_pack_decoder_fold": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "a2f_pack_cross_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int,
                                         c_void_p, c_void_p]),
    "a2f_voca_trunk": (c_int, [C.POINTER(VocaWeights), c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                               c_void_p]),
    "a2f_a2m_assemble": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "a2f_channel_affine": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_ll, c_ll, c_ll, c_ll, c_void_p]),
    "a2f_voca_loss_workspace_bytes": (c_size_t, []),
    "a2f_voca_loss_fwd": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_float, c_float, c_void_p, c_void_p, c_size_t,
                                  c_void_p]),
    "a2f_voca_loss_bwd": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p]),
    "a2f_vertex_head_loss_workspace_bytes": (c_size_t, []),
    "a2f_vertex_head_loss": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_ll, c_int, c_float, c_float,
                                     c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_size_t, c_void_p]),
    "a2f_debug_set_umma_field": (c_int, [c_int, C.c_uint]),
    "a2f_debug_set_timeline": (c_int, [c_void_p]),
    "a2f_debug_set_decoder_timing": (c_int, [c_void_p]),
    "a2f_act_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_ll, c_int, c_void_p]),
    "a2f_act_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_ll, c_int, c_void_p]),
    "a2f_cast_rows": (c_int, [c_void_p, c_int, c_ll, c_void_p, c_int, c_ll, c_ll, c_int, c_void_p]),
    "a2f_strided_copy_jobs": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "a2f_transpose_cast": (c_int, [c_void_p, c_ll, c_ll, c_int, c_int, c_void_p, c_int, c_ll, c_void_p]),
    "a2f_add_strided3": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_void_p]),
    "a2f_colsum": (c_int, [c_void_p, c_int, c_ll, c_ll, c_int, c_void_p, c_void_p]),
    "a2f_dropout_mask": (c_int, [C.POINTER(DropoutArgs), c_ll, c_void_p, c_void_p]),
    "a2f_dropout_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_ll, C.POINTER(DropoutArgs), c_void_p]),
    "a2f_spec_mask_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_ll, c_int, c_void_p]),
    "a2f_spec_mask_bwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_ll, c_int, c_void_p]),
    "a2f_layernorm_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_float, c_void_p, c_int, c_void_p,
                                  c_void_p, c_void_p, c_ll, c_int, c_void_p]),
    "a2f_interp_ln_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int, c_void_p]),
    "a2f_conv0_gn_offset": (c_size_t, [c_int, c_ll]),
    "a2f_conv0_bwd_workspace_bytes": (c_size_t, [c_int]),
    "a2f_conv0_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_ll,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "a2f_weight_norm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "a2f_pack_posconv_dgrad_weight": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "a2f_posconv_dgrad": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "a2f_posconv_pre": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "a2f_posconv_wgrad": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    "a2f_voca_assemble": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "a2f_bn_train_stats": (c_int, [c_void_p, c_int, c_ll, c_ll, c_ll, c_ll, c_void_p, c_void_p, c_float, c_float, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "a2f_affine_act": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll,
                               c_void_p]),
    "a2f_bn_train_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_ll, c_ll, c_ll, c_ll, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "a2f_bn_frozen_stats": (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "a2f_bn_frozen_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_ll, c_ll, c_ll, c_ll, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "a2f_mfcc_frames": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "a2f_mfcc_mel_db": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "a2f_mfcc_dct_resize": (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                    c_void_p]),
    "a2f_audio_fragments": (c_int, [c_void_p, c_int, c_ll, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "a2f_resample_sinc": (c_int, [c_void_p, c_int, c_ll, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_ll, c_void_p]),
    "a2f_colsum3": (c_int, [c_void_p, c_int, c_ll, c_ll, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "a2f_im2col1d_split": (c_int, [c_void_p, c_ll, c_ll, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                   c_void_p, c_void_p]),
    "a2f_a2m_mlp": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                            c_void_p, c_int, c_void_p, c_int, c_int, c_void_p]),
    "a2f_bilinear_cl": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "a2f_im2col1d": (c_int, [c_void_p, c_ll, c_ll, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                             c_void_p]),
    "a2f_transpose_batched": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "a2f_lstm_recurrence": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "a2f_song2face_resize": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "a2f_lstm_recurrence_train": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "a2f_lstm_bptt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "a2f_col2im1d": (c_int, [c_void_p, c_ll, c_ll, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                             c_void_p]),
    "a2f_song2face_resize_bwd": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "a2f_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_float, c_float, c_float, c_float, c_float,
                              c_int, c_float, c_void_p]),
    "a2f_adam_step_bf16g": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_float, c_float, c_float, c_float, c_float,
                                    c_int, c_float, c_void_p]),
    "a2f_adam_step_dev": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_ll, c_float, c_float, c_float, c_float, c_float,
                                  c_void_p, c_float, c_void_p]),
}

DEC_SAVE_FIELDS = ("X", "Q", "K", "V", "CTX", "Y1PRE", "Y2PRE", "Y2", "HID", "Y3PRE", "LSE")      # a2f.h A2F_DEC_*
DEC_GRAD_FIELDS = ("GD", "G3", "GHID", "GY2", "G2", "G1", "GQKV", "DEFB")                        # a2f.h A2F_DECG_*

_lib = None


def load() -> C.CDLL:
    """Load the shared library (building is build.py's job) and attach the signatures."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise A2FError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU/PyTorch fallback for the hot path)"
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name, None)
        if fn is None:
            continue  # reported by tests/test_abi.py; callers of a missing symbol fail loudly with AttributeError
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != A2F_OK:
        lib = load()
        msg = lib.a2f_last_error().decode(errors="replace")
        name = lib.a2f_status_string(status).decode(errors="replace")
        raise A2FError(f"{what or 'a2f call'} failed: {name}: {msg}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
