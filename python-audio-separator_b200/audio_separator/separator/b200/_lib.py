"""ctypes binding of the C-ABI library (include/b200sep.h).  This is the stub a reference maintainer would add.

There is NO fallback: if libb200sep.so is missing or fails to load, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_PKG_ROOT = os.path.abspath(os.path.join(_HERE, "..", "..", ".."))  # python-audio-separator_b200/
LIB_PATH = os.environ.get("B200SEP_LIB", os.path.join(_PKG_ROOT, "libb200sep.so"))

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"libb200sep.so not found at {LIB_PATH}: build it with `python python-audio-separator_b200/build.py` "
        "(the B200 engine has no CPU / PyTorch fallback)"
    )
lib = C.CDLL(LIB_PATH)

LAYOUT_CFT = 0
LAYOUT_CTF = 1

i32, i64, f32, vp = C.c_int, C.c_int64, C.c_float, C.c_void_p


class MdxNetConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("dim_c", "dim_f", "dim_t", "num_blocks", "l", "g", "k", "bn", "max_batch", "precision")]


class TfcNetConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("dim_f", "dim_t", "num_subbands", "audio_channels", "num_scales", "l", "c", "g", "bn", "num_targets", "max_batch")]


_SIGS = {
    "b200sep_abi_version": (i32, []),
    "b200sep_last_error": (C.c_char_p, []),
    "b200sep_launch_count": (C.c_uint64, []),
    "b200sep_stft_plan_create": (i32, [C.POINTER(vp), i32, i32]),
    "b200sep_stft_plan_destroy": (None, [vp]),
    "b200sep_stft_forward": (i32, [vp, vp, i64, i64, i64, i32, i32, i32, i32, i32, vp, vp]),
    "b200sep_stft_inverse_work_floats": (i64, [vp, i32, i32, i32, i32]),
    "b200sep_stft_inverse": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp]),
    "b200sep_demix_overlap_add": (i32, [vp, i32, i32, i64, i64, i64, i64, i32, f32, vp, f32, i32, vp, vp, vp]),
    "b200sep_demix_overlap_add_range": (i32, [vp, i32, i32, i32, i32, i64, i64, i64, i64, i64, i64, i32, f32, vp, f32, i32, vp, vp, vp]),
    "b200sep_demix_overlap_add_range_ex": (i32, [vp, i32, i32, i32, i32, i64, i64, i64, i64, i64, i64, i32, f32, vp, i64, i64, f32, i32, vp, vp, i64, vp]),
    "b200sep_absmax": (i32, [vp, i64, vp, vp]),
    "b200sep_normalize": (i32, [vp, i64, vp, f32, f32, vp, vp]),
    "b200sep_to_pcm16": (i32, [vp, i64, vp, vp]),
    "b200sep_to_pcm_bytes": (i32, [vp, i64, i32, i32, vp, vp]),
    "b200sep_mdxnet_param_count": (i64, [C.POINTER(MdxNetConfig)]),
    "b200sep_mdxnet_create": (i32, [C.POINTER(vp), C.POINTER(MdxNetConfig), vp, i64]),
    "b200sep_mdxnet_destroy": (None, [vp]),
    "b200sep_mdxnet_device_bytes": (i64, [vp]),
    "b200sep_mdxnet_forward": (i32, [vp, vp, vp, i32, i32, vp]),
    "b200sep_mdxnet_profile_enable": (i32, [vp, i32]),
    "b200sep_mdxnet_profile_read": (i32, [vp, i32, vp, vp, vp, vp]),
    "b200sep_mdxnet_profile_name": (C.c_char_p, [i32]),
    "b200sep_tfcnet_param_count": (i64, [C.POINTER(TfcNetConfig)]),
    "b200sep_tfcnet_create": (i32, [C.POINTER(vp), C.POINTER(TfcNetConfig), vp, i64]),
    "b200sep_tfcnet_destroy": (None, [vp]),
    "b200sep_tfcnet_device_bytes": (i64, [vp]),
    "b200sep_tfcnet_forward": (i32, [vp, vp, vp, i32, vp]),
    "b200sep_rect_overlap_add": (i32, [vp, i32, i32, i32, i64, i64, i64, f32, vp, vp]),
    "b200sep_rect_overlap_add_range": (i32, [vp, i32, i32, i32, i32, i32, i64, i64, i64, i64, i64, f32, vp, i64, i64, vp]),
    "b200sep_stft_forward_ex": (i32, [vp, vp, i64, i64, i64, i32, i32, i32, i32, f32, i32, i32, i32, i32, vp, vp]),
    "b200sep_stft_inverse_ex": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, vp, vp, vp]),
    "b200sep_conv2d_f32": (i32, [vp, vp, vp, vp, vp] + [i32] * 23 + [vp, vp]),
    "b200sep_lstm_bidir_f32": (i32, [vp, vp, vp, i32, i32, i32, vp]),
    "b200sep_add_rowvec_f32": (i32, [vp, vp, i32, i32, i64, vp]),
    "b200sep_groupnorm_work_floats": (i64, [i32, i32, i32, i64]),
    "b200sep_groupnorm_f32": (i32, [vp, vp, vp, vp, i32, i32, i32, i64, i32, vp, vp]),
    "b200sep_lstm_bidir_wide_f32": (i32, [vp, vp, vp, i32, i32, i32, vp]),
    "b200sep_lstm_frames_gather_f32": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    "b200sep_lstm_frames_scatter_f32": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    "b200sep_local_state_attn_f32": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200sep_tc_packed_floats": (i64, [i32, i32]),
    "b200sep_tc_pack_linear_weights": (i32, [vp, i32, i32, i32, vp, vp]),
    "b200sep_tc_pack_conv_weights": (i32, [vp, i32, i32, i32, vp, vp]),
    "b200sep_groupnorm1_work_floats": (i64, [i32, i32, i32, i64]),
    "b200sep_groupnorm1_f32": (i32, [vp, vp, vp, vp, i32, i32, i32, i64, i32, i32, vp, vp]),
    "b200sep_permute4_f32": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    "b200sep_glu_f32": (i32, [vp, vp, vp, vp, i32, i32, i64, vp]),
    "b200sep_layernorm_f32": (i32, [vp, vp, vp, vp, i64, i32, vp]),
    "b200sep_gemm_f32": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i64, i64, i64, f32, vp, vp, i32, vp, vp, vp, vp]),
    "b200sep_softmax_rows_f32": (i32, [vp, i64, i32, i64, vp]),
    "b200sep_attention_f32": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, i64, i64, i64, i64, i64, i64, i64, i64, f32, i32, vp, vp]),
    "b200sep_attention_work_floats": (i64, [i32, i32, i32, i32]),
    "b200sep_ew_f32": (i32, [vp, vp, vp, i64, f32, f32, i32, vp]),
    "b200sep_meanstd_f32": (i32, [vp, i64, vp, vp]),
    "b200sep_meanstd_work_floats": (i64, [i32]),
    "b200sep_meanstd_batch_f32": (i32, [vp, i64, i32, i64, vp, i32, vp, vp]),
    "b200sep_dconv_work_floats": (i64, [i32, i32, i32, i64, i32]),
    "b200sep_dconv_f32": (i32, [vp] * 11 + [i32, i32, i32, i64, i32, i32, vp, vp, vp]),
    "b200sep_triangle_overlap_add": (i32, [vp, i32, i32, i32, i64, i64, i64, i64, f32, vp, i32, vp, vp]),
    "b200sep_triangle_overlap_add_range": (i32, [vp, i32, i32, i32, i32, i32, i64, i64, i64, i64, f32, vp, i32, vp, i64, i64, vp]),
    "b200sep_dwconv3x3_f32": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "b200sep_upsample2x_bilinear_f32": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp]),
    "b200sep_mean_h_f32": (i32, [vp, vp, i32, i32, i32, vp]),
    "b200sep_copy4_f32": (i32, [vp, vp, i32, i32, i32, i32] + [i64] * 8 + [vp]),
    "b200sep_bin_gain_f32": (i32, [vp, vp, i32, i32, i32, vp]),
    "b200sep_vr_magnitude_pad": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "b200sep_vr_apply_mask": (i32, [vp, i32, vp, i32, i32, i32, f32, f32, f32, f32, vp, vp, vp]),
    "b200sep_vr_mask_pow": (i32, [vp, i32, i32, i32, i32, f32, f32, f32, f32, vp]),
    "b200sep_vr_frame_min": (i32, [vp, i32, i32, i32, vp, vp]),
    "b200sep_vr_mask_merge": (i32, [vp, vp, i32, i32, i32, vp]),
    "b200sep_vr_mirror_high_end": (i32, [vp, i32, vp, i32, i32, vp, i32, i32, i32, i32, i32, vp]),
    "b200sep_resample_poly_f32": (i32, [vp, vp, i32, i32, i32, i64, i32, i64, i64, vp, vp]),
    "b200sep_rmsnorm_f32": (i32, [vp, vp, vp, i64, i32, i64, i64, vp]),
    "b200sep_rope_split_heads_f32": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    "b200sep_gemm_kn_f32": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i64, i64, i64, f32, vp]),
    "b200sep_gate_merge_heads_f32": (i32, [vp, vp, vp, i32, i32, i32, i32, vp]),
    "b200sep_glu_rows_f32": (i32, [vp, vp, i64, i32, i64, i64, vp]),
    "b200sep_roformer_mask_apply": (i32, [vp, vp, vp, i32, i32, i32, i32, vp]),
    "b200sep_gather_pairs_f32": (i32, [vp, vp, vp, i64, i32, i32, vp]),
    "b200sep_mask_average_f32": (i32, [vp, vp, vp, vp, i64, i32, i32, vp]),
    "b200sep_overlap_add_starts": (i32, [vp, vp, vp, i32, i32, i32, i64, vp, vp]),
    "b200sep_overlap_add_starts_range": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i64, i64, i64, vp, i64, i64, vp]),
    "b200sep_ensemble_f32": (i32, [vp, i32, i64, vp, i32, vp, vp]),
    "b200sep_ensemble_spec_abs": (i32, [vp, i32, i64, i32, i32, vp, vp]),
    "b200sep_selftest_umma_gemm": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, i32, vp]),
    "b200sep_selftest_umma_conv3x3": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, i32, vp]),
    "b200sep_selftest_umma_updown": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, i32, i32, vp]),
    "b200sep_selftest_umma_ex": (i32, [i32, vp, vp, vp, vp, vp] + [i32] * 9 + [vp]),
    "b200sep_selftest_instnorm_act": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i64, i32, vp]),
    "b200sep_capture_begin": (i32, [vp]),
    "b200sep_capture_end": (i32, [vp, vp]),
    "b200sep_graph_launch": (i32, [vp, vp]),
    "b200sep_graph_destroy": (None, [vp]),
    "b200sep_mdx_run_model_work_floats": (i64, [vp, i32, i32, i32]),
    "b200sep_mdx_run_model": (i32, [vp, vp, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, vp]),
}
EXPORTED = tuple(_SIGS)
for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name)  # AttributeError here = the library does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args

if lib.b200sep_abi_version() != 1:
    raise ImportError("libb200sep.so ABI version mismatch")


class B200SepError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        raise B200SepError(f"{what} failed (rc={rc}): {lib.b200sep_last_error().decode(errors='replace')}")


def launch_count() -> int:
    return int(lib.b200sep_launch_count())
