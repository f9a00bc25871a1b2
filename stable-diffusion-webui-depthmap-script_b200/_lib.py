"""ctypes binding of include/depthmap_b200.h.  Fails loudly: no library -> ImportError-like RuntimeError, no GPU -> RuntimeError."""
from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DEPTHMAP_B200_LIB", os.path.join(_HERE, "_native", "libdepthmap_b200.so"))

DM_OK, DM_E_INVALID, DM_E_CUDA, DM_E_OOM, DM_E_UNSUPPORTED, DM_E_WORKSPACE = 0, -1, -2, -3, -4, -5
DM_DEPTH_U16, DM_DEPTH_ND64 = 0, 1
DM_FILL = {"none": 0, "naive": 1, "naive_interpolating": 2, "polylines_soft": 3, "polylines_sharp": 4}
DM_EYE_WARP, DM_EYE_IDENTITY, DM_EYE_SKIP = 0, 1, 2
DM_PACK_STRIDED, DM_PACK_ANAGLYPH = 0, 1


class StereoParams(ctypes.Structure):
    _fields_ = [
        ("div_px", ctypes.c_double * 2),
        ("sep_px", ctypes.c_double * 2),
        ("exponent", ctypes.c_double),
        ("eye_mode", ctypes.c_int32 * 2),
        ("fill", ctypes.c_int32),
        ("pack", ctypes.c_int32),
        ("anaglyph_red_eye", ctypes.c_int32),
        ("depth_kind", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("dst_row_stride", ctypes.c_int64 * 2),
        ("dst_img_stride", ctypes.c_int64 * 2),
    ]


class Weight(ctypes.Structure):
    """mirror of dm_weight"""
    _fields_ = [("name", ctypes.c_char_p), ("data_host", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("ndim", ctypes.c_int32),
                ("shape", ctypes.c_int64 * 4)]


class WeightBlob(ctypes.Structure):
    _fields_ = [("items", ctypes.POINTER(Weight)), ("count", ctypes.c_int32)]


class GemmDesc(ctypes.Structure):
    """mirror of dm_gemm_desc (include/depthmap_b200.h)"""
    _fields_ = [
        ("M", ctypes.c_int32), ("N", ctypes.c_int32), ("K", ctypes.c_int32),
        ("epi", ctypes.c_int32), ("act", ctypes.c_int32),
        ("bias", ctypes.c_void_p),
        ("C", ctypes.c_void_p), ("ldc", ctypes.c_int32),
        ("C2", ctypes.c_void_p),
        ("R", ctypes.c_void_p), ("ldr", ctypes.c_int32),
        ("R2", ctypes.c_void_p), ("ldr2", ctypes.c_int32),
        ("X", ctypes.c_void_p), ("ldx", ctypes.c_int32),
        ("gamma", ctypes.c_void_p),
        ("head_b2", ctypes.c_float),
        ("ps_s", ctypes.c_int32), ("ps_cout", ctypes.c_int32), ("ps_h", ctypes.c_int32), ("ps_w", ctypes.c_int32),
    ]


EPI_STORE_F16, EPI_RESID_F32, EPI_PIXSHUF, EPI_HEAD, EPI_STORE_F32 = 0, 1, 2, 3, 4
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2

_lock = threading.Lock()
_lib = None

# every symbol include/depthmap_b200.h declares; tests check the built library exports all of them
EXPORTS = [
    "dm_last_error", "dm_version", "dm_device_name",
    "dm_normalize_u16_workspace_bytes", "dm_normalize_u16", "dm_normalize_u16_outliers_workspace_bytes", "dm_normalize_u16_outliers",
    "dm_stereo_workspace_bytes", "dm_stereo", "dm_stereo_pack", "dm_depth_to_nd64", "dm_convert_to_i16_f64",
    "dm_normalmap_workspace_bytes", "dm_normalmap",
    "dm_gemm_ex", "dm_conv3x3_ex", "dm_gemm_f16", "dm_conv3x3_f16", "dm_attention_f16", "dm_attention_relpos_f16", "dm_preprocess_patchify",
    "dm_assemble_tokens", "dm_layernorm_f16", "dm_resize_bilinear_nhwc_f16", "dm_resize_f32", "dm_im2col_s2_f16", "dm_concat_readout_f16",
    "dm_zoe_preprocess_patchify", "dm_layernorm_post_f16", "dm_attention_small_f16", "dm_cast_f32_f16", "dm_zoe_select_softplus",
    "dm_resize_add_nhwc_f16", "dm_zoe_attractor", "dm_zoe_clb_final", "dm_zoe_tta_combine",
    "dm_zoe_attractor_single", "dm_zoe_seed_normed", "dm_zoe_clb_final_single",
    "dm_video_workspace_bytes", "dm_video_blend", "dm_video_minmax", "dm_video_scale_f32", "dm_video_select_init", "dm_video_select_hist",
    "dm_video_select_pick", "dm_video_select_bounds", "dm_video_scale_f64",
    "dm_model_create", "dm_model_destroy", "dm_model_net_size", "dm_model_launches", "dm_depth_forward", "dm_dinov2_pos_embed", "dm_beit_rel_table", "dm_vit_pos_embed",
    "dm_leres_stem_im2col", "dm_maxpool3x3s2_nhwc_f16", "dm_subsample2_nhwc_f16", "dm_add_f16", "dm_resize_f32_ld",
    "dm_boost_partials", "dm_unet_first_cols", "dm_unet_down_cols", "dm_unet_up_cols", "dm_unet_interleave", "dm_unet_final", "dm_unet_first", "dm_unet_last", "dm_sum_chunks_f32", "dm_boost_minmax",
    "dm_boost_merge_input", "dm_boost_post", "dm_boost_fit_sums", "dm_boost_blend", "dm_boost_resize_cubic", "dm_boost_u8_to_planar",
    "dm_leres_stem_im2col_f32", "dm_leres_stem_im2col_f32_batch",
]


def load() -> ctypes.CDLL:
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"depthmap_b200: native library missing ({LIB_PATH}). Build it with "
                f"`python {os.path.join(_HERE, 'csrc', 'build.py')}` — there is no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        c = ctypes
        vp, i32, i64, f32, sz = c.c_void_p, c.c_int, c.c_int64, c.c_float, c.c_size_t
        L.dm_last_error.restype = c.c_char_p
        L.dm_version.restype = i32
        L.dm_device_name.argtypes = [c.c_char_p, i32]
        L.dm_normalize_u16_workspace_bytes.argtypes = [i32]
        L.dm_normalize_u16_workspace_bytes.restype = sz
        L.dm_normalize_u16.argtypes = [vp, i32, i32, i32, i32, i32, f32, f32, vp, vp, vp, sz, vp]
        L.dm_normalize_u16_outliers_workspace_bytes.argtypes = [i32]
        L.dm_normalize_u16_outliers_workspace_bytes.restype = sz
        L.dm_normalize_u16_outliers.argtypes = [vp, i32, i32, i32, i32, ctypes.POINTER(ctypes.c_int64), ctypes.c_double, ctypes.c_double, vp, vp, vp, sz, vp]
        L.dm_stereo_workspace_bytes.argtypes = [i32, i32, i32]
        L.dm_stereo_workspace_bytes.restype = sz
        L.dm_stereo.argtypes = [vp, vp, i32, i32, i32, c.POINTER(StereoParams), vp, vp, vp, sz, vp]
        L.dm_stereo_pack.argtypes = [vp, i32, i32, i32, i32, vp, vp]
        L.dm_depth_to_nd64.argtypes = [vp, i32, i32, c.c_longlong, vp, vp, vp]
        L.dm_convert_to_i16_f64.argtypes = [vp, c.c_longlong, vp, vp]
        L.dm_normalmap_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32]
        L.dm_normalmap_workspace_bytes.restype = sz
        L.dm_normalmap.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, sz, vp]
        if hasattr(L, "dm_video_blend"):
            ll, dbl = c.c_longlong, c.c_double
            L.dm_video_workspace_bytes.restype = sz
            L.dm_video_blend.argtypes = [vp, ll, i32, i32, i32, i32, i32, vp, vp]
            L.dm_video_minmax.argtypes = [vp, ll, vp, vp, sz, vp]
            L.dm_video_scale_f32.argtypes = [vp, ll, vp, vp, vp]
            L.dm_video_select_init.argtypes = [vp, c.POINTER(ll), vp]
            L.dm_video_select_hist.argtypes = [vp, ll, i32, vp, vp]
            L.dm_video_select_pick.argtypes = [vp, i32, vp]
            L.dm_video_select_bounds.argtypes = [vp, dbl, dbl, vp, vp]
            L.dm_video_scale_f64.argtypes = [vp, ll, vp, vp, vp]
        if hasattr(L, "dm_model_create"):
            L.dm_model_create.argtypes = [c.POINTER(vp), i32, c.POINTER(WeightBlob), i32, i32]
            L.dm_model_destroy.argtypes = [vp]
            L.dm_model_net_size.argtypes = [vp, i32, i32, i32, i32, c.POINTER(i32), c.POINTER(i32)]
            L.dm_model_launches.argtypes = [vp]
            L.dm_model_launches.restype = c.c_longlong
            L.dm_depth_forward.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, i32, i32, vp]
            L.dm_dinov2_pos_embed.argtypes = [vp, i32, i32, i32, i32, vp]
            L.dm_beit_rel_table.argtypes = [vp, i32, i32, i32, i32, vp]
            L.dm_vit_pos_embed.argtypes = [vp, i32, i32, i32, i32, vp]
        _bind_optional(L)
        _lib = L
        return L


def _bind_optional(L):
    """Model entry points (present once the tensor-core units are linked in)."""
    c = ctypes
    vp, i32, i64, f32, sz = c.c_void_p, c.c_int, c.c_int64, c.c_float, c.c_size_t
    if hasattr(L, "dm_gemm_f16"):
        L.dm_gemm_f16.argtypes = [vp, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, vp]
        L.dm_conv3x3_f16.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, i32, i32, vp]
        L.dm_gemm_ex.argtypes = [vp, i32, vp, i32, c.POINTER(GemmDesc), vp]
        L.dm_conv3x3_ex.argtypes = [vp, i32, i32, i32, i32, vp, c.POINTER(GemmDesc), vp]
    if hasattr(L, "dm_attention_f16"):
        L.dm_attention_f16.argtypes = [vp, i32, i32, i32, f32, vp, i32, vp, vp]
        L.dm_attention_relpos_f16.argtypes = [vp, i32, i32, i32, i32, f32, vp, vp, i32, vp, vp]
    if hasattr(L, "dm_layernorm_f16"):
        L.dm_preprocess_patchify.argtypes = [vp, i32, i32, i32, i32, i32, i32, c.POINTER(c.c_float), c.POINTER(c.c_float),
                                             c.POINTER(c.c_int), vp, i32, vp]
        L.dm_assemble_tokens.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp]
        L.dm_layernorm_f16.argtypes = [vp, c.c_longlong, i32, vp, vp, f32, vp, i32, i32, vp]
        L.dm_resize_bilinear_nhwc_f16.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, vp]
        L.dm_resize_f32.argtypes = [vp, i32, i32, i32, vp, i32, i32, i32, vp]
        L.dm_im2col_s2_f16.argtypes = [vp, i32, i32, i32, i32, vp, vp]
        L.dm_concat_readout_f16.argtypes = [vp, i32, i32, i32, vp, vp]
    if hasattr(L, "dm_leres_stem_im2col"):
        L.dm_leres_stem_im2col.argtypes = [vp, i32, i32, i32, i32, i32, c.POINTER(c.c_float), c.POINTER(c.c_float), vp, vp]
        L.dm_maxpool3x3s2_nhwc_f16.argtypes = [vp, i32, i32, i32, i32, vp, vp]
        L.dm_subsample2_nhwc_f16.argtypes = [vp, i32, i32, i32, i32, vp, vp]
        L.dm_add_f16.argtypes = [vp, vp, vp, c.c_longlong, vp]
        L.dm_resize_f32_ld.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, i32, vp]
    if hasattr(L, "dm_unet_first_cols"):
        ll = c.c_longlong
        L.dm_unet_first_cols.argtypes = [vp, i32, i32, vp, i32, vp]
        L.dm_unet_down_cols.argtypes = [vp, i32, i32, i32, vp, i32, vp]
        L.dm_unet_up_cols.argtypes = [vp, i32, vp, i32, i32, i32, vp, i32, vp]
        L.dm_unet_interleave.argtypes = [vp, i32, i32, i32, i32, vp, vp]
        L.dm_unet_final.argtypes = [vp, i32, i32, i32, f32, vp, vp]
        L.dm_boost_minmax.argtypes = [vp, ll, vp, vp]
        L.dm_sum_chunks_f32.argtypes = [vp, i32, ll, i32, vp, vp, vp]
        L.dm_unet_first.argtypes = [vp, i32, i32, vp, vp, vp]
        L.dm_unet_last.argtypes = [vp, i32, vp, i32, i32, i32, vp, f32, vp, vp]
        L.dm_boost_merge_input.argtypes = [vp, vp, ll, vp, vp, vp, vp]
        L.dm_boost_post.argtypes = [vp, ll, vp, i32, vp, vp]
        L.dm_boost_fit_sums.argtypes = [vp, vp, ll, vp, vp]
        L.dm_boost_blend.argtypes = [vp, i32, vp, vp, i32, vp, i32, i32, i32, i32, i32, vp]
        L.dm_boost_resize_cubic.argtypes = [vp, i32, ll, i32, i32, vp, i32, ll, i32, i32, i32, vp]
        L.dm_boost_u8_to_planar.argtypes = [vp, i32, i32, vp, vp]
        L.dm_leres_stem_im2col_f32.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, i32, c.POINTER(c.c_float), c.POINTER(c.c_float), vp, vp]
        L.dm_leres_stem_im2col_f32_batch.argtypes = [vp, i32, i32, vp, i32, i32, i32, c.POINTER(c.c_float), c.POINTER(c.c_float), vp, vp]
    if hasattr(L, "dm_zoe_clb_final"):
        L.dm_zoe_preprocess_patchify.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, i32, vp]
        L.dm_layernorm_post_f16.argtypes = [vp, c.c_longlong, i32, vp, vp, f32, vp, vp]
        L.dm_attention_small_f16.argtypes = [vp, i32, i32, i32, f32, vp, vp]
        L.dm_cast_f32_f16.argtypes = [vp, c.c_longlong, vp, vp]
        L.dm_zoe_select_softplus.argtypes = [vp, i32, vp, i32, i32, i32, vp, vp]
        L.dm_resize_add_nhwc_f16.argtypes = [vp, vp, i32, i32, i32, i32, vp, i32, i32, vp]
        L.dm_zoe_attractor.argtypes = [vp, i32, vp, i32, vp, i32, i32, i32, i32, i32, vp, vp]
        L.dm_zoe_clb_final.argtypes = [vp, i32, vp, i32, vp, vp, i32, vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, f32, vp, vp]
        L.dm_zoe_tta_combine.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, vp, vp]
    if hasattr(L, "dm_zoe_clb_final_single"):
        L.dm_zoe_attractor_single.argtypes = [vp, i32, i32, i32, vp, i32, i32, i32, i32, i32, f32, f32, vp, vp, vp]
        L.dm_zoe_seed_normed.argtypes = [vp, i32, c.c_longlong, f32, f32, vp, vp]
        L.dm_zoe_clb_final_single.argtypes = [vp, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, f32, i32, i32, i32, i32, i32, f32, f32, vp, vp]


def check(rc: int, what: str = ""):
    if rc == DM_OK:
        return
    msg = load().dm_last_error().decode("utf-8", "replace")
    if rc == DM_E_OOM:
        raise RuntimeError(f"CUDA out of memory. {msg}")  # src/core.py:310 matches 'out of memory'
    if rc == DM_E_INVALID:
        raise ValueError(msg or what)
    if rc == DM_E_UNSUPPORTED:
        raise NotImplementedError(msg or what)
    raise RuntimeError(f"depthmap_b200 {what} failed ({rc}): {msg}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("depthmap_b200: no CUDA device visible; the B200 kernels have no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
