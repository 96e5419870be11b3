"""ctypes mirror of include/wrcu.h (the C ABI of the B200 frame-draw backend).

Enumerations and struct layouts only; no logic.  Field order must match
include/wrcu.h exactly.
"""
import ctypes as C

ABI_VERSION = 1

# wrcu_status
OK, ERR_INVALID, ERR_OOM, ERR_CUDA, ERR_UNSUPPORTED, ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5

# wrcu_format
FMT_RGBA8, FMT_R8, FMT_RGBAF32, FMT_RGBAI32, FMT_DEPTH24, FMT_RG8, FMT_R16, FMT_RG16 = 1, 2, 3, 4, 5, 6, 7, 8
FMT_BPP = {FMT_RGBA8: 4, FMT_R8: 1, FMT_RGBAF32: 16, FMT_RGBAI32: 16, FMT_DEPTH24: 4, FMT_RG8: 2, FMT_R16: 2,
           FMT_RG16: 4}

NEAREST, LINEAR = 0, 1

# wrcu_kind
(KIND_QUAD_TEXTURED, KIND_QUAD_MASK, KIND_BRUSH_SOLID, KIND_BRUSH_IMAGE,
 KIND_BRUSH_LINEAR_GRADIENT, KIND_BRUSH_BLEND, KIND_BRUSH_MIX_BLEND,
 KIND_BRUSH_OPACITY, KIND_TEXT_RUN, KIND_CLIP_RECTANGLE, KIND_CLIP_BOX_SHADOW,
 KIND_COMPOSITE, KIND_CLEAR, KIND_BLUR, KIND_SCALE,
 KIND_FAST_LINEAR_GRADIENT, KIND_LINEAR_GRADIENT, KIND_RADIAL_GRADIENT, KIND_CONIC_GRADIENT,
 KIND_LINE_DECORATION, KIND_BORDER_SOLID, KIND_BORDER_SEGMENT,
 KIND_QUAD_RADIAL_GRADIENT, KIND_QUAD_CONIC_GRADIENT, KIND_BRUSH_YUV_IMAGE, KIND_SPLIT_COMPOSITE) = range(1, 27)

KIND_PROGRAM = {
    KIND_QUAD_TEXTURED: "ps_quad_textured",
    KIND_QUAD_MASK: "ps_quad_mask",
    KIND_BRUSH_SOLID: "brush_solid",
    KIND_BRUSH_IMAGE: "brush_image",
    KIND_BRUSH_LINEAR_GRADIENT: "brush_linear_gradient",
    KIND_BRUSH_BLEND: "brush_blend",
    KIND_BRUSH_MIX_BLEND: "brush_mix_blend",
    KIND_BRUSH_OPACITY: "brush_opacity",
    KIND_TEXT_RUN: "ps_text_run",
    KIND_CLIP_RECTANGLE: "cs_clip_rectangle",
    KIND_CLIP_BOX_SHADOW: "cs_clip_box_shadow",
    KIND_COMPOSITE: "composite",
    KIND_CLEAR: "ps_clear",
    KIND_BLUR: "cs_blur",
    KIND_SCALE: "cs_scale",
    KIND_FAST_LINEAR_GRADIENT: "cs_fast_linear_gradient",
    KIND_LINEAR_GRADIENT: "cs_linear_gradient",
    KIND_RADIAL_GRADIENT: "cs_radial_gradient",
    KIND_CONIC_GRADIENT: "cs_conic_gradient",
    KIND_LINE_DECORATION: "cs_line_decoration",
    KIND_BORDER_SOLID: "cs_border_solid",
    KIND_BORDER_SEGMENT: "cs_border_segment",
    KIND_QUAD_RADIAL_GRADIENT: "ps_quad_radial_gradient",
    KIND_QUAD_CONIC_GRADIENT: "ps_quad_conic_gradient",
    KIND_BRUSH_YUV_IMAGE: "brush_yuv_image",
    KIND_SPLIT_COMPOSITE: "ps_split_composite",
}

FEAT_ALPHA_PASS = 1 << 0
FEAT_FAST_PATH = 1 << 1
FEAT_ANTIALIASING = 1 << 2
FEAT_REPETITION = 1 << 3
FEAT_DUAL_SOURCE_BLENDING = 1 << 4
FEAT_ADVANCED_BLEND = 1 << 5
FEAT_GLYPH_TRANSFORM = 1 << 6
FEAT_TEXTURE_2D = 1 << 7
FEAT_ALPHA_TARGET = 1 << 8
FEAT_COLOR_TARGET = 1 << 9
FEAT_YUV = 1 << 10
FEATURE_NAMES = [
    (FEAT_ADVANCED_BLEND, "ADVANCED_BLEND"),
    (FEAT_ALPHA_PASS, "ALPHA_PASS"),
    (FEAT_ALPHA_TARGET, "ALPHA_TARGET"),
    (FEAT_ANTIALIASING, "ANTIALIASING"),
    (FEAT_COLOR_TARGET, "COLOR_TARGET"),
    (FEAT_DUAL_SOURCE_BLENDING, "DUAL_SOURCE_BLENDING"),
    (FEAT_FAST_PATH, "FAST_PATH"),
    (FEAT_GLYPH_TRANSFORM, "GLYPH_TRANSFORM"),
    (FEAT_REPETITION, "REPETITION"),
    (FEAT_TEXTURE_2D, "TEXTURE_2D"),
    (FEAT_YUV, "YUV"),
]


def program_key(kind, features):
    """Reference program key "<shader>[ FEAT,FEAT]" (swgl/build.rs:13-31):
    features sorted alphabetically, comma-joined."""
    feats = [n for bit, n in FEATURE_NAMES if features & bit]
    name = KIND_PROGRAM[kind]
    return name + (" " + ",".join(sorted(feats)) if feats else "")


# wrcu_blend
(BLEND_NONE, BLEND_ALPHA, BLEND_PREMULTIPLIED_ALPHA, BLEND_SUBPIXEL_PASS0,
 BLEND_SUBPIXEL_PASS0_KEEP_A, BLEND_PREMULTIPLIED_DEST_OUT, BLEND_MULTIPLY,
 BLEND_PLUS_LIGHTER, BLEND_ADD_KEEP_ALPHA_OVER, BLEND_DST_ALPHA_ADD,
 BLEND_CONSTANT_COLOR, BLEND_SUBPIXEL_DUAL_SOURCE, BLEND_MIN, BLEND_MAX,
 BLEND_ADV_MULTIPLY, BLEND_ADV_SCREEN, BLEND_ADV_OVERLAY, BLEND_ADV_DARKEN,
 BLEND_ADV_LIGHTEN, BLEND_ADV_COLOR_DODGE, BLEND_ADV_COLOR_BURN,
 BLEND_ADV_HARD_LIGHT, BLEND_ADV_SOFT_LIGHT, BLEND_ADV_DIFFERENCE,
 BLEND_ADV_EXCLUSION, BLEND_ADV_HUE, BLEND_ADV_SATURATION, BLEND_ADV_COLOR,
 BLEND_ADV_LUMINOSITY) = range(29)
BLEND_COUNT = 29

DEPTH_OFF, DEPTH_TEST, DEPTH_TEST_WRITE = 0, 1, 2


class FrameTables(C.Structure):
    _fields_ = [
        ("prim_headers_f", C.c_void_p), ("prim_headers_f_texels", C.c_size_t),
        ("prim_headers_i", C.c_void_p), ("prim_headers_i_texels", C.c_size_t),
        ("transforms", C.c_void_p), ("transforms_texels", C.c_size_t),
        ("render_tasks", C.c_void_p), ("render_tasks_texels", C.c_size_t),
        ("gpu_cache", C.c_void_p), ("gpu_cache_texels", C.c_size_t),
        ("gpu_buffer_f", C.c_void_p), ("gpu_buffer_f_texels", C.c_size_t),
        ("gpu_buffer_i", C.c_void_p), ("gpu_buffer_i_texels", C.c_size_t),
    ]


class UploadRect(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32),
                ("offset", C.c_uint64), ("stride", C.c_uint64)]


class GpuCacheCopy(C.Structure):
    _fields_ = [("block_index", C.c_uint32), ("block_count", C.c_uint32), ("u", C.c_uint16), ("v", C.c_uint16)]


class DrawState(C.Structure):
    _fields_ = [
        ("blend", C.c_int32),
        ("depth", C.c_int32),
        ("color", C.c_uint32 * 3),
        ("clip_mask", C.c_uint32),
        ("scissor_enabled", C.c_int32),
        ("scissor", C.c_int32 * 4),
        ("blend_color", C.c_float * 4),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_uint64),
        ("draw_calls", C.c_uint64),
        ("instances", C.c_uint64),
        ("h2d_bytes", C.c_uint64),
        ("d2h_bytes", C.c_uint64),
    ]


# Every symbol include/wrcu.h declares (checked by tests/test_abi.py).
SYMBOLS = [
    "wrcu_ctx_create", "wrcu_ctx_destroy", "wrcu_get_error",
    "wrcu_last_error_string", "wrcu_get_string", "wrcu_abi_version",
    "wrcu_finish", "wrcu_texture_create", "wrcu_texture_set_filter",
    "wrcu_texture_upload", "wrcu_texture_destroy", "wrcu_read_pixels",
    "wrcu_frame_begin", "wrcu_frame_end", "wrcu_target_bind", "wrcu_clear",
    "wrcu_draw_batch", "wrcu_draw_composite_tiles", "wrcu_program_from_name", "wrcu_get_stats",
    "wrcu_reset_stats", "wrcu_timer_begin", "wrcu_timer_end",
    "wrcu_texture_device_ptr", "wrcu_stream", "wrcu_host_alloc", "wrcu_host_free",
    "wrcu_read_pixels_async", "wrcu_fence_wait", "wrcu_fence_insert",
    "wrcu_profile_enable", "wrcu_last_raster_ms",
    "wrcu_texture_export", "wrcu_texture_import", "wrcu_peer_flags_create", "wrcu_peer_flags_open",
    "wrcu_peer_signal", "wrcu_peer_wait", "wrcu_composite_blit", "wrcu_composite_blit_yuv",
    "wrcu_texture_upload_batch", "wrcu_texture_copy", "wrcu_gpu_cache_update",
]


class IpcTexture(C.Structure):   # wrcu_ipc_texture
    _fields_ = [("handle", C.c_uint8 * 64), ("pid", C.c_uint64), ("address", C.c_uint64), ("pitch", C.c_uint64),
                ("format", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("device", C.c_int32)]


class IpcFlags(C.Structure):     # wrcu_ipc_flags
    _fields_ = [("handle", C.c_uint8 * 64), ("pid", C.c_uint64), ("address", C.c_uint64),
                ("count", C.c_int32), ("device", C.c_int32)]
