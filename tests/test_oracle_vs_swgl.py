"""Pins the C oracle (oracle/wr_oracle.c) against the UNMODIFIED reference
rasteriser (oracle/_ref/libswgl_ref.so, built by oracle/Makefile from a WebRender
checkout): same frames through both, byte-for-byte — against the digests of the
reference's output stored in golden/reference_digests.json (the `reference`
fixture), so no reference build is needed to run them."""
import numpy as np
import pytest

from oracle.backends import OracleDevice, SwglDevice
from webrender_b200 import abi
from workloads import scenes

from common import reference, render  # noqa: F401 (reference: fixture)

BLENDS = [abi.BLEND_PREMULTIPLIED_ALPHA, abi.BLEND_ALPHA, abi.BLEND_PREMULTIPLIED_DEST_OUT, abi.BLEND_MULTIPLY,
          abi.BLEND_PLUS_LIGHTER, abi.BLEND_SUBPIXEL_PASS0, abi.BLEND_NONE]


@pytest.mark.parametrize("blend", BLENDS)
@pytest.mark.parametrize("random_rects", [False, True])
def test_alpha_rects(blend, random_rects, reference):
    f = scenes.alpha_rects_frame(333, 141, 41, random_rects=random_rects, seed=5, blend=blend,
                                 color=(0.25, 0.125, 0.05, 0.3))
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("blend", list(range(abi.BLEND_ADV_MULTIPLY, abi.BLEND_ADV_LUMINOSITY + 1)) +
                         [abi.BLEND_MIN, abi.BLEND_MAX, abi.BLEND_ADD_KEEP_ALPHA_OVER, abi.BLEND_DST_ALPHA_ADD,
                          abi.BLEND_SUBPIXEL_PASS0_KEEP_A])
def test_blend_keys_random_layers(blend, reference):
    """Every blend key of the reference's blend stage over random premultiplied layers."""
    f = scenes.alpha_rects_frame(160, 64, 24, random_rects=True, seed=100 + blend, blend=blend,
                                 color=None, clear_color=(0.4, 0.7, 0.2, 0.8))
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["plain", "fractional", "force_aa", "aa_fractional", "scaled"])
def test_brush_solid_opaque_alpha_masks(seed, variant, reference):
    f = scenes.brush_solid_frame(333, 207, seed=seed, fractional="fractional" in variant,
                                 force_aa="aa" in variant,
                                 device_pixel_scale=1.5 if variant == "scaled" else 1.0)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled"])
def test_clip_rectangle_masks(seed, variant, reference):
    """cs_clip_rectangle fast + general paths, Clip/ClipOut, primary (overwrite) and
    secondary (multiply) — bit-exact R8 masks."""
    f = scenes.clip_mask_frame(seed=seed, fractional=variant != "integer", scale=1.25 if variant == "scaled" else 1.0)
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled", "nearest"])
def test_rounded_rects_indirect(seed, variant, reference):
    """Config A flavour: off-screen quad + ps_quad_mask (fast/slow) multiply, then a
    textured composite quad sampling the off-screen task."""
    f = scenes.rounded_rects_frame(seed=seed, fractional=variant in ("fractional", "scaled"),
                                   device_pixel_scale=1.5 if variant == "scaled" else 1.0,
                                   filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["linear", "nearest", "linear_1to1", "nearest_1to1", "linear_fractional"])
def test_brush_image(seed, variant, reference):
    f = scenes.image_frame(seed=seed, filter=abi.NEAREST if "nearest" in variant else abi.LINEAR,
                           one_to_one="1to1" in variant, fractional="fractional" in variant)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["r8_alpha", "r8_fractional", "r8_scaled", "rgba_modes", "r8_shadow_masks"])
def test_text_run(seed, variant, reference):
    kw = dict(seed=seed, width=480, height=270, n_runs=8, glyphs_per_run=20)
    if variant == "r8_fractional":
        kw.update(fractional=True)
    elif variant == "r8_scaled":
        kw.update(device_pixel_scale=1.5, fractional=True)
    elif variant == "rgba_modes":
        kw.update(atlas="rgba8", color_modes=(3, 1, 2))
    elif variant == "r8_shadow_masks":
        kw.update(color_modes=(0, 2), with_masks=True)
    f = scenes.text_frame(**kw)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["opaque", "alpha", "fractional", "repeat", "full_frame"])
def test_linear_gradient(seed, variant, reference):
    """brush_linear_gradient incl. the span shader's merged-run 16-bit colour
    stepping (swgl_commitLinearGradientRGBA8) — the oracle restates it exactly."""
    f = scenes.gradient_frame(seed=seed, fractional=variant == "fractional", repeat=variant == "repeat",
                              full_frame=variant == "full_frame",
                              blend=abi.BLEND_PREMULTIPLIED_ALPHA if variant == "alpha" else abi.BLEND_NONE)
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


BOX_SHADOW_VARIANTS = ["integer", "fractional", "scaled", "nearest"]


def _box_shadow_frame(seed, variant):
    f = scenes.box_shadow_frame(seed=seed, fractional=variant in ("fractional", "scaled"),
                                scale=1.5 if variant == "scaled" else 1.0)
    if variant == "nearest":
        f.textures["shadow"].filter = abi.NEAREST
    return f


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
@pytest.mark.parametrize("variant", BOX_SHADOW_VARIANTS)
def test_clip_box_shadow(seed, variant, reference):
    """cs_clip_box_shadow: nine-patch / simple stretch of a blurred R8 mask, both
    clip modes, span shader with solid, per-fragment and texture-span sections."""
    f = _box_shadow_frame(seed, variant)
    reference(render(OracleDevice, f, ["mask"]), lambda: render(SwglDevice, f, ["mask"]))


COMPOSITE_VARIANTS = ["tiles", "fractional", "external", "external_fractional"]


def _composite_frame(seed, variant):
    return scenes.composite_frame(seed=seed, external="external" in variant, fractional="fractional" in variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", COMPOSITE_VARIANTS)
def test_composite(seed, variant, reference):
    """composite_simple: opaque FAST_PATH tile copies, clear tile (dest-out), alpha
    and solid-colour tiles, external RGB surfaces with unnormalised uv rects,
    linear filtering, colour modulation and flips."""
    f = _composite_frame(seed, variant)
    reference(render(OracleDevice, f, ["fb"]), lambda: render(SwglDevice, f, ["fb"]))



@pytest.mark.parametrize("seed", [1, 2])
def test_composite_tile_lists_oracle(seed, reference):
    """The oracle's wro_draw_composite_tiles (one draw per instance) equals SWGL's per-texture draws."""
    f = _composite_frame(seed, "external_fractional")
    reference(render(OracleDevice, f, ["fb"], tile_lists=True), lambda: render(SwglDevice, f, ["fb"]))


YUV_FORMATS = ["planar", "nv12", "interleaved"]
YUV_VARIANTS = ["opaque", "blend", "fractional", "nearest"]


def _yuv_frame(fmt, color_space, variant):
    return scenes.yuv_composite_frame(fmt, color_space, seed=1 + color_space, linear=variant != "nearest",
                                      opaque=variant != "blend", fractional=variant == "fractional")


@pytest.mark.parametrize("color_space", [0, 1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_composite_yuv_color_spaces(fmt, color_space, reference):
    """composite with WR_FEATURE_YUV (composite.glsl:83-130, 163-176, 197-214; yuv.glsl): 8-bit PLANAR / NV12 /\n    INTERLEAVED video surfaces in every YuvRangedColorSpace; span body through the fixed-point YUVMatrix\n    (composite.h:636-779), tails and nearest-filtered planes through sample_yuv's float matrix."""
    f = _yuv_frame(fmt, color_space, "opaque")
    reference(render(OracleDevice, f, ["fb"]), lambda: render(SwglDevice, f, ["fb"]))


@pytest.mark.parametrize("variant", YUV_VARIANTS[1:])
@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_composite_yuv_variants(fmt, variant, reference):
    f = _yuv_frame(fmt, 2 if variant != "fractional" else 5, variant)
    reference(render(OracleDevice, f, ["fb"]), lambda: render(SwglDevice, f, ["fb"]))


YUV_IMAGE_VARIANTS = ["alpha", "opaque", "fractional", "nearest", "rotated"]


def _yuv_image_frame(fmt, variant, color_space=2):
    return scenes.yuv_image_frame(fmt, color_space, seed=1 + color_space, linear=variant != "nearest",
                                  alpha_pass=variant != "opaque", fractional=variant == "fractional",
                                  rotate=17.0 if variant == "rotated" else None)


@pytest.mark.parametrize("variant", YUV_IMAGE_VARIANTS)
@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_brush_yuv_image(fmt, variant, reference):
    """Brush(YuvImage) (brush_yuv_image.glsl): video frames as primitives — opaque and alpha pass, AA edges,
    clip masks, a rotated spatial node, NEAREST planes (fragment path with sample_yuv's ALPHA_PASS clamp)."""
    f = _yuv_image_frame(fmt, variant, 5 if variant == "fractional" else 2)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


OPACITY_VARIANTS = ["scaled", "fractional", "one_to_one", "nearest"]


def _opacity_frame(seed, variant):
    return scenes.opacity_frame(seed=seed, fractional=variant == "fractional", one_to_one=variant == "one_to_one",
                                filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", OPACITY_VARIANTS)
def test_brush_opacity(seed, variant, reference):
    f = _opacity_frame(seed, variant)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("r8", [False, True])
def test_ps_clear(seed, r8, reference):
    f = scenes.clear_frame(seed=seed, r8=r8)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["alpha", "fractional", "opaque"])
def test_brush_blend(seed, variant, reference):
    """brush_blend: every CSS filter op incl. the vector pow() approximation
    behind sRGB<->linear and gamma transfer."""
    f = scenes.blend_frame(seed=seed, fractional=variant == "fractional", opaque_source=variant == "opaque")
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["integer", "fractional"])
def test_brush_mix_blend(seed, variant, reference):
    f = scenes.mix_blend_frame(seed=seed, fractional=variant == "fractional")
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("rot", [17.0, -33.5, 90.0, 45.0, 180.0, 3.0])
@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("masks", [False, True])
def test_rotated_brush_solid(rot, seed, masks, reference):
    """Non-axis-aligned quads: the full edge walk of draw_quad_spans (edge
    switches at vertices, AA on every edge in the alpha pass, none in the opaque
    pass), depth and clip masks."""
    f = scenes.brush_solid_frame(seed=seed, rotate=rot, fractional=True, with_masks=masks)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("rot", [17.0, -33.5, 90.0])
@pytest.mark.parametrize("kind", ["image", "image_occluded", "gradient_alpha", "gradient_opaque"])
def test_rotated_textured(rot, kind, reference):
    if kind.startswith("image"):
        f = scenes.image_frame(seed=2, rotate=rot, fractional=True, n_opaque=0 if kind == "image" else 8)
    elif kind == "gradient_alpha":
        f = scenes.gradient_frame(seed=2, rotate=rot, fractional=True, blend=abi.BLEND_PREMULTIPLIED_ALPHA)
    else:
        f = scenes.gradient_frame(seed=2, rotate=rot)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("color", [False, True])
def test_cs_blur(seed, color, reference):
    """cs_blur ALPHA_TARGET / COLOR_TARGET: vertical then horizontal pass, clamped
    sampling at region edges, zero radius, 16-bit saturating accumulation."""
    f = scenes.blur_frame(seed=seed, color=color)
    reference(render(OracleDevice, f, ["mid", "target"]), lambda: render(SwglDevice, f, ["mid", "target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["rgba", "r8", "nearest"])
def test_cs_scale(seed, variant, reference):
    f = scenes.scale_frame(seed=seed, r8=variant == "r8", filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


CS_GRADIENT_KINDS = {"fast_linear": abi.KIND_FAST_LINEAR_GRADIENT, "linear": abi.KIND_LINEAR_GRADIENT,
                     "radial": abi.KIND_RADIAL_GRADIENT, "conic": abi.KIND_CONIC_GRADIENT}


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["plain", "repeat", "hard"])
@pytest.mark.parametrize("kind", list(CS_GRADIENT_KINDS))
def test_cached_gradient_tasks(kind, variant, seed, reference):
    """cs_{fast_linear,linear,radial,conic}_gradient render tasks
    (draw_texture_cache_target): span paths swgl_commitLinearGradientRGBA8
    (tileRepeat off) and swgl_commitRadialGradientRGBA8 restated exactly."""
    f = scenes.cached_gradient_frame(CS_GRADIENT_KINDS[kind], seed=seed, repeat=variant == "repeat",
                                     hard=variant == "hard")
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_line_decoration_tasks(seed, reference):
    """cs_line_decoration: solid / dotted / dashed / wavy masks at several device scales."""
    f = scenes.line_decoration_frame(seed=seed)
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("scale", [1.0, 1.5])
@pytest.mark.parametrize("kind", ["solid", "segment"])
def test_border_tasks(kind, scale, seed, reference):
    """cs_border_solid / cs_border_segment: corner and edge tasks with elliptical
    corner clips, adjacent-corner clips, double/groove/ridge styling, dash and dot clips."""
    f = scenes.border_frame(abi.KIND_BORDER_SOLID if kind == "solid" else abi.KIND_BORDER_SEGMENT, seed=seed,
                            scale=scale)
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("seed", [1, 2])
def test_texture_cache_target_all_task_lists(seed, reference):
    """All task lists of one texture-cache target in draw_texture_cache_target's order."""
    f = scenes.texture_cache_frame(seed=seed)
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


QUAD_GRADIENT_KINDS = {"radial": abi.KIND_QUAD_RADIAL_GRADIENT, "conic": abi.KIND_QUAD_CONIC_GRADIENT}


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled", "rotated", "opaque"])
@pytest.mark.parametrize("kind", list(QUAD_GRADIENT_KINDS))
def test_quad_gradients(kind, variant, seed, reference):
    """ps_quad_radial_gradient (span: swgl_commitRadialGradientRGBA8) and
    ps_quad_conic_gradient (approx_atan2 polynomial, fragment only)."""
    f = scenes.quad_gradient_frame(QUAD_GRADIENT_KINDS[kind], seed=seed, fractional=variant in ("fractional", "scaled"),
                                   device_pixel_scale=1.5 if variant == "scaled" else 1.0,
                                   rotate=23.0 if variant == "rotated" else None,
                                   blend=abi.BLEND_NONE if variant == "opaque" else abi.BLEND_PREMULTIPLIED_ALPHA)
    reference(render(OracleDevice, f), lambda: render(SwglDevice, f))


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
@pytest.mark.parametrize("variant", ["linear", "nearest", "fractional", "scaled"])
def test_brush_image_repetition(seed, variant, reference):
    """brush_image ANTIALIASING,REPETITION: tiled images and border-image segments through
    swgl_commitTextureRepeat[Color]RGBA8 (blendTextureLinearRepeat / blendTextureNearestRepeat)."""
    f = scenes.image_repeat_frame(seed=seed, filter=abi.NEAREST if variant == "nearest" else abi.LINEAR,
                                  fractional=variant in ("fractional", "scaled"),
                                  device_pixel_scale=1.5 if variant == "scaled" else 1.0)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


GLYPH_TRANSFORMS = {"identity": (0.0, 1.0, 1.0), "scaled": (0.0, 1.25, 0.8), "rotated": (17.0, 1.0, 1.0),
                    "rotated_scaled": (-33.0, 1.3, 0.9), "quarter_turn": (90.0, 1.0, 1.0)}


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("atlas", ["r8", "rgba"])
@pytest.mark.parametrize("xf", list(GLYPH_TRANSFORMS))
def test_text_run_glyph_transform(xf, atlas, seed, reference):
    """ps_text_run GLYPH_TRANSFORM: glyph rects in the transformed space, quads trimmed by
    gl_ClipDistance (clip_distance_range, rasterize.h:566-596), incl. runs cut by a local clip rect."""
    f = scenes.text_frame(seed=seed, width=480, height=270, n_runs=8, glyphs_per_run=16, atlas=atlas,
                          color_modes=(0,) if atlas == "r8" else (0, 1, 2, 3), fractional=True,
                          glyph_transform=GLYPH_TRANSFORMS[xf], clip_runs=True)
    reference(render(OracleDevice, f, ["target"]), lambda: render(SwglDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
def test_page_of_many_small_batches(seed, reference):
    """The multi-pass page scene (clip-mask pass, picture-cache tiles, tile list) through both CPU checkers."""
    f = scenes.page_frame(width=2048, height=1024, seed=seed)
    names = ["mask", "tile0", "tile3", "fb"]
    reference(render(OracleDevice, f, names), lambda: render(SwglDevice, f, names))
