"""CPU tier: the CUDA sources' per-instance / per-pixel device functions,
executed on the host (tests/emu.py), against the oracle.  This is a development
aid for a box without a GPU; the parity tests proper are test_cuda_parity.py."""
import numpy as np
import pytest

from oracle.backends import OracleDevice
from webrender_b200 import abi
from workloads import scenes

from common import assert_same, reference, render  # noqa: F401 (reference: fixture)
from emu import EmuDevice


@pytest.mark.parametrize("blend", [abi.BLEND_PREMULTIPLIED_ALPHA, abi.BLEND_ALPHA, abi.BLEND_ADV_SOFT_LIGHT,
                                   abi.BLEND_ADV_HUE, abi.BLEND_NONE])
def test_quads(blend):
    f = scenes.alpha_rects_frame(257, 91, 23, random_rects=True, seed=blend, blend=blend, color=None)
    assert_same(render(EmuDevice, f), render(OracleDevice, f))


@pytest.mark.parametrize("variant", ["plain", "fractional", "scaled"])
def test_brush_solid(variant):
    f = scenes.brush_solid_frame(333, 207, seed=2, fractional=variant == "fractional",
                                 device_pixel_scale=1.5 if variant == "scaled" else 1.0)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled"])
def test_clip_rectangle(seed, variant):
    f = scenes.clip_mask_frame(seed=seed, fractional=variant != "integer", scale=1.25 if variant == "scaled" else 1.0)
    assert_same(render(EmuDevice, f), render(OracleDevice, f), variant)


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled", "nearest"])
def test_rounded_rects_indirect(seed, variant):
    f = scenes.rounded_rects_frame(seed=seed, fractional=variant in ("fractional", "scaled"),
                                   device_pixel_scale=1.5 if variant == "scaled" else 1.0,
                                   filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    assert_same(render(EmuDevice, f), render(OracleDevice, f), variant)


IMAGE_VARIANTS = ["linear", "nearest", "linear_1to1", "nearest_1to1", "linear_fractional"]


def _image_frame(seed, variant, n_opaque):
    return scenes.image_frame(seed=seed, n_opaque=n_opaque, filter=abi.NEAREST if "nearest" in variant else abi.LINEAR,
                              one_to_one="1to1" in variant, fractional="fractional" in variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", IMAGE_VARIANTS)
def test_brush_image_unoccluded_exact(seed, variant):
    """No opaque occluders: every span is one depth run → bit-exact for every filter path."""
    f = _image_frame(seed, variant, 0)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", IMAGE_VARIANTS)
def test_brush_image_occluded(seed, variant):
    """Opaque occluders inside the opaque batch (depth LEQUAL + write, front to back): every passing depth
    run is a span of its own (draw_depth_span, rasterize.h:612-657) — byte-exact for every filter path."""
    f = _image_frame(seed, variant, 8)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", IMAGE_VARIANTS + ["rotated"])
def test_brush_image_alpha_behind_opaque(seed, variant):
    """Alpha images partly hidden by opaque prims in front of them (what every page does): the alpha batch's
    spans are cut into depth runs whose chunk phase, span-shader body / fragment tail split and interpolant
    sums restart as the reference's do — byte-exact."""
    f = scenes.image_frame(seed=seed, n_opaque=8, filter=abi.NEAREST if "nearest" in variant else abi.LINEAR,
                           one_to_one="1to1" in variant, fractional="fractional" in variant or variant == "rotated",
                           rotate=23.0 if variant == "rotated" else None, occlude_alpha=True)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("rotate", [None, 17.0])
def test_brush_solid_aa_behind_opaque(seed, rotate):
    """AA edges and clip masks of alpha solids partly hidden by opaque prims: AA ramps and the mask-first
    ordering of solid span bodies follow the depth runs — byte-exact."""
    f = scenes.brush_solid_frame(640, 360, n_opaque=12, n_alpha=40, seed=seed, fractional=True, force_aa=True,
                                 occlude_alpha=True, rotate=rotate)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
def test_brush_image_repetition_behind_opaque(seed):
    f = scenes.image_repeat_frame(seed=seed, fractional=True, occlude_alpha=True)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


TEXT_VARIANTS = ["r8_alpha", "r8_fractional", "r8_scaled", "rgba_modes", "r8_shadow_masks"]


def _text_frame(seed, variant, **extra):
    kw = dict(seed=seed, width=480, height=270, n_runs=8, glyphs_per_run=20)
    if variant == "r8_fractional":
        kw.update(fractional=True)
    elif variant == "r8_scaled":
        kw.update(device_pixel_scale=1.5, fractional=True)
    elif variant == "rgba_modes":
        kw.update(atlas="rgba8", color_modes=(3, 1, 2))
    elif variant == "r8_shadow_masks":
        kw.update(color_modes=(0, 2), with_masks=True)
    kw.update(extra)
    return scenes.text_frame(**kw)


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", TEXT_VARIANTS)
def test_text_run(seed, variant):
    f = _text_frame(seed, variant)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


GRADIENT_VARIANTS = ["opaque", "alpha", "fractional", "repeat", "full_frame"]


def _gradient_frame(seed, variant):
    return scenes.gradient_frame(seed=seed, fractional=variant == "fractional", repeat=variant == "repeat",
                                 full_frame=variant == "full_frame",
                                 blend=abi.BLEND_PREMULTIPLIED_ALPHA if variant == "alpha" else abi.BLEND_NONE)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", GRADIENT_VARIANTS)
def test_linear_gradient(seed, variant):
    f = _gradient_frame(seed, variant)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


BOX_SHADOW_VARIANTS = ["integer", "fractional", "scaled", "nearest"]


def _box_shadow_frame(seed, variant):
    f = scenes.box_shadow_frame(seed=seed, fractional=variant in ("fractional", "scaled"),
                                scale=1.5 if variant == "scaled" else 1.0)
    if variant == "nearest":
        f.textures["shadow"].filter = abi.NEAREST
    return f


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
@pytest.mark.parametrize("variant", BOX_SHADOW_VARIANTS)
def test_clip_box_shadow(seed, variant):
    f = _box_shadow_frame(seed, variant)
    assert_same(render(EmuDevice, f, ["mask"]), render(OracleDevice, f, ["mask"]), variant)


COMPOSITE_VARIANTS = ["tiles", "fractional", "external", "external_fractional"]


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", COMPOSITE_VARIANTS)
def test_composite(seed, variant):
    f = scenes.composite_frame(seed=seed, external="external" in variant, fractional="fractional" in variant)
    assert_same(render(EmuDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]), variant)



@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", COMPOSITE_VARIANTS)
def test_composite_tile_lists(seed, variant):
    """wrcu_draw_composite_tiles: draw_tile_list (renderer/mod.rs:3126-3334) submitted as runs of
    instances with one texture each, against the reference's one draw per texture change."""
    f = scenes.composite_frame(seed=seed, external="external" in variant, fractional="fractional" in variant)
    assert_same(render(EmuDevice, f, ["fb"], tile_lists=True), render(OracleDevice, f, ["fb"]), variant)


YUV_FORMATS = ["planar", "nv12", "interleaved"]
YUV_VARIANTS = ["opaque", "blend", "fractional", "nearest"]


def _yuv_frame(fmt, color_space, variant):
    return scenes.yuv_composite_frame(fmt, color_space, seed=1 + color_space, linear=variant != "nearest",
                                      opaque=variant != "blend", fractional=variant == "fractional")


@pytest.mark.parametrize("color_space", [0, 1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_composite_yuv_color_spaces(fmt, color_space):
    """composite with WR_FEATURE_YUV (composite.glsl:83-130, 163-176, 197-214; yuv.glsl): 8-bit PLANAR / NV12 /\n    INTERLEAVED video surfaces in every YuvRangedColorSpace; span body through the fixed-point YUVMatrix\n    (composite.h:636-779), tails and nearest-filtered planes through sample_yuv's float matrix."""
    f = _yuv_frame(fmt, color_space, "opaque")
    assert_same(render(EmuDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]), fmt)


@pytest.mark.parametrize("variant", YUV_VARIANTS[1:])
@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_composite_yuv_variants(fmt, variant):
    f = _yuv_frame(fmt, 2 if variant != "fractional" else 5, variant)
    assert_same(render(EmuDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]), variant)


YUV_IMAGE_VARIANTS = ["alpha", "opaque", "fractional", "nearest", "rotated"]


def _yuv_image_frame(fmt, variant, color_space=2):
    return scenes.yuv_image_frame(fmt, color_space, seed=1 + color_space, linear=variant != "nearest",
                                  alpha_pass=variant != "opaque", fractional=variant == "fractional",
                                  rotate=17.0 if variant == "rotated" else None)


@pytest.mark.parametrize("variant", YUV_IMAGE_VARIANTS)
@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_brush_yuv_image(fmt, variant):
    """Brush(YuvImage) (brush_yuv_image.glsl): video frames as primitives — opaque and alpha pass, AA edges,
    clip masks, a rotated spatial node, NEAREST planes (fragment path with sample_yuv's ALPHA_PASS clamp)."""
    f = _yuv_image_frame(fmt, variant, 5 if variant == "fractional" else 2)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


OPACITY_VARIANTS = ["scaled", "fractional", "one_to_one", "nearest"]


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", OPACITY_VARIANTS)
def test_brush_opacity(seed, variant):
    f = scenes.opacity_frame(seed=seed, fractional=variant == "fractional", one_to_one=variant == "one_to_one",
                             filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("r8", [False, True])
def test_ps_clear(seed, r8):
    f = scenes.clear_frame(seed=seed, r8=r8)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["alpha", "fractional", "opaque"])
def test_brush_blend(seed, variant):
    f = scenes.blend_frame(seed=seed, fractional=variant == "fractional", opaque_source=variant == "opaque")
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["integer", "fractional"])
def test_brush_mix_blend(seed, variant):
    f = scenes.mix_blend_frame(seed=seed, fractional=variant == "fractional")
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("rot", [17.0, -33.5, 90.0, 45.0, 180.0, 3.0])
@pytest.mark.parametrize("seed", [1, 2])
def test_rotated_brush_solid(rot, seed):
    f = scenes.brush_solid_frame(seed=seed, rotate=rot, fractional=True, with_masks=seed == 2)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), f"rot {rot}")


@pytest.mark.parametrize("rot", [17.0, -33.5, 90.0])
@pytest.mark.parametrize("kind", ["image", "gradient_alpha", "gradient_opaque"])
def test_rotated_textured(rot, kind):
    """Rotated image / gradient brushes: per-row spans from the edge walk, uv rows
    that change along the span (fallback bilinear filter), AA on all edges."""
    if kind == "image":
        f = scenes.image_frame(seed=2, rotate=rot, fractional=True, n_opaque=0)
    elif kind == "gradient_alpha":
        f = scenes.gradient_frame(seed=2, rotate=rot, fractional=True, blend=abi.BLEND_PREMULTIPLIED_ALPHA)
    else:
        f = scenes.gradient_frame(seed=2, rotate=rot)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), kind)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("color", [False, True])
def test_cs_blur(seed, color):
    f = scenes.blur_frame(seed=seed, color=color)
    assert_same(render(EmuDevice, f, ["mid", "target"]), render(OracleDevice, f, ["mid", "target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["rgba", "r8", "nearest"])
def test_cs_scale(seed, variant):
    f = scenes.scale_frame(seed=seed, r8=variant == "r8", filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


CS_GRADIENT_KINDS = {"fast_linear": abi.KIND_FAST_LINEAR_GRADIENT, "linear": abi.KIND_LINEAR_GRADIENT,
                     "radial": abi.KIND_RADIAL_GRADIENT, "conic": abi.KIND_CONIC_GRADIENT}


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["plain", "repeat", "hard"])
@pytest.mark.parametrize("kind", list(CS_GRADIENT_KINDS))
def test_cached_gradient_tasks(kind, variant, seed):
    f = scenes.cached_gradient_frame(CS_GRADIENT_KINDS[kind], seed=seed, repeat=variant == "repeat",
                                     hard=variant == "hard")
    assert_same(render(EmuDevice, f), render(OracleDevice, f), kind + "/" + variant)


@pytest.mark.parametrize("kind", ["linear", "radial"])
def test_cached_gradient_wide_task(kind):
    """One 700-wide task: the span walk is resumed in six tiles per row."""
    f = scenes.cached_gradient_frame(CS_GRADIENT_KINDS[kind], width=704, height=40, n_tasks=1, seed=5, big=(700, 37))
    assert_same(render(EmuDevice, f), render(OracleDevice, f), kind)


@pytest.mark.parametrize("seed", [1, 2])
def test_line_decoration_tasks(seed):
    f = scenes.line_decoration_frame(seed=seed)
    assert_same(render(EmuDevice, f), render(OracleDevice, f))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("scale", [1.0, 1.5])
@pytest.mark.parametrize("kind", ["solid", "segment"])
def test_border_tasks(kind, scale, seed):
    f = scenes.border_frame(abi.KIND_BORDER_SOLID if kind == "solid" else abi.KIND_BORDER_SEGMENT, seed=seed,
                            scale=scale)
    assert_same(render(EmuDevice, f), render(OracleDevice, f), kind)


def test_texture_cache_target_all_task_lists():
    f = scenes.texture_cache_frame(seed=1)
    assert_same(render(EmuDevice, f), render(OracleDevice, f))


QUAD_GRADIENT_KINDS = {"radial": abi.KIND_QUAD_RADIAL_GRADIENT, "conic": abi.KIND_QUAD_CONIC_GRADIENT}


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled", "rotated", "opaque"])
@pytest.mark.parametrize("kind", list(QUAD_GRADIENT_KINDS))
def test_quad_gradients(kind, variant, seed):
    f = scenes.quad_gradient_frame(QUAD_GRADIENT_KINDS[kind], seed=seed, fractional=variant in ("fractional", "scaled"),
                                   device_pixel_scale=1.5 if variant == "scaled" else 1.0,
                                   rotate=23.0 if variant == "rotated" else None,
                                   blend=abi.BLEND_NONE if variant == "opaque" else abi.BLEND_PREMULTIPLIED_ALPHA)
    assert_same(render(EmuDevice, f), render(OracleDevice, f), kind + "/" + variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["linear", "nearest", "fractional", "scaled"])
def test_brush_image_repetition(seed, variant):
    """Exact.  (With opaque occluders in the same pass the known depth-run chunk-phase deviation
    applies, as for every non-1:1 textured span: DESIGN.md §4.4; bounded in test_cuda_parity.)"""
    f = scenes.image_repeat_frame(seed=seed, n_opaque=0, filter=abi.NEAREST if variant == "nearest" else abi.LINEAR,
                                  fractional=variant in ("fractional", "scaled"),
                                  device_pixel_scale=1.5 if variant == "scaled" else 1.0)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


GLYPH_TRANSFORMS = {"identity": (0.0, 1.0, 1.0), "scaled": (0.0, 1.25, 0.8), "rotated": (17.0, 1.0, 1.0),
                    "rotated_scaled": (-33.0, 1.3, 0.9), "quarter_turn": (90.0, 1.0, 1.0)}


@pytest.mark.parametrize("atlas", ["r8", "rgba"])
@pytest.mark.parametrize("xf", list(GLYPH_TRANSFORMS))
def test_text_run_glyph_transform(xf, atlas):
    f = scenes.text_frame(seed=1, width=480, height=270, n_runs=8, glyphs_per_run=16, atlas=atlas,
                          color_modes=(0,) if atlas == "r8" else (0, 1, 2, 3), fractional=True,
                          glyph_transform=GLYPH_TRANSFORMS[xf], clip_runs=True)
    assert_same(render(EmuDevice, f, ["target"]), render(OracleDevice, f, ["target"]), xf)


def _swgl_blit(src, dst, sr, dr, opaque, fx, fy, lin, cr):
    from oracle.backends import SwglDevice
    sh, sw = src.shape[:2]
    d = SwglDevice()
    ts, td = d.texture_create(abi.FMT_RGBA8, sw, sh), d.texture_create(abi.FMT_RGBA8, 640, 360)
    d.texture_upload(ts, 0, 0, sw, sh, src.reshape(sh, sw * 4))
    d.texture_upload(td, 0, 0, 640, 360, dst.reshape(360, 2560))
    d.sw_composite(td, ts, sr, dr, opaque, fx, fy, lin, cr)
    ref = d.locked_pixels(td)
    d.close()
    return {"dst": ref}


def _emu_blit(src, dst, sr, dr, opaque, fx, fy, lin, cr):
    import ctypes as C
    sh, sw = src.shape[:2]
    I4 = C.c_int32 * 4
    e = EmuDevice()
    es, ed = e.texture_create(abi.FMT_RGBA8, sw, sh), e.texture_create(abi.FMT_RGBA8, 640, 360)
    e.texture_upload(es, 0, 0, sw, sh, src.reshape(sh, sw * 4))
    e.texture_upload(ed, 0, 0, 640, 360, dst.reshape(360, 2560))
    f = e.lib.wremu_composite_blit
    f.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, C.c_int,
                  C.c_int, C.c_int, C.POINTER(C.c_int32)]
    assert f(e.ctx, ed, es, I4(*sr), I4(*dr), int(opaque), int(fx), int(fy), int(lin), I4(*cr)) == 0
    got = e.read_pixels(ed, 0, 0, 640, 360, 4)
    e.close()
    return {"dst": got}


def test_sw_compositor_blit_math_against_swgl(reference):
    """wrcu_composite_blit's arithmetic (the device function, run on the host) against the unmodified reference's
    Composite (swgl/src/composite.h:532-590): nearest / bilinear, flips, clips, over — bytes equal.  (The GPU
    tier repeats this through libwrcu_gl.so's LockTexture / Composite / GetResourceBuffer.)"""
    import test_gl_shim as T
    for case in T.SW_COMPOSITE_CASES:
        name, (sw, sh), sr, dr, opaque, fx, fy, lin, cr = case
        rng = np.random.RandomState(11)
        src = rng.randint(0, 256, (sh, sw, 4)).astype(np.uint8)
        al = src[..., 3:4].astype(np.uint16)
        src[..., :3] = (src[..., :3].astype(np.uint16) * al // 255).astype(np.uint8)
        dst = rng.randint(0, 256, (360, 640, 4)).astype(np.uint8)
        call = (src, dst, sr, dr, opaque, fx, fy, lin, cr)
        reference(_emu_blit(*call), lambda: _swgl_blit(*call), part=name)


def test_sw_compositor_blit_random_cases_against_swgl(reference):
    """Sixty seeded Composite calls (source / destination rects also partly outside, integer and fractional scale
    ratios, opaque and over, flips, both filters, clips) — device functions on the host against the unmodified
    reference: bytes equal."""
    rng = np.random.RandomState(77)
    for i in range(60):
        sw, sh = int(rng.randint(2, 300)), int(rng.randint(2, 200))
        src = rng.randint(0, 256, (sh, sw, 4)).astype(np.uint8)
        al = src[..., 3:4].astype(np.uint16)
        src[..., :3] = (src[..., :3].astype(np.uint16) * al // 255).astype(np.uint8)
        dst = rng.randint(0, 256, (360, 640, 4)).astype(np.uint8)
        rw, rh = int(rng.randint(1, sw + 1)), int(rng.randint(1, sh + 1))
        sr = (int(rng.randint(-5, sw - rw + 6)), int(rng.randint(-5, sh - rh + 6)), rw, rh)
        if i % 4 == 0:
            dr = (int(rng.randint(-20, 500)), int(rng.randint(-20, 300)), rw, rh)           # 1:1
        elif i % 4 == 1:
            k = int(rng.randint(2, 4))
            dr = (int(rng.randint(-20, 300)), int(rng.randint(-20, 150)), rw * k, rh * k)   # integer upscale
        else:
            dr = (int(rng.randint(-20, 400)), int(rng.randint(-20, 250)), int(rng.randint(1, 500)), int(rng.randint(1, 300)))
        cr = (0, 0, 640, 360) if i % 3 else (int(rng.randint(0, 300)), int(rng.randint(0, 150)), int(rng.randint(1, 400)), int(rng.randint(1, 250)))
        opaque, fx, fy, lin = bool(rng.randint(0, 2)), bool(rng.randint(0, 2)), bool(rng.randint(0, 2)), bool(rng.randint(0, 2))
        call = (src, dst, sr, dr, opaque, fx, fy, lin, cr)
        reference(_emu_blit(*call), lambda: _swgl_blit(*call), part=i)


def _emu_composite_yuv(case, planes):
    import ctypes as C
    import test_gl_shim as T
    I4 = C.c_int32 * 4

    def via(e, td, ty, tu, tv, cs, sr, dr, fx, fy, cr):
        f = e.lib.wremu_composite_blit_yuv
        f.argtypes = [C.c_void_p] + [C.c_uint32] * 4 + [C.c_int, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                                     C.c_int, C.c_int, C.POINTER(C.c_int32)]
        assert f(e.ctx, td, ty, tu, tv, int(cs), 8, I4(*sr), I4(*dr), int(fx), int(fy), I4(*cr)) == 0

    e = EmuDevice()
    got = T.run_sw_composite_yuv(e, case, planes, via=via)
    e.close()
    return {"dst": got}


def _swgl_composite_yuv(case, planes):
    from oracle.backends import SwglDevice
    import test_gl_shim as T
    d = SwglDevice()
    ref = T.run_sw_composite_yuv(d, case, planes)
    d.close()
    return {"dst": ref}


def test_sw_compositor_yuv_blit_math_against_swgl(reference):
    """wrcu_composite_blit_yuv's arithmetic (the device functions of csrc/blit_yuv.cuh, run on the host) against the
    unmodified reference's CompositeYUV (swgl/src/composite.h:1335-1384) — bytes equal.  (The GPU tier repeats this
    through libwrcu_gl.so.)"""
    import test_gl_shim as T
    for case in T.SW_COMPOSITE_YUV_CASES:
        planes = T.sw_yuv_planes(case)
        got = reference(_emu_composite_yuv(case, planes), lambda: _swgl_composite_yuv(case, planes), part=case[0])
        assert (got["dst"] != planes[3]).any(), case[0]


def test_sw_compositor_yuv_blit_random_cases_against_swgl(reference):
    """Eighty seeded CompositeYUV calls — plane sizes, chroma subsampling, source and destination rects (also partly
    outside the planes / the target), flips, clips, colour spaces drawn at random — device functions on the host
    against the unmodified reference: bytes equal."""
    import test_gl_shim as T
    rng = np.random.RandomState(2024)
    for i in range(80):
        yw, yh = int(rng.randint(2 if i % 10 == 9 else 8, 400)), int(rng.randint(2, 300))
        sub = [(1, 1), (2, 2), (2, 1)][int(rng.randint(0, 3))]
        cw, ch = max(2, (yw + sub[0] - 1) // sub[0]), max(2, (yh + sub[1] - 1) // sub[1])
        sx, sy = int(rng.randint(-10, yw // 2)), int(rng.randint(-8, yh // 2))
        sw, sh = int(rng.randint(1, yw + 1)), int(rng.randint(1, yh + 1))
        dx, dy = int(rng.randint(-40, 400)), int(rng.randint(-30, 250))
        dw, dh = int(rng.randint(1, 700)), int(rng.randint(1, 400))
        clip = (0, 0, 640, 360) if i % 3 else (int(rng.randint(0, 300)), int(rng.randint(0, 150)), int(rng.randint(1, 400)), int(rng.randint(1, 250)))
        case = ("rand%d" % i, (yw, yh), (cw, ch), int(rng.randint(0, 7)), (sx, sy, sw, sh), (dx, dy, dw, dh),
                bool(rng.randint(0, 2)), bool(rng.randint(0, 2)), clip)
        planes = T.sw_yuv_planes(case)
        reference(_emu_composite_yuv(case, planes), lambda: _swgl_composite_yuv(case, planes), part=case[0])


# ---- perspective quads / plane-split polygons: against the reference build itself -------------------------
PERSP_CAMERAS = [(800.0, 35.0, 0.0), (800.0, -20.0, 15.0), (220.0, 60.0, -30.0), (220.0, 80.0, 40.0)]


def _swgl(f, names):
    from oracle.backends import SwglDevice
    return lambda: render(SwglDevice, f, names)


@pytest.mark.parametrize("cam", PERSP_CAMERAS)
@pytest.mark.parametrize("kind", ["solid", "solid_aa", "image", "quad"])
def test_perspective_brushes(kind, cam, reference):
    """draw_perspective (rasterize.h:1422-1545): w differs between the vertices — near-plane clipping (the d=220
    cameras put part of the page behind the eye), the polygon edge walk, per-sample z and 1/w-corrected varyings."""
    d, ry, rx = cam
    kw = dict(seed=3, n_opaque=6, n_alpha=12)
    if kind == "solid_aa":
        kw.update(seed=4, force_aa=True)
    if kind == "quad":   # ps_quad_textured: the textured composite quads of the Indirect path under the 3-D node
        f = scenes.perspective_frame("quad", height=400, d=d, ry=ry, rx=rx, seed=2)
    else:
        f = scenes.perspective_frame("image" if kind == "image" else "solid", d=d, ry=ry, rx=rx,
                                     **({"seed": 2} if kind == "image" else kw))
    reference(render(EmuDevice, f, ["target"]), _swgl(f, ["target"]))


@pytest.mark.parametrize("cam", PERSP_CAMERAS)
@pytest.mark.parametrize("kind", ["opacity", "blend", "mix_blend"])
def test_perspective_picture_brushes(kind, cam, reference):
    """brush_opacity / brush_blend / brush_mix_blend drawing a picture's surface under a perspective node: fragment
    path only, varyings times w, mix(gl_FragCoord.w, 1, v_perspective) per sample (with and without
    BrushFlags::PERSPECTIVE_INTERPOLATION for opacity)."""
    d, ry, rx = cam
    kw = dict(seed=2)
    if kind == "opacity":
        kw.update(brush_flags=1)
    f = scenes.perspective_frame(kind, height=400 if kind != "opacity" else 360, d=d, ry=ry, rx=rx, **kw)
    reference(render(EmuDevice, f, ["target"]), _swgl(f, ["target"]))


@pytest.mark.parametrize("kw", [dict(), dict(d=220.0, ry=65.0, rx=20.0), dict(perspective_interpolate=1, seed=3),
                                dict(d=1e9, ry=0.0, rx=0.0, seed=4), dict(seed=5, filter=abi.NEAREST)])
def test_split_composite(kw, reference):
    """ps_split_composite: plane-split polygons (arbitrary convex quads) of a preserve-3d picture, with and
    without perspective (d=1e9: the 2-D edge walk and the span shader), clip masks, depth test."""
    f = scenes.split_composite_frame(**kw)
    reference(render(EmuDevice, f, ["target"]), _swgl(f, ["target"]))
