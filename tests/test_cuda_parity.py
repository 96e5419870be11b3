"""Parity tests proper: the CUDA backend (through the C ABI) against the CPU
oracle on the same seeded frames — bit-exact for this integer path."""
import numpy as np
import pytest

from oracle.backends import OracleDevice
from webrender_b200 import abi
from workloads import scenes
from webrender_b200.device import CudaDevice

from common import assert_same, reference, render  # noqa: F401 (reference: fixture)

pytestmark = pytest.mark.gpu

ALL_BLENDS = [b for b in range(abi.BLEND_COUNT) if b not in (abi.BLEND_SUBPIXEL_DUAL_SOURCE, abi.BLEND_CONSTANT_COLOR)]


@pytest.mark.parametrize("blend", ALL_BLENDS)
def test_blend_keys_random_layers(blend):
    f = scenes.alpha_rects_frame(515, 131, 48, random_rects=True, seed=100 + blend, blend=blend,
                                 color=None, clear_color=(0.4, 0.7, 0.2, 0.8))
    assert_same(render(CudaDevice, f), render(OracleDevice, f), f"blend={blend}")


@pytest.mark.parametrize("size", [(1, 1), (3, 2), (127, 7), (128, 8), (129, 9), (1000, 333), (2048, 64)])
def test_target_sizes_and_tile_edges(size):
    w, h = size
    f = scenes.alpha_rects_frame(w, h, 19, random_rects=True, seed=w * 7 + h)
    assert_same(render(CudaDevice, f), render(OracleDevice, f), f"size={size}")


def test_config_b_small_full_cover():
    f = scenes.alpha_rects_frame(640, 360, 300)
    assert_same(render(CudaDevice, f), render(OracleDevice, f))


def test_empty_batch_and_offscreen_rects():
    f = scenes.alpha_rects_frame(200, 100, 5, random_rects=True, seed=1)
    # move every rect off screen: nothing may change but the clear
    gf = f.tables["gpu_buffer_f"]
    gf[:, :] = np.where(np.arange(gf.shape[0])[:, None] % 5 < 2, gf + 5000.0, gf)
    assert_same(render(CudaDevice, f), render(OracleDevice, f))


def test_config_b_full_size_closed_form():
    """BASELINE config B at full size: 1000 full-frame alpha rects at 3840x2160.
    Size-independent property: every pixel sees the same layer sequence, so the
    frame is constant and equals the scalar recurrence of the blend equation."""
    w, h, n = 3840, 2160, 1000
    f = scenes.alpha_rects_frame(w, h, n)
    out = render(CudaDevice, f)["target"].reshape(h, w, 4)
    px = [0, 0, int(0.3 * 255 + 0.5), 255]  # clear colour (0.3,0,0,1) as B,G,R,A
    s = int(0.05 * 255.0 + 0.5)
    for _ in range(n):
        px = [min(255, s + d - ((d * s + d) >> 8)) for d in px]
    assert (out == np.array(px, dtype=np.uint8)).all()


def max_abs_diff(a, b):
    return int(np.abs(a.astype(np.int16) - b.astype(np.int16)).max())


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["plain", "fractional", "scaled"])
def test_brush_solid_opaque_alpha_masks_exact(seed, variant):
    """Opaque pass (depth LEQUAL + write, front to back) then alpha pass with
    per-instance clip masks: bit-exact."""
    f = scenes.brush_solid_frame(777, 431, n_opaque=20, n_alpha=40, seed=seed,
                                 fractional=variant == "fractional",
                                 device_pixel_scale=1.5 if variant == "scaled" else 1.0)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2])
def test_brush_solid_aa_no_depth_exact(seed):
    """Edge AA + clip masks without occluders: bit-exact (AA weights, mask-first
    ordering of solid span bodies)."""
    f = scenes.brush_solid_frame(640, 360, n_opaque=0, n_alpha=40, seed=seed, fractional=True, force_aa=True)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
def test_brush_solid_aa_with_occluders_exact(seed):
    """AA edges with opaque prims in the same pass: byte-exact (depth runs reproduced)."""
    f = scenes.brush_solid_frame(640, 360, n_opaque=12, n_alpha=40, seed=seed, fractional=True, force_aa=True)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled"])
def test_clip_rectangle_masks_bit_exact(seed, variant):
    """cs_clip_rectangle (fast + general, Clip/ClipOut, overwrite + multiply): R8 masks bit-exact."""
    f = scenes.clip_mask_frame(seed=seed, fractional=variant != "integer", scale=1.25 if variant == "scaled" else 1.0)
    assert_same(render(CudaDevice, f), render(OracleDevice, f), variant)


def test_clip_rectangle_large():
    f = scenes.clip_mask_frame(2048, 1024, n_clips=40, seed=9, fractional=True)
    assert_same(render(CudaDevice, f), render(OracleDevice, f))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled", "nearest"])
def test_rounded_rects_indirect(seed, variant):
    """Config A flavour: quad → off-screen, ps_quad_mask multiply, textured composite."""
    f = scenes.rounded_rects_frame(seed=seed, fractional=variant in ("fractional", "scaled"),
                                   device_pixel_scale=1.5 if variant == "scaled" else 1.0,
                                   filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    assert_same(render(CudaDevice, f), render(OracleDevice, f), variant)


IMAGE_VARIANTS = ["linear", "nearest", "linear_1to1", "nearest_1to1", "linear_fractional"]


def _image_frame(seed, variant, n_opaque):
    return scenes.image_frame(seed=seed, n_opaque=n_opaque, filter=abi.NEAREST if "nearest" in variant else abi.LINEAR,
                              one_to_one="1to1" in variant, fractional="fractional" in variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", IMAGE_VARIANTS)
def test_brush_image_unoccluded_exact(seed, variant):
    f = _image_frame(seed, variant, 0)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", IMAGE_VARIANTS)
def test_brush_image_occluded(seed, variant):
    """Opaque occluders inside the opaque batch (depth LEQUAL + write, front to back): every passing depth
    run is a span of its own (draw_depth_span, rasterize.h:612-657) — byte-exact for every filter path."""
    f = _image_frame(seed, variant, 8)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", IMAGE_VARIANTS + ["rotated"])
def test_brush_image_alpha_behind_opaque(seed, variant):
    """Alpha images partly hidden by opaque prims in front of them (what every page does): the alpha batch's
    spans are cut into depth runs whose chunk phase, span-shader body / fragment tail split and interpolant
    sums restart as the reference's do — byte-exact."""
    f = scenes.image_frame(seed=seed, n_opaque=8, filter=abi.NEAREST if "nearest" in variant else abi.LINEAR,
                           one_to_one="1to1" in variant, fractional="fractional" in variant or variant == "rotated",
                           rotate=23.0 if variant == "rotated" else None, occlude_alpha=True)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("rotate", [None, 17.0])
def test_brush_solid_aa_behind_opaque(seed, rotate):
    """AA edges and clip masks of alpha solids partly hidden by opaque prims: AA ramps and the mask-first
    ordering of solid span bodies follow the depth runs — byte-exact."""
    f = scenes.brush_solid_frame(640, 360, n_opaque=12, n_alpha=40, seed=seed, fractional=True, force_aa=True,
                                 occlude_alpha=True, rotate=rotate)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
def test_brush_image_repetition_behind_opaque(seed):
    f = scenes.image_repeat_frame(seed=seed, fractional=True, occlude_alpha=True)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


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
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


def test_text_run_config_c_size():
    """Config C flavour at full size: ~6000 glyphs on a 3840x2160 target, 2048^2 R8 atlas."""
    f = scenes.text_frame(width=3840, height=2160, n_runs=68, glyphs_per_run=89, seed=2, atlas_size=2048)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("variant", ["r8_alpha", "r8_fractional", "rgba_modes", "r8_shadow_masks"])
@pytest.mark.parametrize("n_runs,glyphs", [(40, 40), (12, 40)])
def test_text_run_dense_overlapping(n_runs, glyphs, variant):
    """Runs crossing one another on a small page: many glyphs overlap EARLIER glyphs of the batch, so the glyph-major
    kernel must leave them (and only them) to the ordered tile kernel — binned (1600 glyphs) and unbinned (480)."""
    f = _text_frame(3, variant, width=640, height=200, n_runs=n_runs, glyphs_per_run=glyphs)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


def test_text_run_tile_kernel_only(monkeypatch):
    """WRCU_GLYPH_MAJOR=0: the ordered tile kernel alone draws the batch (the path glyph-major falls back to)."""
    monkeypatch.setenv("WRCU_GLYPH_MAJOR", "0")
    f = _text_frame(2, "r8_fractional", width=640, height=200, n_runs=40, glyphs_per_run=40)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


GRADIENT_VARIANTS = ["opaque", "alpha", "fractional", "repeat", "full_frame"]


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", GRADIENT_VARIANTS)
def test_linear_gradient(seed, variant):
    f = scenes.gradient_frame(seed=seed, fractional=variant == "fractional", repeat=variant == "repeat",
                              full_frame=variant == "full_frame",
                              blend=abi.BLEND_PREMULTIPLIED_ALPHA if variant == "alpha" else abi.BLEND_NONE)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


def test_linear_gradient_config_d_size():
    """Config D: full-frame two-stop gradients at 3840x2160 (aligned + unaligned)."""
    f = scenes.gradient_frame(width=3840, height=2160, n_grad=4, full_frame=True)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


BOX_SHADOW_VARIANTS = ["integer", "fractional", "scaled", "nearest"]


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
@pytest.mark.parametrize("variant", BOX_SHADOW_VARIANTS)
def test_clip_box_shadow(seed, variant):
    f = scenes.box_shadow_frame(seed=seed, fractional=variant in ("fractional", "scaled"),
                                scale=1.5 if variant == "scaled" else 1.0)
    if variant == "nearest":
        f.textures["shadow"].filter = abi.NEAREST
    assert_same(render(CudaDevice, f, ["mask"]), render(OracleDevice, f, ["mask"]), variant)


def test_clip_box_shadow_config_d_size():
    """Config D: one 1024x1024 box-shadow mask instance (large-boxshadow-ellipse style)."""
    f = scenes.box_shadow_frame(width=1024, height=1024, n_clips=1, full_size=(1024, 1024), seed=7)
    assert_same(render(CudaDevice, f, ["mask"]), render(OracleDevice, f, ["mask"]))


COMPOSITE_VARIANTS = ["tiles", "fractional", "external", "external_fractional"]


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", COMPOSITE_VARIANTS)
def test_composite(seed, variant):
    f = scenes.composite_frame(seed=seed, external="external" in variant, fractional="fractional" in variant)
    assert_same(render(CudaDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]), variant)


def test_composite_4k():
    """Row 15 at full size: 4x5 picture-cache tiles of 1024x512 into a 3840x2160 framebuffer."""
    f = scenes.composite_frame(width=3840, height=2160, tile_w=1024, tile_h=512, seed=4)
    assert_same(render(CudaDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]))



@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", COMPOSITE_VARIANTS)
def test_composite_tile_lists(seed, variant):
    """wrcu_draw_composite_tiles: draw_tile_list (renderer/mod.rs:3126-3334) submitted as runs of
    instances with one texture each, against the reference's one draw per texture change."""
    f = scenes.composite_frame(seed=seed, external="external" in variant, fractional="fractional" in variant)
    assert_same(render(CudaDevice, f, ["fb"], tile_lists=True), render(OracleDevice, f, ["fb"]), variant)


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
    assert_same(render(CudaDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]), fmt)


@pytest.mark.parametrize("variant", YUV_VARIANTS[1:])
@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_composite_yuv_variants(fmt, variant):
    f = _yuv_frame(fmt, 2 if variant != "fractional" else 5, variant)
    assert_same(render(CudaDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]), variant)


@pytest.mark.parametrize("fmt", YUV_FORMATS)
def test_composite_yuv_4k_video(fmt):
    """A 1080p video frame scaled to the whole 3840x2160 framebuffer (the bench's video workloads)."""
    f = scenes.video_frame(3840, 2160, 1920, 1080, fmt)
    assert_same(render(CudaDevice, f, ["fb"]), render(OracleDevice, f, ["fb"]), fmt)


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
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


OPACITY_VARIANTS = ["scaled", "fractional", "one_to_one", "nearest"]


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", OPACITY_VARIANTS)
def test_brush_opacity(seed, variant):
    f = scenes.opacity_frame(seed=seed, fractional=variant == "fractional", one_to_one=variant == "one_to_one",
                             filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("r8", [False, True])
def test_ps_clear(seed, r8):
    f = scenes.clear_frame(seed=seed, r8=r8)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("variant", ["alpha", "fractional", "opaque"])
def test_brush_blend(seed, variant):
    """Bit-exact except the hue-rotate picture: its matrix comes from cosf/sinf,
    evaluated by the host libm in the reference and on the device here
    (correctly rounded via double) — at most 1 LSB apart on a few pixels."""
    import numpy as np
    f = scenes.blend_frame(seed=seed, fractional=variant == "fractional", opaque_source=variant == "opaque")
    a = render(CudaDevice, f, ["target"])["target"].astype(int)
    b = render(OracleDevice, f, ["target"])["target"].astype(int)
    hue = np.zeros(a.shape, dtype=bool)
    hue[0:140, 4 * (8 + 2 * 126 - 2):4 * (8 + 3 * 126 + 2)] = True   # filters[2] = hue-rotate cell
    assert (a[~hue] == b[~hue]).all()
    assert np.abs(a - b).max() <= 1 and (a != b).mean() < 2e-3


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["integer", "fractional"])
def test_brush_mix_blend(seed, variant):
    f = scenes.mix_blend_frame(seed=seed, fractional=variant == "fractional")
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


def test_async_readback_matches_sync():
    """wrcu_read_pixels_async into page-locked memory + fence == wrcu_read_pixels."""
    import numpy as np
    from webrender_b200.frame import draw_frame
    f = scenes.alpha_rects_frame(640, 360, 40, random_rects=True, seed=5, color=None)
    dev = CudaDevice(0)
    try:
        h = draw_frame(dev, f)
        want = dev.read_pixels(h["target"], 0, 0, 640, 360, 4)
        buf = dev.host_alloc((360, 640 * 4))
        buf[:] = 0
        fence = dev.read_pixels_async(h["target"], 0, 0, 640, 360, buf)
        # drawing to the same texture again must wait for the copy
        draw_frame(dev, f, h)
        dev.fence_wait(fence)
        assert (buf == want).all()
        dev.finish()
    finally:
        dev.close()


@pytest.mark.parametrize("rot", [17.0, -33.5, 90.0, 45.0, 180.0, 3.0])
@pytest.mark.parametrize("seed", [1, 2])
def test_rotated_brush_solid(rot, seed):
    """Non-axis-aligned quads through the edge-walk path (CMD_GENERAL)."""
    f = scenes.brush_solid_frame(seed=seed, rotate=rot, fractional=True, with_masks=seed == 2)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), f"rot {rot}")


@pytest.mark.parametrize("rot", [17.0, -33.5, 90.0])
@pytest.mark.parametrize("kind", ["image", "gradient_alpha", "gradient_opaque"])
def test_rotated_textured(rot, kind):
    if kind == "image":
        f = scenes.image_frame(seed=2, rotate=rot, fractional=True, n_opaque=0)
    elif kind == "gradient_alpha":
        f = scenes.gradient_frame(seed=2, rotate=rot, fractional=True, blend=abi.BLEND_PREMULTIPLIED_ALPHA)
    else:
        f = scenes.gradient_frame(seed=2, rotate=rot)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), kind)


def test_rotated_full_size():
    """A 4K frame of rotated brushes (rows up to 2160: long edge walks)."""
    f = scenes.brush_solid_frame(width=3840, height=2160, seed=3, rotate=23.0, fractional=True, with_masks=False,
                                 n_opaque=6, n_alpha=20)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("color", [False, True])
def test_cs_blur(seed, color):
    f = scenes.blur_frame(seed=seed, color=color)
    assert_same(render(CudaDevice, f, ["mid", "target"]), render(OracleDevice, f, ["mid", "target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["rgba", "r8", "nearest"])
def test_cs_scale(seed, variant):
    f = scenes.scale_frame(seed=seed, r8=variant == "r8", filter=abi.NEAREST if variant == "nearest" else abi.LINEAR)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


def test_binned_batch_mixed_sizes():
    """n >= 512 takes the bitmask-bin path: small commands scattered into per-tile
    masks, large ones through the wide mask; blend order must survive."""
    f = scenes.alpha_rects_frame(1920, 1080, 900, random_rects=True, seed=11, color=None)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


CS_GRADIENT_KINDS = {"fast_linear": abi.KIND_FAST_LINEAR_GRADIENT, "linear": abi.KIND_LINEAR_GRADIENT,
                     "radial": abi.KIND_RADIAL_GRADIENT, "conic": abi.KIND_CONIC_GRADIENT}


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["plain", "repeat", "hard"])
@pytest.mark.parametrize("kind", list(CS_GRADIENT_KINDS))
def test_cached_gradient_tasks(kind, variant, seed):
    """Cached gradient render tasks (draw_texture_cache_target).  Bit-exact; the
    conic gradient's angle comes from libm atan2f in the reference and from a
    correctly rounded atan2 on the device, so a conic pixel whose offset lands
    within an ulp of a LUT entry boundary may differ by 1 LSB."""
    f = scenes.cached_gradient_frame(CS_GRADIENT_KINDS[kind], seed=seed, repeat=variant == "repeat",
                                     hard=variant == "hard")
    a = render(CudaDevice, f, ["target"])["target"]
    b = render(OracleDevice, f, ["target"])["target"]
    if kind != "conic":
        assert (a == b).all(), (kind, variant, int((a != b).sum()))
        return
    d = np.abs(a.astype(int) - b.astype(int))
    # hard stops: a pixel exactly on the discontinuity may take either side
    bad = (d > 1).reshape(d.shape[0], -1, 4).any(axis=2)
    assert bad.sum() <= (8 if variant == "hard" else 0), (kind, variant, int(bad.sum()), int(d.max()))
    assert (d > 0).reshape(d.shape[0], -1, 4).any(axis=2).mean() < 1e-3


@pytest.mark.parametrize("kind", ["linear", "radial"])
def test_cached_gradient_full_width(kind):
    """One 3840-wide task: the span walks cross 30 tiles per row."""
    f = scenes.cached_gradient_frame(CS_GRADIENT_KINDS[kind], width=3840, height=64, n_tasks=1, seed=5,
                                     big=(3840, 64))
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), kind)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_line_decoration_tasks(seed):
    f = scenes.line_decoration_frame(seed=seed)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("scale", [1.0, 1.5])
@pytest.mark.parametrize("kind", ["solid", "segment"])
def test_border_tasks(kind, scale, seed):
    """cs_border_solid / cs_border_segment render tasks (draw_texture_cache_target)."""
    f = scenes.border_frame(abi.KIND_BORDER_SOLID if kind == "solid" else abi.KIND_BORDER_SEGMENT, seed=seed,
                            scale=scale)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), kind)


QUAD_GRADIENT_KINDS = {"radial": abi.KIND_QUAD_RADIAL_GRADIENT, "conic": abi.KIND_QUAD_CONIC_GRADIENT}


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("variant", ["integer", "fractional", "scaled", "rotated", "opaque"])
@pytest.mark.parametrize("kind", list(QUAD_GRADIENT_KINDS))
def test_quad_gradients(kind, variant, seed):
    """ps_quad_radial_gradient / ps_quad_conic_gradient (the conic's approx_atan2 is a
    polynomial, so both are bit-exact)."""
    f = scenes.quad_gradient_frame(QUAD_GRADIENT_KINDS[kind], seed=seed, fractional=variant in ("fractional", "scaled"),
                                   device_pixel_scale=1.5 if variant == "scaled" else 1.0,
                                   rotate=23.0 if variant == "rotated" else None,
                                   blend=abi.BLEND_NONE if variant == "opaque" else abi.BLEND_PREMULTIPLIED_ALPHA)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), kind + "/" + variant)


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
@pytest.mark.parametrize("variant", ["linear", "nearest", "fractional", "scaled"])
def test_brush_image_repetition(seed, variant):
    """brush_image REPETITION (tiled images, border-image segments): bit-exact."""
    f = scenes.image_repeat_frame(seed=seed, n_opaque=0, filter=abi.NEAREST if variant == "nearest" else abi.LINEAR,
                                  fractional=variant in ("fractional", "scaled"),
                                  device_pixel_scale=1.5 if variant == "scaled" else 1.0)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), variant)


@pytest.mark.parametrize("seed", [1, 2])
def test_brush_image_repetition_occluded(seed):
    """With opaque occluders in the same pass: the depth-run chunk-phase deviation of DESIGN.md §4.4
    (<= 2 LSB on a noise atlas, only on partially hidden primitives)."""
    f = scenes.image_repeat_frame(seed=seed, fractional=True, device_pixel_scale=1.5)
    a = render(CudaDevice, f, ["target"])["target"].astype(int)
    b = render(OracleDevice, f, ["target"])["target"].astype(int)
    d = np.abs(a - b)
    assert d.max() <= 2 and (d > 0).mean() < 5e-3, (int(d.max()), float((d > 0).mean()))


GLYPH_TRANSFORMS = {"identity": (0.0, 1.0, 1.0), "scaled": (0.0, 1.25, 0.8), "rotated": (17.0, 1.0, 1.0),
                    "rotated_scaled": (-33.0, 1.3, 0.9), "quarter_turn": (90.0, 1.0, 1.0)}


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("atlas", ["r8", "rgba"])
@pytest.mark.parametrize("xf", list(GLYPH_TRANSFORMS))
def test_text_run_glyph_transform(xf, atlas, seed):
    """ps_text_run GLYPH_TRANSFORM: quads trimmed per row by gl_ClipDistance; bit-exact."""
    f = scenes.text_frame(seed=seed, width=480, height=270, n_runs=8, glyphs_per_run=16, atlas=atlas,
                          color_modes=(0,) if atlas == "r8" else (0, 1, 2, 3), fractional=True,
                          glyph_transform=GLYPH_TRANSFORMS[xf], clip_runs=True)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), xf)


def test_binned_batch_two_list_passes():
    """9600 glyphs in one batch: the per-tile command list is built in two passes of 8192 commands."""
    f = scenes.text_frame(seed=4, width=1920, height=1080, n_runs=120, glyphs_per_run=80, atlas_size=1024)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]))


# ---- perspective quads / plane-split polygons: against the reference build itself -------------------------
# (the plain-C port does not restate draw_perspective: the expected bytes are the host emulation's, which the
# `reference` fixture holds to the digest of the reference build's output)
PERSP_CAMERAS = [(800.0, 35.0, 0.0), (800.0, -20.0, 15.0), (220.0, 60.0, -30.0), (220.0, 80.0, 40.0), (150.0, -70.0, 55.0)]


def _reference_pixels(reference, f, names):
    from emu import EmuDevice
    from oracle.backends import SwglDevice
    return reference(render(EmuDevice, f, names), lambda: render(SwglDevice, f, names))


@pytest.mark.parametrize("cam", PERSP_CAMERAS)
@pytest.mark.parametrize("kind", ["solid", "solid_aa", "image", "image_nearest", "quad"])
def test_perspective_brushes(kind, cam, reference):
    """draw_perspective (rasterize.h:1422-1545): near-plane clipping, polygon edge walk, per-sample z and
    1/w-corrected varyings — byte-exact against SWGL."""
    d, ry, rx = cam
    if kind == "quad":
        f = scenes.perspective_frame("quad", height=400, d=d, ry=ry, rx=rx, seed=2)
    elif kind.startswith("image"):
        f = scenes.perspective_frame("image", d=d, ry=ry, rx=rx, seed=2,
                                     filter=abi.NEAREST if kind == "image_nearest" else abi.LINEAR)
    else:
        f = scenes.perspective_frame("solid", d=d, ry=ry, rx=rx, seed=4 if kind == "solid_aa" else 3,
                                     force_aa=kind == "solid_aa", n_opaque=6, n_alpha=12)
    want = _reference_pixels(reference, f, ["target"])
    assert_same(render(CudaDevice, f, ["target"]), want, f"{kind} {cam}")


@pytest.mark.parametrize("cam", PERSP_CAMERAS[:4])
@pytest.mark.parametrize("kind", ["opacity", "blend", "mix_blend"])
def test_perspective_picture_brushes(kind, cam, reference):
    """brush_opacity / brush_blend / brush_mix_blend drawing a picture's surface under a perspective node —
    byte-exact against SWGL (hue-rotate's cosf/sinf aside: <= 1 LSB, DESIGN.md section 4.4)."""
    d, ry, rx = cam
    kw = dict(seed=2)
    if kind == "opacity":
        kw.update(brush_flags=1)
    f = scenes.perspective_frame(kind, height=400 if kind != "opacity" else 360, d=d, ry=ry, rx=rx, **kw)
    want = _reference_pixels(reference, f, ["target"])
    got = render(CudaDevice, f, ["target"])
    if kind == "blend":
        dd = np.abs(got["target"].astype(int) - want["target"].astype(int))
        assert dd.max() <= 1 and (dd != 0).mean() < 2e-3, (int(dd.max()), float((dd != 0).mean()))
    else:
        assert_same(got, want, f"{kind} {cam}")


def test_perspective_full_size(reference):
    """4K: long polygon edges (rows up to 2160) and spans up to 3840 samples of stepped z/w."""
    f = scenes.perspective_frame("solid", width=3840, height=2160, d=3000.0, ry=50.0, rx=-20.0, seed=5, n_opaque=4,
                                 n_alpha=10, with_masks=False)
    want = _reference_pixels(reference, f, ["target"])
    assert_same(render(CudaDevice, f, ["target"]), want)


@pytest.mark.parametrize("kw", [dict(), dict(d=220.0, ry=65.0, rx=20.0), dict(perspective_interpolate=1, seed=3),
                                dict(d=1e9, ry=0.0, rx=0.0, seed=4), dict(seed=5, filter=abi.NEAREST),
                                dict(seed=6, width=1920, height=1080, n_polys=40, d=900.0)])
def test_split_composite(kw, reference):
    f = scenes.split_composite_frame(**kw)
    want = _reference_pixels(reference, f, ["target"])
    assert_same(render(CudaDevice, f, ["target"]), want, str(kw))


@pytest.mark.parametrize("seed", [1, 2])
def test_page_of_many_small_batches(seed):
    """Three passes, ~40 draws of a few instances each (clip masks, picture-cache tiles with seven batches each,
    the tile list): what bench.py --workload page times at 4K."""
    f = scenes.page_frame(width=2048, height=1024, seed=seed)
    names = ["mask", "tile0", "tile1", "tile2", "tile3", "fb"]
    assert_same(render(CudaDevice, f, names), render(OracleDevice, f, names))
    assert_same(render(CudaDevice, f, ["fb"], tile_lists=True), render(OracleDevice, f, ["fb"]))


@pytest.mark.parametrize("rot", [17.0, -33.5])
def test_rotated_textured_quads(rot):
    """ps_quad_textured under a rotated spatial node (the Indirect path's composite quads): edge walk + textured spans."""
    f = scenes.rounded_rects_frame(seed=2, rotate=rot)
    assert_same(render(CudaDevice, f, ["target"]), render(OracleDevice, f, ["target"]), f"rot {rot}")
