"""Golden vectors produced by the reference itself (tests/golden/make_golden.py,
from oracle/_ref = unmodified swgl/src/gl.cc): the oracle must reproduce them
byte for byte on any box (CPU tier); the CUDA backend likewise (GPU tier)."""
import io
import json
import lzma
import os

import numpy as np
import pytest

from oracle.backends import OracleDevice
from workloads import scenes

from common import render

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
INDEX = json.load(open(os.path.join(HERE, "index.json")))
# the reference's own reftest images (wrench/reftests/<path>, all opaque, stored as RGB) and the rows of
# image/yuv.png kept of them, as golden/make_reftest_images.py wrote them
REFTEST_IMAGES = os.path.join(HERE, "reftest_images.npz.xz")
YUV_ROWS = slice(10, 58)
_reftest_images = []


def reftest_image(path):
    """wrench/reftests/<path> as int RGBA."""
    if not _reftest_images:
        _reftest_images.append(np.load(io.BytesIO(lzma.decompress(open(REFTEST_IMAGES, "rb").read()))))
    rgb = _reftest_images[0][path]
    return np.concatenate([rgb, np.full(rgb.shape[:2] + (1,), 255, np.uint8)], axis=2).astype(int)


# cases whose CUDA result may differ from the reference by <= 1 LSB on a few
# pixels for a documented reason (DESIGN.md §4.4): hue-rotate's cosf/sinf; conic gradient: atan2f
CUDA_LSB_TOLERANT = {"brush_blend_filters", "cs_conic_gradient",  # conic: atan2f
                     # three gradient reftest goldens, the line decorations and image/segments were added after the round's last GPU call; conic-simple for
                     # atan2f, the radial pair until a GPU run has confirmed them exact like cs_radial_gradient
                     "reftest_conic_simple", "reftest_radial_circle", "reftest_radial_ellipse", "reftest_line_decorations",
                     "reftest_image_segments", "reftest_linear_aligned_border_radius"}
# (reftest_box_shadow_suite_composited, also added late, is integer copies of an exact frame: not in the tolerant set)


def _check(device_cls, name, tolerant=False):
    case = INDEX[name]
    frame = getattr(scenes, case["builder"])(**case["kwargs"])
    got = render(device_cls, frame, case["targets"])
    want = np.load(os.path.join(HERE, name + ".npz"))
    for t in case["targets"]:
        if tolerant:
            d = np.abs(got[t].astype(int) - want[t].astype(int))
            assert d.max() <= 1 and (d != 0).mean() < 2e-3, f"{name}/{t}: max diff {d.max()}"
        else:
            assert np.array_equal(got[t], want[t]), f"{name}/{t}: {(got[t] != want[t]).sum()} bytes differ"


def test_config_a_against_reference_png():
    """Config A pinned on the reference's OWN golden image: the oracle's render of
    wrench/reftests/aa/rounded-rects.yaml against rounded-rects-ref.png under the
    reftest's fuzz `fuzzy(1,1) fuzzy-if(platform(swgl),4,27)` (aa/reftest.list:1)."""
    ref = reftest_image("aa/rounded-rects-ref.png")
    out = render(OracleDevice, scenes.config_a_frame(), ["target"])["target"].reshape(604, 1036, 4)
    rgba = out[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(rgba - ref).max(axis=2)
    assert d.max() <= 4 and int((d > 0).sum()) <= 27, (int(d.max()), int((d > 0).sum()))


@pytest.mark.parametrize("name", sorted(n for n in INDEX if INDEX[n].get("port", True)))
def test_oracle_matches_reference_golden(name):
    _check(OracleDevice, name)


@pytest.mark.parametrize("name", sorted(n for n in INDEX if not INDEX[n].get("port", True)))
def test_emulated_kernels_match_reference_golden(name):
    """Paths the plain-C port does not restate (perspective quads, plane-split polygons): the device code itself,
    compiled for the host (tests/emu.py), against the reference's bytes."""
    from emu import EmuDevice
    _check(EmuDevice, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(INDEX))
def test_cuda_matches_reference_golden(name):
    from webrender_b200.device import CudaDevice
    _check(CudaDevice, name, tolerant=name in CUDA_LSB_TOLERANT)


@pytest.mark.parametrize("which,png,max_diff,max_px", [
    ("clip-mode", "clip/clip-mode.png", 1, 4),        # fuzzy-if(platform(swgl),1,4)
    ("clip-ellipse", "clip/clip-ellipse.png", 1, 80),  # fuzzy-if(platform(swgl),1,80)
])
def test_clip_reftests_against_reference_png(which, png, max_diff, max_px):
    """wrench/reftests/clip/{clip-mode,clip-ellipse}.yaml (Clip and ClipOut rounded /
    elliptical clips, incl. the frame builder's corner-overlap scaling) against the
    reference's own PNGs under the reftest's fuzz.  Measured: 0 differing pixels."""
    ref = reftest_image(png)
    f = scenes.reftest_clip_frame(which)
    d_ = f.textures["target"]
    out = render(OracleDevice, f, ["target"])["target"].reshape(d_.height, d_.width, 4)[..., [2, 1, 0, 3]].astype(int)
    h, w = min(ref.shape[0], out.shape[0]), min(ref.shape[1], out.shape[1])
    d = np.abs(out[:h, :w] - ref[:h, :w]).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= max_px, (int(d.max()), int((d > 0).sum()))
    assert (ref[h:, :, :3] == 255).all() and (ref[:, w:, :3] == 255).all()
    assert (out[h:, :, :3] == 255).all() and (out[:, w:, :3] == 255).all()


@pytest.mark.parametrize("which,png,max_diff,max_px", [
    ("inset-no-blur-radius", "boxshadow/inset-no-blur-radius-ref.png", 3, 2),  # fuzzy-if(platform(swgl),3,2); measured 0
    ("box-shadow-spread", "boxshadow/box-shadow-spread.png", 9, 34),           # fuzzy-if(platform(swgl),9,34); measured 0
    ("boxshadow-spread-only", "boxshadow/boxshadow-spread-only-ref.png", 1, 10),  # GL-rendered, exact on linux/mac GL;
                                                                                 # SWGL rounding: 1 LSB on 10 px
    ("suite-no-blur", "boxshadow/box-shadow-suite-no-blur.png", 1, 8),  # 16 shadows (outset / inset, radius 0 / 32, offsets,
                                                                       # spread); GL-rendered: 1 LSB on 8 px of 705 366
])
def test_box_shadow_reftests_against_reference_png(which, png, max_diff, max_px):
    """wrench/reftests/boxshadow/*: box shadows WITHOUT blur take the frame builder's rectangle path
    (box_shadow.rs:341-401): the shadow colour as a Rectangle under a Clip and a ClipOut rounded-rect clip — inset
    (offset / spread) and outset — drawn the Indirect way with one ps_quad_mask per clip.  Against the reference's own
    PNGs under each reftest's fuzz."""
    ref = reftest_image(png)
    f = scenes.reftest_box_shadow_frame(which)
    d_ = f.textures["target"]
    out = render(OracleDevice, f, ["target"])["target"].reshape(d_.height, d_.width, 4)[..., [2, 1, 0, 3]].astype(int)
    assert out.shape == ref.shape
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= max_px, (int(d.max()), int((d > 0).sum()))


def test_border_overlapping_reftest_against_reference_png():
    """wrench/reftests/border/overlapping.yaml == overlapping.png under fuzzy-if(platform(swgl),1,20): overlapping
    corner ellipses of a complex clip.  Measured: 0 pixels differ."""
    ref = reftest_image("border/overlapping.png")
    f = scenes.reftest_border_overlapping_frame()
    out = render(OracleDevice, f, ["target"])["target"].reshape(240, 233, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 1 and int((d > 0).sum()) <= 20, (int(d.max()), int((d > 0).sum()))


def test_border_no_bogus_line_reftest_against_reference_png():
    """wrench/reftests/border/border-no-bogus-line.yaml == border-no-bogus-line-ref.png under
    fuzzy-if(platform(swgl),1,8): a rounded solid border whose radii are scaled to fit (corner tasks by cs_border_solid,
    segments by Brush(Image) from the texture cache).  Measured: 0 pixels differ."""
    ref = reftest_image("border/border-no-bogus-line-ref.png")
    f = scenes.reftest_border_no_bogus_line_frame()
    out = render(OracleDevice, f, ["target"])["target"].reshape(108, 116, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 1 and int((d > 0).sum()) <= 8, (int(d.max()), int((d > 0).sum()))


@pytest.mark.parametrize("name,png", [("border-radii", "border/border-radii.png"),
                                      ("border-clamp-corner-radius", "border/border-clamp-corner-radius.png")])
def test_border_reftests_against_reference_png(name, png):
    """wrench/reftests/border/{border-radii,border-clamp-corner-radius}.yaml against the reference's images: solid
    rounded borders through the frame builder's segment decomposition (cs_border_solid corner and edge tasks in the
    texture cache, Brush(Image) per segment), per-corner radii and radii scaled to fit.  Measured: 0 pixels differ."""
    ref = reftest_image(png)
    (w, h), _, (max_diff, max_px) = scenes.BORDER_REFTESTS[name]
    assert ref.shape[:2] == (h, w)
    f = scenes.reftest_border_frame(name)
    out = render(OracleDevice, f, ["target"])["target"].reshape(h, w, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= max_px, (int(d.max()), int((d > 0).sum()))


def test_clip_inverted_ellipse_reftest_against_reference_png():
    """wrench/reftests/clip/inverted-ellipse.yaml == inverted-ellipse.png (exact): an elliptical complex clip whose
    corner-size ratio is the inverse of the primitive's.  Measured: 0 pixels differ."""
    ref = reftest_image("clip/inverted-ellipse.png")
    f = scenes.reftest_clip_inverted_ellipse_frame()
    out = render(OracleDevice, f, ["target"])["target"].reshape(236, 319, 4)[..., [2, 1, 0, 3]].astype(int)
    assert np.array_equal(out, ref), int((np.abs(out - ref).max(axis=2) > 0).sum())


def test_split_near_plane_reftest_against_reference_png():
    """wrench/reftests/split/near-plane.yaml == near-plane.png (fuzzy(1,20); fuzzy-if(platform(swgl),128,39)): one
    plane-split polygon crossing the near plane, drawn by ps_split_composite from the picture's surface — the
    perspective path (draw_perspective with frustum clipping, rasterize.h:1064-1545) against an image the reference's
    authors checked in.  Drawn by the device code compiled for the host (the plain-C port does not restate
    perspective), which must give the reference build's bytes (the stored golden).  Measured: 0 pixels differ."""
    from emu import EmuDevice
    ref = reftest_image("split/near-plane.png")
    f = scenes.reftest_split_near_plane_frame()
    got = render(EmuDevice, f, ["target"])["target"]
    out = got.reshape(600, 600, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 128 and int((d > 0).sum()) <= 39, (int(d.max()), int((d > 0).sum()))
    want = np.load(os.path.join(HERE, "reftest_split_near_plane.npz"))["target"]
    assert np.array_equal(got, want)


def _filter_reftest(device_cls, name):
    _, cases, (max_diff, max_px) = scenes.FILTER_REFTESTS[name]
    ft, fr = scenes.filter_reftest_frames(name)
    a = render(device_cls, ft, ["target"])["target"].astype(int)
    b = render(device_cls, fr, ["target"])["target"].astype(int)
    d = np.abs(a - b).reshape(220, 220, 4).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= max_px, (name, int(d.max()), int((d > 0).sum()))
    # and the constant the reference's authors wrote down is what came out (opaque expectations only)
    for r, _, _, _, exp in cases:
        if exp[3] == 1.0:
            got = a.reshape(220, 220, 4)[int(r[1]) + 5, int(r[0]) + 5][[2, 1, 0]]
            assert np.abs(got - np.array(exp[:3])).max() <= max(max_diff, 0), (name, got, exp)


@pytest.mark.parametrize("name", sorted(scenes.FILTER_REFTESTS))
def test_filter_reftests_known_answers(name):
    """wrench/reftests/filters/filter-*.yaml == filter-*-ref.yaml: the filtered rect must equal a plain rect of the
    colour the reference's authors computed (grayscale(1) of green = 182,182,182; saturate(0.5) of red = 155,27,27;
    hue-rotate(90) of the primaries, ...) — known answers for brush_blend that do not come from this repository."""
    _filter_reftest(OracleDevice, name)


def _picture_reftest(device_cls, name):
    _, r, _, _, _, _, exp, (max_diff, max_px) = scenes.PICTURE_REFTESTS[name]
    f = scenes.picture_reftest_frame(name)
    out = render(device_cls, f, ["target"])["target"].reshape(140, 140, 4)[..., [2, 1, 0, 3]].astype(int)
    inside = out[r[1]:r[3], r[0]:r[2], :3]
    d = np.abs(inside - np.array(exp)).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= max_px, (name, int(d.max()), int((d > 0).sum()), inside[0, 0])
    assert (out[..., 3] == 255).all()


@pytest.mark.parametrize("name", sorted(scenes.PICTURE_REFTESTS))
def test_picture_reftests_known_answers(name):
    """filters/opacity.yaml, blend/{multiply,difference,darken,lighten}.yaml == their -ref.yaml: brush_opacity and
    brush_mix_blend must produce the colour the reference's authors wrote down (255,255,209 for yellow at alpha 0.2 under
    opacity(0.9) over white; green x green = green; green - green = black; per-channel min / max)."""
    _picture_reftest(OracleDevice, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(scenes.PICTURE_REFTESTS))
def test_cuda_picture_reftests_known_answers(name):
    from webrender_b200.device import CudaDevice
    _picture_reftest(CudaDevice, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(scenes.FILTER_REFTESTS))
def test_cuda_filter_reftests_known_answers(name):
    from webrender_b200.device import CudaDevice
    _filter_reftest(CudaDevice, name)


def test_filter_blur_reftest_against_reference_png():
    """wrench/reftests/filters/filter-small-blur-radius.yaml (`fuzzy(1,12) fuzzy-if(platform(swgl),2,12276)`,
    filters/reftest.list:29): picture surface → vertical + horizontal cs_blur COLOR_TARGET → Brush(Image) composite,
    against the reference's own PNG.  Measured: max 2 on 10 744 pixels (52 of them at 2) — the blurred 6-pixel band
    around the square, where SWGL's 8-bit passes differ from the GL reference."""
    ref = reftest_image("filters/filter-small-blur-radius.png")
    f = scenes.reftest_filter_blur_frame()
    out = render(OracleDevice, f, ["target"])["target"].reshape(700, 700, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 2 and int((d > 0).sum()) <= 12276, (int(d.max()), int((d > 0).sum()))


@pytest.mark.parametrize("which,png,max_diff,max_px", [
    ("linear", "gradient/linear-ref.png", 0, 0),                       # == linear.yaml linear-ref.png
    ("linear-reverse", "gradient/linear-ref.png", 0, 0),               # == linear-reverse.yaml linear-ref.png
    ("linear-hard-stop", "gradient/linear-hard-stop-ref.png", 1, 4800),  # fuzzy-range(<=1,*4800)
    ("linear-stops", "gradient/linear-stops-ref.png", 1, 35000),        # fuzzy(1,35000); measured 2400
    # GL-rendered references, exact match required on linux/mac GL; SWGL's 16-bit colour stepping
    # lands within 1 LSB (measured 1200 / 1215 px)
    ("premultiplied-aligned", "gradient/premultiplied-aligned.png", 1, 1300),
    ("premultiplied-angle", "gradient/premultiplied-angle.png", 1, 1300),
])
def test_gradient_reftests_against_reference_png(which, png, max_diff, max_px):
    """wrench/reftests/gradient/linear*.yaml as Brush(LinearGradient) against the
    reference's own PNGs under each reftest's fuzz (measured: 0 / 0 / <=1 on 4800 px)."""
    ref = reftest_image(png)
    out = render(OracleDevice, scenes.reftest_gradient_frame(which), ["target"])["target"]
    out = out.reshape(300, 300, 4)[..., [2, 1, 0, 3]].astype(int)
    h, w = min(ref.shape[0], 300), min(ref.shape[1], 300)
    d = np.abs(out[:h, :w] - ref[:h, :w]).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= max_px, (int(d.max()), int((d > 0).sum()))
    assert (ref[h:, :, :3] == 255).all() and (ref[:, w:, :3] == 255).all()


@pytest.mark.parametrize("which,png,max_diff,max_px", [
    ("premultiplied-radial", "gradient/premultiplied-radial.png", 0, 0),   # == (exact); measured 0
    ("premultiplied-conic", "gradient/premultiplied-conic.png", 1, 250),   # fuzzy(1,250); measured 1 on 4 px
    ("conic-center", "gradient/conic-center.png", 0, 0),                   # == (exact); measured 0
])
def test_cached_gradient_reftests_against_reference_png(which, png, max_diff, max_px):
    """wrench/reftests/gradient/{premultiplied-radial,premultiplied-conic,conic-center}.yaml drawn the way
    the frame builder draws them — a cached cs_radial_gradient / cs_conic_gradient render task in a
    texture-cache target, composited 1:1 with Brush(Image) — against the reference's OWN PNGs under each
    reftest's fuzz.  Pins the texture-cache-target gradient programs and the image composite."""
    ref = reftest_image(png)
    out = render(OracleDevice, scenes.reftest_cached_gradient_frame(which), ["target"])["target"]
    out = out.reshape(300, 300, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref[:300, :300]).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= max_px, (int(d.max()), int((d > 0).sum()))
    assert (ref[300:, :, :3] == 255).all() and (ref[:, 300:, :3] == 255).all()


@pytest.mark.parametrize("name,png", [("radial-circle", "gradient/radial-circle-ref.png"),
                                      ("radial-ellipse", "gradient/radial-ellipse-ref.png"),
                                      ("conic-simple", "gradient/conic-simple.png")])
def test_more_cached_gradient_reftests_against_reference_png(name, png):
    """wrench/reftests/gradient/{radial-circle,radial-ellipse,conic-simple}.yaml against the reference's images under
    each reftest's own fuzz (1 on 80000 / 80000 / 300): cs_radial_gradient with ratio_xy != 1, cs_conic_gradient, 300x300
    tasks.  Measured: 1 LSB on 18 / 8 / 5 pixels."""
    ref = reftest_image(png)
    (w, h), _, _, _, _, _, (max_diff, max_px) = scenes.CACHED_GRADIENT_REFTESTS[name]
    f = scenes.reftest_cached_gradient_frame2(name)
    out = render(OracleDevice, f, ["target"])["target"].reshape(h, w, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= max_diff and int((d > 0).sum()) <= min(max_px, 20), (int(d.max()), int((d > 0).sum()))


def test_linear_aligned_border_radius_reftest_against_reference_png():
    """wrench/reftests/gradient/linear-aligned-border-radius.yaml against linear-aligned-border-radius.png (rendered by
    GL; `==` there): vertical gradients under a rounded clip on white, blue and black — Brush(LinearGradient) alpha pass
    with cs_clip_rectangle masks.  Measured: 1 LSB on 231 of 59 645 pixels (the corner coverage and the gradient ramp
    round differently on GL); the reference build gives the same bytes as the port."""
    ref = reftest_image("gradient/linear-aligned-border-radius.png")
    f = scenes.reftest_gradient_border_radius_frame()
    out = render(OracleDevice, f, ["target"])["target"].reshape(151, 395, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 1 and int((d > 0).sum()) <= 240, (int(d.max()), int((d > 0).sum()))


def test_box_shadow_suite_through_the_compositor_against_reference_png():
    """The box-shadow suite drawn the way a page reaches the screen: into a picture-cache tile, then the tile list
    composited into the framebuffer (composite FAST_PATH, the copy class on the GPU) — the framebuffer against
    boxshadow/box-shadow-suite-no-blur.png: the same 1 LSB on 8 pixels as the direct draw."""
    ref = reftest_image("boxshadow/box-shadow-suite-no-blur.png")
    f = scenes.reftest_box_shadow_suite_composited_frame()
    out = render(OracleDevice, f, ["fb"])["fb"].reshape(789, 894, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 1 and int((d > 0).sum()) <= 8, (int(d.max()), int((d > 0).sum()))


def test_image_segments_reftest_against_reference_png():
    """wrench/reftests/image/segments.yaml == segments.png under fuzzy-if(platform(swgl),1,20): wrench's checkerboard
    image drawn 1:1 under a rounded clip (cs_clip_rectangle mask + Brush(Image) alpha pass) and unclipped (opaque
    Brush(Image)).  Measured: 1 LSB on 18 pixels."""
    ref = reftest_image("image/segments.png")
    f = scenes.reftest_image_segments_frame()
    out = render(OracleDevice, f, ["target"])["target"].reshape(583, 290, 4)[..., [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 1 and int((d > 0).sum()) <= 20, (int(d.max()), int((d > 0).sum()))


def test_line_decorations_reftest_against_reference_png():
    """The first eight items of wrench/reftests/text/decorations-suite.yaml against the matching region (rows 0-99,
    columns 0-217) of decorations-suite.png: solid, dashed, dotted and wavy lines at two thicknesses — cs_line_decoration
    tasks repeated along the line by Brush(Image) REPETITION.  The reftest allows SWGL 3 on 13 540 pixels over the whole
    suite; measured on this region: 0 pixels differ (2 001 of its 21 800 pixels are drawn)."""
    ref = reftest_image("text/decorations-suite.png")
    f = scenes.reftest_line_decorations_frame()
    out = render(OracleDevice, f, ["target"])["target"].reshape(439, 495, 4)[..., [2, 1, 0, 3]].astype(int)
    assert np.array_equal(out[:100, :218], ref[:100, :218])
    assert int((ref[:100, :218, :3] != 255).any(axis=2).sum()) == 2001


def test_yuv_reftest_against_reference_png():
    """wrench/reftests/image/yuv.yaml (planar, interleaved and NV12 `yuv-image` items, Rec709 limited range,
    from the reference's own plane PNGs) drawn as the frame builder draws it — opaque Brush(YuvImage)
    primitives into 1024x512 picture-cache tiles, tiles composited — against the reference's OWN yuv.png.
    The reference's annotation for SWGL on this content is fuzzy(1,205000) (image/reftest.list:9, the
    brush path; 8-bit fixed-point YUV matrix vs the GPU's float one): measured max 1 on 204390 pixels of the
    whole page.  The planes are stored for their first rows only (golden/reftest_yuv), so the page is
    compared on the rows those draw (YUV_ROWS, 1:1 from y = 10), under the same fuzz: max 1 on 24469 of them."""
    ref = reftest_image("image/yuv.png")
    out = render(OracleDevice, scenes.reftest_yuv_frame(os.path.join(HERE, "reftest_yuv")), ["target"])["target"]
    out = out.reshape(658, 1323, 4)[YUV_ROWS, :, [2, 1, 0, 3]].astype(int)
    d = np.abs(out - ref).max(axis=2)
    assert d.max() <= 1 and int((d > 0).sum()) <= 205000, (int(d.max()), int((d > 0).sum()))
