"""10-, 12- and 16-bit YUV video: R16 / RG16 planes through `composite` YUV, brush_yuv_image and CompositeYUV.

The plain-C port restates 8-bit video only, so the expected bytes are the host emulation's (tests/emu.py), which
the `reference` fixture holds to the digest of the unmodified reference rasteriser's output for the same input
(golden/yuv_high_bit_depth_digests.json, written by golden/make_yuv_high_bit_depth_digests.py).
CPU tier: the emulation against those digests.  GPU tier: the CUDA kernels against the same expected bytes."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from webrender_b200 import abi, draw_frame
from webrender_b200.device import WrcuError
from workloads import scenes

from common import RECORD_ENV, assert_same, digest, render
from emu import EmuDevice

DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "yuv_high_bit_depth_digests.json")
_digests = {}


@pytest.fixture
def reference(request):
    """common.reference over this module's digest file: check(got, live, part=None) -> got, where `got` must be byte
    for byte what the unmodified reference rasteriser drew; `live()` draws it with the reference build and runs only
    when recording (RECORD_ENV names the file to append to), after which a GPU test ends."""
    base = f"{request.node.module.__name__}::{request.node.name}"

    def check(got, live, part=None):
        key = base if part is None else f"{base}/{part}"
        record = os.environ.get(RECORD_ENV)
        if record:
            want = live()
            assert_same(got, want, key)
            with open(record, "a") as f:
                f.write(json.dumps({key: digest(want)}) + "\n")
            if request.node.get_closest_marker("gpu"):
                pytest.skip("reference recorded; the rest of this test needs a GPU")
            return got
        if not _digests:
            _digests.update(json.load(open(DIGESTS)))
        assert key in _digests, f"{key}: no stored reference digest (golden/make_yuv_high_bit_depth_digests.py)"
        assert digest(got) == _digests[key], f"{key}: differs from the reference rasteriser's output"
        return got
    return check


# GL internal formats / transfers of the 16-bit planes (gl_defs.h; gl.cc:257-285, 1755-1757)
GL_R16, GL_RG16, GL_RED, GL_RG, GL_UNSIGNED_SHORT = 0x822A, 0x822C, 0x1903, 0x8227, 0x1403


def _swgl_device(lib_path=None):
    """SwglDevice (the reference build, or any library with its GL surface) that also creates R16 / RG16 textures"""
    from oracle.backends import SwglDevice
    SwglDevice._IFMT.setdefault(abi.FMT_R16, GL_R16)
    SwglDevice._IFMT.setdefault(abi.FMT_RG16, GL_RG16)
    SwglDevice._XFER.setdefault(abi.FMT_R16, (GL_RED, GL_UNSIGNED_SHORT))
    SwglDevice._XFER.setdefault(abi.FMT_RG16, (GL_RG, GL_UNSIGNED_SHORT))
    return SwglDevice(lib_path)


def _reference_pixels(reference, f, names, part=None):
    return reference(render(EmuDevice, f, names), lambda: render(_swgl_device, f, names), part)


# ---- frames ---------------------------------------------------------------------------------------------------
COMPOSITE_FORMATS = [("planar", 10), ("planar", 12), ("planar", 16), ("nv12", 10), ("p010", 10), ("p010", 16)]
COMPOSITE_VARIANTS = ["blend", "fractional", "nearest", "right_edge"]
IMAGE_VARIANTS = ["opaque", "alpha", "fractional", "rotated", "nearest"]


def _composite(fmt, depth, color_space=2, variant="opaque"):
    return scenes.hdr_yuv_composite_frame(fmt, depth, color_space, seed=1 + color_space, linear=variant != "nearest",
                                          opaque=variant != "blend", fractional=variant == "fractional",
                                          right_edge=variant == "right_edge")


def _image(fmt, variant, color_space=2):
    return scenes.hdr_yuv_image_frame(fmt, 10, color_space, seed=1 + color_space, linear=variant != "nearest",
                                      alpha_pass=variant != "opaque", fractional=variant == "fractional",
                                      rotate=17.0 if variant == "rotated" else None)


def _composite_cases():
    cases = [(f"{fmt}{d}", _composite, (fmt, d)) for fmt, d in COMPOSITE_FORMATS]
    cases += [(f"{fmt}10_cs{cs}", _composite, (fmt, 10, cs)) for fmt in ("planar", "p010") for cs in range(7)]
    cases += [(f"{fmt}10_{v}", _composite, (fmt, 10, 5 if v == "fractional" else 2, v))
              for fmt in ("planar", "p010") for v in COMPOSITE_VARIANTS]
    return cases


def _image_cases():
    return [(f"{fmt}10_{v}", _image, (fmt, v, 5 if v == "fractional" else 2))
            for fmt in ("planar", "p010") for v in IMAGE_VARIANTS]


def _target(f):
    return "fb" if "fb" in f.textures else "target"


# ---- CPU tier: the device functions on the host against the reference build -----------------------------------
@pytest.mark.parametrize("case", _composite_cases(), ids=lambda c: c[0])
def test_composite_yuv_high_bit_depth(case, reference):
    """composite YUV with R16 / RG16 planes: PLANAR 10/12/16, NV12 10-bit, P010 10/16-bit; every colour space;
    opaque and premultiplied over, fractional rects, NEAREST planes (fragment path), flips, clips and uv rects
    that reach the last texel column (the 16-bit fetches' 127/128 edge weight)."""
    _, make, args = case
    f = make(*args)
    got = _reference_pixels(reference, f, [_target(f)])
    assert (got["fb"].reshape(320, 512, 4)[..., :3] != np.array([77, 51, 26], np.uint8)).any(axis=2).sum() > 10000


@pytest.mark.parametrize("case", _image_cases(), ids=lambda c: c[0])
def test_brush_yuv_image_high_bit_depth(case, reference):
    """Brush(YuvImage) with 10-bit PLANAR and P010 planes: opaque pass, alpha pass with AA edges and clip masks, a
    rotated spatial node, NEAREST planes."""
    _, make, args = case
    f = make(*args)
    _reference_pixels(reference, f, [_target(f)])


def _sw_cases():
    from test_gl_shim import SW_COMPOSITE_YUV_CASES
    return SW_COMPOSITE_YUV_CASES


def sw_yuv_planes16(case, depth):
    """LSB-aligned 16-bit planes over the geometry of a SW_COMPOSITE_YUV_CASES entry, every code of `depth` bits"""
    _, (yw, yh), (cw, ch), _, _, _, _, _, _ = case
    rng = np.random.RandomState(depth)
    top = 1 << depth
    y, u, v = (rng.randint(0, top, s).astype(np.uint16) for s in ((yh, yw), (ch, cw), (ch, cw)))
    return y, u, v, rng.randint(0, 256, (360, 640 * 4)).astype(np.uint8)


def run_sw_composite_yuv16(dev, case, planes, depth, via=None):
    """Uploads R16 planes, runs CompositeYUV at `depth` (through `via` when given), returns the destination."""
    _, (yw, yh), (cw, ch), cs, sr, dr, fx, fy, cr = case
    yp, up, vp, dst = planes
    ty, tu, tv = (dev.texture_create(abi.FMT_R16, yw, yh), dev.texture_create(abi.FMT_R16, cw, ch),
                  dev.texture_create(abi.FMT_R16, cw, ch))
    td = dev.texture_create(abi.FMT_RGBA8, 640, 360)
    dev.texture_upload(ty, 0, 0, yw, yh, yp)
    dev.texture_upload(tu, 0, 0, cw, ch, up)
    dev.texture_upload(tv, 0, 0, cw, ch, vp)
    dev.texture_upload(td, 0, 0, 640, 360, dst)
    if via is None:
        dev.sw_composite_yuv(td, ty, tu, tv, cs, sr, dr, fx, fy, cr, color_depth=depth)
        return dev.locked_pixels(td)
    via(dev, td, ty, tu, tv, cs, sr, dr, fx, fy, cr)
    return dev.read_pixels(td, 0, 0, 640, 360, 4)


def _blit_yuv(dev, lib, prefix, depth):
    I4 = C.c_int32 * 4

    def via(e, td, ty, tu, tv, cs, sr, dr, fx, fy, cr):
        f = getattr(lib, prefix + "composite_blit_yuv")
        f.argtypes = [C.c_void_p] + [C.c_uint32] * 4 + [C.c_int, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                                     C.c_int, C.c_int, C.POINTER(C.c_int32)]
        e._check(f(e.ctx, td, ty, tu, tv, int(cs), depth, I4(*sr), I4(*dr), int(fx), int(fy), I4(*cr)))
    return via


def _emu_composite_yuv16(case, planes, depth):
    e = EmuDevice()
    try:
        return {"dst": run_sw_composite_yuv16(e, case, planes, depth, via=_blit_yuv(e, e.lib, "wremu_", depth))}
    finally:
        e.close()


def _swgl_composite_yuv16(case, planes, depth):
    d = _swgl_device()
    try:
        return {"dst": run_sw_composite_yuv16(d, case, planes, depth)}
    finally:
        d.close()


@pytest.mark.parametrize("depth", [10, 12, 16])
def test_sw_compositor_yuv_blit_r16(depth, reference):
    """CompositeYUV with three R16 planes at colorDepth 10 / 12 / 16 (linear_row_yuv's R16 branch,
    composite.h:1025-1058) over every geometry of the 8-bit cases: 4:2:0 / 4:2:2 / 4:4:4, scaling, flips, clips."""
    for case in _sw_cases():
        planes = sw_yuv_planes16(case, depth)
        got = reference(_emu_composite_yuv16(case, planes, depth), lambda: _swgl_composite_yuv16(case, planes, depth),
                        part=case[0])
        assert (got["dst"] != planes[3]).any()


@pytest.mark.parametrize("fmt", [abi.FMT_R16, abi.FMT_RG16])
def test_texture_round_trip_16bit(fmt):
    """R16 / RG16 textures: upload, batched upload, copy and read-back move the bytes unchanged."""
    bpp = abi.FMT_BPP[fmt]
    rng = np.random.RandomState(fmt)
    w, h = 37, 23
    img = rng.randint(0, 256, (h, w * bpp)).astype(np.uint8)
    e = EmuDevice()
    try:
        t = e.texture_create(fmt, w, h)
        e.texture_upload(t, 0, 0, w, h, img)
        assert (e.read_pixels(t, 0, 0, w, h, bpp) == img).all()
        patch = rng.randint(0, 256, (2, 5 * 7 * bpp)).astype(np.uint8).reshape(-1)
        stride = 7 * bpp
        e.texture_upload_batch(t, [(3, 4, 7, 5, 0, stride), (20, 11, 6, 4, 5 * stride, stride)], patch)
        want = img.copy()
        want[4:9, 3 * bpp:10 * bpp] = patch[:5 * stride].reshape(5, stride)
        want[11:15, 20 * bpp:26 * bpp] = patch[5 * stride:5 * stride + 4 * stride].reshape(4, stride)[:, :6 * bpp]
        assert (e.read_pixels(t, 0, 0, w, h, bpp) == want).all()
        t2 = e.texture_create(fmt, w, h)
        e.texture_copy(t, t2, (2, 3, 30, 17), 5, 6)
        got = e.read_pixels(t2, 5, 6, 30, 17, bpp)
        assert (got == want[3:20, 2 * bpp:32 * bpp]).all()
    finally:
        e.close()


def _patch_composite(f, **kw):
    """the frame with every composite instance's params changed (float index 14 = YuvFormat, 15 = bit depth)"""
    for op in f.passes[0][0].ops:
        if hasattr(op, "instances"):
            fl = np.ascontiguousarray(op.instances).view(np.float32).copy()
            if "format" in kw:
                fl[:, 14] = kw["format"]
            if "depth" in kw:
                fl[:, 15] = kw["depth"]
            op.instances = fl.view(np.uint8)
    return f


def _mismatched():
    from webrender_b200.gpu_types import YUV_FORMAT_NV16
    r16_depth8 = _patch_composite(_composite("planar", 10), depth=8)
    r8_depth10 = _patch_composite(scenes.yuv_composite_frame("planar"), depth=10)
    nv12_r8_depth10 = _patch_composite(scenes.yuv_composite_frame("nv12"), depth=10)
    nv16 = _patch_composite(_composite("nv12", 10), format=YUV_FORMAT_NV16)
    p010_depth11 = _patch_composite(_composite("p010", 10), depth=11)
    mixed = _composite("nv12", 10)
    mixed.textures["vuv"].fmt = abi.FMT_RG8
    mixed.textures["vuv"].width *= 2
    image_r16_depth8 = scenes.hdr_yuv_image_frame("planar", 8)
    return dict(r16_depth8=r16_depth8, r8_depth10=r8_depth10, nv12_r8_depth10=nv12_r8_depth10, nv16_10bit=nv16,
                p010_depth11=p010_depth11, r16_with_rg8_chroma=mixed, brush_r16_depth8=image_r16_depth8)


def _unsupported_untouched(device_cls, f):
    """draws f: the batch must be reported as WRCU_ERR_UNSUPPORTED and the target must hold only its clear"""
    name = _target(f)
    d = device_cls()
    try:
        handles = draw_frame(d, f)
        with pytest.raises(WrcuError) as err:
            d.finish()
            d.read_pixels(handles[name], 0, 0, 1, 1, 4)
        assert err.value.code == abi.ERR_UNSUPPORTED
        desc = f.textures[name]
        got = d.read_pixels(handles[name], 0, 0, desc.width, desc.height, 4)
    finally:
        d.close()
    from webrender_b200.frame import Frame, Target
    clear_only = Frame(f.tables, f.textures, [[Target(name, ops=f.passes[0][0].ops[:1])]])
    assert (got == render(device_cls, clear_only, [name])[name]).all()


@pytest.mark.parametrize("which", list(_mismatched()))
def test_mismatched_planes_unsupported(which):
    """R16 planes at depth 8, R8 planes at depth 10, NV16, depths other than 10/12/16, R16 luma with RG8 chroma:
    not drawn, reported as WRCU_ERR_UNSUPPORTED."""
    _unsupported_untouched(EmuDevice, _mismatched()[which])


def _blit_status(dev, lib, prefix, fmt, depth):
    ty, tu, tv = (dev.texture_create(fmt, 64, 32), dev.texture_create(fmt, 32, 16), dev.texture_create(fmt, 32, 16))
    td = dev.texture_create(abi.FMT_RGBA8, 64, 32)
    before = dev.read_pixels(td, 0, 0, 64, 32, 4)
    I4 = C.c_int32 * 4
    f = getattr(lib, prefix + "composite_blit_yuv")
    f.argtypes = [C.c_void_p] + [C.c_uint32] * 4 + [C.c_int, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                                 C.c_int, C.c_int, C.POINTER(C.c_int32)]
    rc = f(dev.ctx, td, ty, tu, tv, 2, depth, I4(0, 0, 64, 32), I4(0, 0, 64, 32), 0, 0, I4(0, 0, 64, 32))
    return rc, before, dev.read_pixels(td, 0, 0, 64, 32, 4)


@pytest.mark.parametrize("fmt,depth", [(abi.FMT_R16, 8), (abi.FMT_R8, 10), (abi.FMT_R16, 11), (abi.FMT_RG16, 10)])
def test_blit_yuv_mismatched_unsupported(fmt, depth):
    e = EmuDevice()
    try:
        rc, before, after = _blit_status(e, e.lib, "wremu_", fmt, depth)
    finally:
        e.close()
    assert rc == abi.ERR_UNSUPPORTED and (before == after).all()


# ---- sanity: the expected bytes are a YCbCr -> RGB conversion ------------------------------------------------
# BT.709 narrow range, 1:1: the reference's fixed-point span body (15-bit samples cut to 8 bits, 6-bit
# coefficients, chroma bilinear at half resolution) against a float conversion of the same codes with the same
# chroma interpolation.  Measured: at most 6 (planar 10-bit) and 5 (P010) levels of 255 on any channel, 99% of
# channels within 4 and 3; the mean is 1-2 levels off on B and R, the samples being truncated, not rounded.
SANITY_BOUND = 6


def _float_bt709(frame, fmt, depth):
    """the 1:1 surface of `frame` (instance 0: a 1:1 rect at an even uv offset) converted in float64"""
    inst = frame.passes[0][0].ops[1].instances.view(np.float32)[0]
    r, uvr = inst[0:4], inst[16:20]
    vw, vh = 192, 128
    planes = scenes.hdr_yuv_planes(vw, vh, 1 + 2 + 5, fmt, depth)
    y = planes[0].view(np.uint16).astype(np.float64)
    if fmt == "planar":
        u, v = planes[1].view(np.uint16).astype(np.float64), planes[2].view(np.uint16).astype(np.float64)
    else:
        uv = planes[1].view(np.uint16).reshape(vh // 2, vw // 2, 2).astype(np.float64)
        u, v = uv[..., 0], uv[..., 1]
    scale = float(1 << (16 - depth)) if fmt == "p010" else 1.0
    y, u, v = y / scale, u / scale, v / scale
    w, h = int(r[2] - r[0]), int(r[3] - r[1])
    ys, xs = int(uvr[1]), int(uvr[0])
    Y = y[ys:ys + h, xs:xs + w]
    # chroma sampled at the luma pixel centres: ((x + 0.5) / 2 - 0.5), bilinear, clamped to the plane
    cx = np.clip((np.arange(xs, xs + w) + 0.5) / 2 - 0.5, 0, vw // 2 - 1)
    cy = np.clip((np.arange(ys, ys + h) + 0.5) / 2 - 0.5, 0, vh // 2 - 1)

    def bil(p):
        x0, y0 = np.floor(cx).astype(int), np.floor(cy).astype(int)
        x1, y1 = np.minimum(x0 + 1, p.shape[1] - 1), np.minimum(y0 + 1, p.shape[0] - 1)
        fx, fy = cx - x0, (cy - y0)[:, None]
        top = p[y0][:, x0] * (1 - fx) + p[y0][:, x1] * fx
        bot = p[y1][:, x0] * (1 - fx) + p[y1][:, x1] * fx
        return top * (1 - fy) + bot * fy
    U, V = bil(u), bil(v)
    k = float(1 << (depth - 8))
    yn, un, vn = (Y - 16 * k) / (219 * k), (U - 128 * k) / (224 * k), (V - 128 * k) / (224 * k)
    R = yn + 1.5748 * vn
    G = yn - 0.18732 * un - 0.46812 * vn
    B = yn + 1.8556 * un
    rgb = np.clip(np.rint(np.stack([B, G, R], axis=2) * 255), 0, 255)
    return rgb, (int(r[0]), int(r[1]), w, h), inst[4:8]


@pytest.mark.parametrize("fmt", ["planar", "p010"])
def test_high_bit_depth_output_is_a_colour_conversion(fmt, reference):
    """Guards the fixtures against being trivially wrong: the reference's 1:1 BT.709 narrow-range surface is a
    YCbCr -> RGB conversion of the codes to within SANITY_BOUND levels."""
    f = _composite(fmt, 10)
    f.passes[0][0].ops[1].instances = f.passes[0][0].ops[1].instances[:1]  # the 1:1 surface alone
    got = _reference_pixels(reference, f, ["fb"])["fb"].reshape(320, 512, 4).astype(np.float64)
    want, (x, y, w, h), clip = _float_bt709(f, fmt, 10)
    # the 1:1 surface's clip rect is inset (3, 2) / (5, 1); keep the pixels it draws
    cx0, cy0, cx1, cy1 = int(np.ceil(clip[0])), int(np.ceil(clip[1])), int(clip[2]), int(clip[3])
    sub = got[cy0:cy1, cx0:cx1, :3]
    ref = want[cy0 - y:cy1 - y, cx0 - x:cx1 - x]
    assert sub.size > 3 * 2000
    assert np.abs(sub - ref).max() <= SANITY_BOUND, np.abs(sub - ref).max()


# ---- GPU tier: the kernels against the same expected bytes --------------------------------------------------
def _cuda():
    from webrender_b200.device import CudaDevice
    return CudaDevice


@pytest.mark.gpu
@pytest.mark.parametrize("case", _composite_cases() + _image_cases(), ids=lambda c: c[0])
def test_cuda_high_bit_depth_frames(case, reference):
    """The CPU tier's composite and brush_yuv_image frames through the CUDA kernels: byte-equal."""
    _, make, args = case
    f = make(*args)
    names = [_target(f)]
    want = _reference_pixels(reference, f, names)
    assert_same(render(_cuda(), f, names), want, case[0])


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(fmt="p010"), dict(fmt="p010", vw=3840, vh=2160), dict(fmt="planar", depth=12)],
                         ids=["p010_1080p_to_4k", "p010_4k_1to1", "planar12_1080p_to_4k"])
def test_cuda_high_bit_depth_full_size(kw, reference):
    """4K targets: the per-surface u chain table and strip mode over a 3840-pixel span, scaled and 1:1."""
    f = scenes.hdr_video_frame(**kw)
    want = _reference_pixels(reference, f, ["fb"])
    assert_same(render(_cuda(), f, ["fb"]), want)


@pytest.mark.gpu
@pytest.mark.parametrize("which", list(_mismatched()))
def test_cuda_mismatched_planes_unsupported(which):
    _unsupported_untouched(_cuda(), _mismatched()[which])


@pytest.mark.gpu
@pytest.mark.parametrize("case", _sw_cases(), ids=[c[0] for c in _sw_cases()])
@pytest.mark.parametrize("depth", [10, 12, 16])
def test_gl_shim_composite_yuv_r16(depth, case, reference):
    """CompositeYUV with R16 planes through libwrcu_gl.so (GL_R16 storage, GL_RED + GL_UNSIGNED_SHORT uploads) on the
    CUDA backend: bytes equal."""
    import os
    from webrender_b200.device import LIB_PATH
    planes = sw_yuv_planes16(case, depth)
    want = reference(_emu_composite_yuv16(case, planes, depth), lambda: _swgl_composite_yuv16(case, planes, depth))["dst"]
    d = _swgl_device(os.path.join(os.path.dirname(LIB_PATH), "libwrcu_gl.so"))
    try:
        got = run_sw_composite_yuv16(d, case, planes, depth)
    finally:
        d.close()
    assert_same({"dst": got}, {"dst": want}, case[0])


@pytest.mark.gpu
def test_host_renderer_p010(reference):
    """One P010 frame through the C++ host mirror (wr::Renderer over the C ABI): the same bytes."""
    from webrender_b200.host import HostRenderer
    f = scenes.hdr_video_frame(width=1280, height=720, vw=640, vh=360)
    want = _reference_pixels(reference, f, ["fb"])["fb"]
    dev = _cuda()()
    try:
        hr = HostRenderer(dev)
        nf = hr.build(f)
        hr.render_native(nf)
        dev.finish()
        got = dev.read_pixels(nf.handles["fb"], 0, 0, 1280, 720, 4)
        hr.close()
    finally:
        dev.close()
    assert_same({"fb": got}, {"fb": want})
