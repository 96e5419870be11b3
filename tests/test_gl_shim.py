"""The reference's own FFI surface over the CUDA backend: webrender_b200/libwrcu_gl.so exports the
`extern "C"` symbol set WebRender binds for its software rasteriser (swgl/src/swgl_fns.rs:23-320,
defined in swgl/src/gl.cc and composite.h).  CPU tier: every symbol is exported.  GPU tier: the GL call
sequence `Device` issues (the same driver that runs the UNMODIFIED reference rasteriser in
oracle/backends.py::SwglDevice) is replayed against the shim and must reproduce the oracle's pixels."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle.backends import OracleDevice, SwglDevice
from webrender_b200 import abi
from workloads import scenes

from common import assert_same, reference, render  # noqa: F401 (reference: fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GL_LIB = os.path.join(ROOT, "webrender_b200", "libwrcu_gl.so")

# the names in swgl_fns.rs's extern block (99)
SWGL_SYMBOLS = [
    "ActiveTexture", "AttachShader", "BeginQuery", "BindAttribLocation", "BindBuffer", "BindFramebuffer",
    "BindRenderbuffer", "BindTexture", "BindVertexArray", "BlendColor", "BlendEquation", "BlendFunc",
    "BlitFramebuffer", "BufferData", "BufferSubData", "CheckFramebufferStatus", "Clear", "ClearColor",
    "ClearColorRect", "ClearDepth", "ClearTexImage", "ClearTexSubImage", "Composite", "CompositeYUV",
    "CopyImageSubData", "CopyTexSubImage2D", "CreateContext", "CreateProgram", "CreateShader", "DeleteBuffer",
    "DeleteFramebuffer", "DeleteProgram", "DeleteQuery", "DeleteRenderbuffer", "DeleteShader",
    "DeleteTexture", "DeleteVertexArray", "DepthFunc", "DepthMask", "DestroyContext", "Disable",
    "DrawElementsInstanced", "Enable", "EnableVertexAttribArray", "EndQuery", "Finish",
    "FramebufferRenderbuffer", "FramebufferTexture2D", "GenBuffers", "GenFramebuffers", "GenQueries",
    "GenRenderbuffers", "GenTextures", "GenVertexArrays", "GenerateMipmap", "GetAttribLocation",
    "GetBooleanv", "GetColorBuffer", "GetError", "GetIntegerv", "GetLinkStatus", "GetQueryObjectui64v",
    "GetResourceBuffer", "GetString", "GetStringi", "GetUniformLocation", "InitDefaultFramebuffer",
    "InvalidateFramebuffer", "LinkProgram", "LockFramebuffer", "LockResource", "LockTexture", "MakeCurrent",
    "MapBuffer", "MapBufferRange", "PixelStorei", "ReadPixels", "ReferenceContext", "RenderbufferStorage",
    "ReportMemory", "ResolveFramebuffer", "SetScissor", "SetTextureBuffer", "SetTextureParameter",
    "SetViewport", "ShaderSourceByName", "TexImage2D", "TexParameteri", "TexStorage2D", "TexSubImage2D",
    "Uniform1i", "Uniform4fv", "UniformMatrix4fv", "UnlockResource", "UnmapBuffer", "UseProgram",
    "VertexAttribDivisor", "VertexAttribIPointer", "VertexAttribPointer"
]


def test_gl_library_exports_the_reference_symbol_set():
    assert len(SWGL_SYMBOLS) == 99
    lib = C.CDLL(GL_LIB)
    for s in SWGL_SYMBOLS:
        assert hasattr(lib, s), s


class GlShimDevice(SwglDevice):
    def __init__(self):
        super().__init__(lib_path=GL_LIB)


CASES = [
    ("alpha_rects", lambda: scenes.alpha_rects_frame(640, 360, 60, random_rects=True, seed=4, color=None), None),
    ("alpha_rects_softlight", lambda: scenes.alpha_rects_frame(320, 200, 30, random_rects=True, seed=7, color=None,
                                                                 blend=abi.BLEND_ADV_SOFT_LIGHT), None),
    ("brush_solid_masks_depth", lambda: scenes.brush_solid_frame(seed=1), ["target"]),
    ("clip_masks", lambda: scenes.clip_mask_frame(seed=2, fractional=True), None),
    ("rounded_rects_indirect", lambda: scenes.rounded_rects_frame(seed=1), None),
    ("images", lambda: scenes.image_frame(seed=1, one_to_one=True), ["target"]),
    ("text_subpixel", lambda: scenes.text_frame(seed=2, width=480, height=270, n_runs=8, glyphs_per_run=20,
                                                atlas="rgba", color_modes=(0, 1, 2, 3)), ["target"]),
    ("gradients", lambda: scenes.gradient_frame(seed=1, blend=abi.BLEND_PREMULTIPLIED_ALPHA), None),
    ("box_shadows", lambda: scenes.box_shadow_frame(seed=1), None),
    ("composite", lambda: scenes.composite_frame(seed=1), ["fb"]),
    ("composite_yuv_nv12", lambda: scenes.yuv_composite_frame("nv12", 3, seed=2), ["fb"]),
    ("brush_yuv_image", lambda: scenes.yuv_image_frame("planar", 1, seed=2, fractional=True), ["target"]),
    ("composite_yuv_planar", lambda: scenes.yuv_composite_frame("planar", 4, seed=3, fractional=True), ["fb"]),
    ("blur", lambda: scenes.blur_frame(seed=1), ["mid", "target"]),
    ("texture_cache_target", lambda: scenes.texture_cache_frame(seed=1), None),
    ("quad_radial", lambda: scenes.quad_gradient_frame(abi.KIND_QUAD_RADIAL_GRADIENT, seed=2), None),
    ("config_a", lambda: scenes.config_a_frame(), None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,make,targets", CASES, ids=[c[0] for c in CASES])
def test_gl_call_sequence_on_the_cuda_backend(name, make, targets):
    frame = make()
    assert_same(render(GlShimDevice, frame, targets), render(OracleDevice, frame, targets), name)


@pytest.mark.gpu
def test_gl_strings_keep_the_host_on_the_software_path():
    lib = C.CDLL(GL_LIB)
    lib.CreateContext.restype = C.c_void_p
    lib.MakeCurrent.argtypes = [C.c_void_p]
    lib.DestroyContext.argtypes = [C.c_void_p]
    lib.GetString.restype = C.c_char_p
    ctx = lib.CreateContext()
    assert ctx
    lib.MakeCurrent(ctx)
    assert lib.GetString(0x1F01) == b"Software WebRender"   # GL_RENDERER → Device::is_software (device/gl.rs:1645)
    v = C.c_int(0)
    lib.GetIntegerv(0x0D33, C.byref(v))
    assert v.value == 1 << 15                               # GL_MAX_TEXTURE_SIZE, as gl.cc:1158
    assert lib.GetError() == 0
    lib.DestroyContext(ctx)


SW_COMPOSITE_CASES = [
    # (src size, src rect, dst rect, opaque, flip_x, flip_y, linear, clip rect)
    ("copy_1to1", (256, 128), (0, 0, 256, 128), (40, 30, 256, 128), True, False, False, False, (0, 0, 640, 360)),
    ("over_1to1_clipped", (256, 128), (0, 0, 256, 128), (100, 60, 256, 128), False, False, False, False, (130, 70, 180, 90)),
    ("nearest_upscale", (200, 100), (10, 5, 150, 80), (20, 10, 450, 240), True, False, False, False, (0, 0, 640, 360)),
    ("nearest_downscale_over_flipy", (300, 200), (0, 0, 300, 200), (33, 21, 100, 77), False, False, True, False, (0, 0, 640, 360)),
    ("nearest_partly_outside", (200, 100), (-20, -10, 260, 140), (50, 40, 390, 210), True, False, False, False, (60, 50, 300, 150)),
    ("linear_upscale", (120, 90), (0, 0, 120, 90), (15, 25, 481, 301), True, False, False, True, (0, 0, 640, 360)),
    ("linear_downscale_over", (400, 300), (7, 9, 380, 280), (101, 33, 211, 157), False, False, False, True, (90, 40, 300, 200)),
    ("linear_flipx_same_size", (256, 128), (0, 0, 256, 128), (64, 64, 256, 128), True, True, False, False, (0, 0, 640, 360)),
    ("linear_flipxy_over", (160, 120), (5, 5, 150, 110), (200, 100, 333, 222), False, True, True, True, (0, 0, 640, 360)),
]


SW_COMPOSITE_YUV_CASES = [
    # (name, luma size, chroma size, colour space, src rect, dst rect, flip_x, flip_y, clip rect)
    ("420_upscale_bt709", (320, 180), (160, 90), 2, (0, 0, 320, 180), (10, 6, 600, 338), False, False, (0, 0, 640, 360)),
    ("420_1to1_bt601", (320, 180), (160, 90), 0, (0, 0, 320, 180), (100, 50, 320, 180), False, False, (0, 0, 640, 360)),
    ("420_upscale_clipped_full_range", (322, 182), (161, 91), 3, (3, 5, 300, 170), (21, 11, 577, 333), False, False, (60, 40, 400, 200)),
    ("420_partly_outside", (200, 120), (100, 60), 4, (-12, -8, 230, 140), (30, 20, 500, 300), False, False, (0, 0, 640, 360)),
    ("420_downscale", (640, 360), (320, 180), 1, (0, 0, 640, 360), (40, 30, 233, 131), False, False, (0, 0, 640, 360)),
    ("420_flip_xy", (320, 180), (160, 90), 5, (0, 0, 320, 180), (50, 20, 480, 270), True, True, (0, 0, 640, 360)),
    ("444_upscale", (160, 90), (160, 90), 2, (0, 0, 160, 90), (0, 0, 640, 360), False, False, (0, 0, 640, 360)),
    ("444_gbr_identity", (200, 100), (200, 100), 6, (10, 10, 180, 80), (33, 44, 359, 161), False, True, (50, 50, 300, 140)),
    ("422_wide_chroma", (320, 180), (160, 180), 2, (0, 0, 320, 180), (5, 5, 630, 350), False, False, (0, 0, 640, 360)),
    ("420_big_zoom", (64, 48), (32, 24), 0, (8, 8, 40, 30), (0, 0, 640, 360), False, False, (0, 0, 640, 360)),
    ("420_three_pixels_wide", (320, 180), (160, 90), 2, (0, 0, 320, 180), (100, 100, 3, 50), False, False, (0, 0, 640, 360)),
    ("420_odd_planes_flipx", (321, 181), (161, 91), 2, (1, 1, 319, 179), (7, 3, 611, 347), True, False, (0, 0, 640, 360)),
    ("420_dst_partly_off_target", (320, 180), (160, 90), 4, (0, 0, 320, 180), (-50, -40, 800, 450), False, False, (-50, -40, 800, 450)),
]


def sw_yuv_planes(case):
    _, (yw, yh), (cw, ch), _, _, _, _, _, _ = case
    rng = np.random.RandomState(7)
    return (rng.randint(0, 256, (yh, yw)).astype(np.uint8), rng.randint(0, 256, (ch, cw)).astype(np.uint8),
            rng.randint(0, 256, (ch, cw)).astype(np.uint8), rng.randint(0, 256, (360, 640 * 4)).astype(np.uint8))


def run_sw_composite_yuv(dev, case, planes, via=None):
    """Uploads the planes, runs CompositeYUV (through `via(dev, handles...)` when given), returns the destination."""
    _, (yw, yh), (cw, ch), cs, sr, dr, fx, fy, cr = case
    yp, up, vp, dst = planes
    ty, tu, tv = (dev.texture_create(abi.FMT_R8, yw, yh), dev.texture_create(abi.FMT_R8, cw, ch),
                  dev.texture_create(abi.FMT_R8, cw, ch))
    td = dev.texture_create(abi.FMT_RGBA8, 640, 360)
    dev.texture_upload(ty, 0, 0, yw, yh, yp)
    dev.texture_upload(tu, 0, 0, cw, ch, up)
    dev.texture_upload(tv, 0, 0, cw, ch, vp)
    dev.texture_upload(td, 0, 0, 640, 360, dst)
    if via is None:
        dev.sw_composite_yuv(td, ty, tu, tv, cs, sr, dr, fx, fy, cr)
        return dev.locked_pixels(td)
    via(dev, td, ty, tu, tv, cs, sr, dr, fx, fy, cr)
    return dev.read_pixels(td, 0, 0, 640, 360, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("case", SW_COMPOSITE_YUV_CASES, ids=[c[0] for c in SW_COMPOSITE_YUV_CASES])
def test_sw_compositor_composite_yuv(case, reference):
    """CompositeYUV (swgl/src/composite.h:1335-1384: linear_convert_yuv / linear_row_yuv / upscaleYUV42R8) through
    libwrcu_gl.so on the CUDA backend against the unmodified reference: 4:2:0, 4:2:2 and 4:4:4 planes, up- and
    downscaling, flips, clips, sources partly outside the planes, every colour space — bytes equal.  The expected
    bytes are the host emulation's, held to the digest of the reference build's output."""
    from test_emu_parity import _emu_composite_yuv, _swgl_composite_yuv
    planes = sw_yuv_planes(case)
    want = reference(_emu_composite_yuv(case, planes), lambda: _swgl_composite_yuv(case, planes))["dst"]
    d = GlShimDevice()
    got = run_sw_composite_yuv(d, case, planes)
    d.close()
    diff = got != want
    assert not diff.any(), f"{int(diff.sum())} bytes differ, first at {np.argwhere(diff)[0]}"
    assert (got != planes[3]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("case", SW_COMPOSITE_CASES, ids=[c[0] for c in SW_COMPOSITE_CASES])
def test_sw_compositor_composite(case, reference):
    """SwCompositor's hooks (LockTexture / Composite / GetResourceBuffer / UnlockResource,
    swgl/src/composite.h:485-590) on the CUDA backend against the unmodified reference: integer-ratio
    nearest blits, 7-bit bilinear blits with their per-chunk running sums, flips, clips, over — bytes equal.
    The expected bytes are the host emulation's, held to the digest of the reference build's output."""
    from test_emu_parity import _emu_blit, _swgl_blit
    _, (sw, sh), sr, dr, opaque, fx, fy, lin, cr = case
    rng = np.random.RandomState(11)
    src = rng.randint(0, 256, (sh, sw, 4)).astype(np.uint8)
    a = src[..., 3:4].astype(np.uint16)
    src[..., :3] = (src[..., :3].astype(np.uint16) * a // 255).astype(np.uint8)
    dst = rng.randint(0, 256, (360, 640, 4)).astype(np.uint8)
    call = (src, dst, sr, dr, opaque, fx, fy, lin, cr)
    want = reference(_emu_blit(*call), lambda: _swgl_blit(*call))["dst"]
    d = GlShimDevice()
    ts = d.texture_create(abi.FMT_RGBA8, sw, sh)
    td = d.texture_create(abi.FMT_RGBA8, 640, 360)
    d.texture_upload(ts, 0, 0, sw, sh, src.reshape(sh, sw * 4))
    d.texture_upload(td, 0, 0, 640, 360, dst.reshape(360, 640 * 4))
    d.sw_composite(td, ts, sr, dr, opaque, fx, fy, lin, cr)
    got = d.locked_pixels(td)
    d.close()
    diff = got != want
    assert not diff.any(), f"{int(diff.sum())} bytes differ, first at {np.argwhere(diff)[0]}"
    assert (got != dst.reshape(360, 640 * 4)).any()
