"""Stores the reference's own reftest images that tests/test_golden.py compares with, from a WebRender
checkout:  python tests/golden/make_reftest_images.py <webrender checkout>

* reftest_images.npz.xz: wrench/reftests/<path> as RGB arrays (every one is opaque), keyed by <path>;
  of image/yuv.png only the rows YUV_ROWS.
* reftest_yuv/: the plane PNGs image/yuv.yaml reads, cut to their first YUV_ROWS.stop - YUV_ROWS.start rows
  and zero below.  The planes are drawn 1:1 from y = YUV_ROWS.start, so those rows of the page depend on
  these plane rows alone.
"""
import io
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
IMAGES = os.path.join(HERE, "reftest_images.npz.xz")
YUV_PLANES = os.path.join(HERE, "reftest_yuv")
YUV_ROWS = slice(10, 58)
PNGS = ["aa/rounded-rects-ref.png", "border/border-clamp-corner-radius.png", "border/border-no-bogus-line-ref.png",
        "border/border-radii.png", "border/overlapping.png", "boxshadow/box-shadow-spread.png",
        "boxshadow/box-shadow-suite-no-blur.png", "boxshadow/boxshadow-spread-only-ref.png",
        "boxshadow/inset-no-blur-radius-ref.png", "clip/clip-ellipse.png", "clip/clip-mode.png",
        "clip/inverted-ellipse.png", "filters/filter-small-blur-radius.png", "gradient/conic-center.png",
        "gradient/conic-simple.png", "gradient/linear-aligned-border-radius.png", "gradient/linear-hard-stop-ref.png",
        "gradient/linear-ref.png", "gradient/linear-stops-ref.png", "gradient/premultiplied-aligned.png",
        "gradient/premultiplied-angle.png", "gradient/premultiplied-conic.png", "gradient/premultiplied-radial.png",
        "gradient/radial-circle-ref.png", "gradient/radial-ellipse-ref.png", "image/segments.png",
        "split/near-plane.png", "text/decorations-suite.png", "image/yuv.png"]
YUV_PLANE_PNGS = ["spacex-y.png", "spacex-u.png", "spacex-v.png", "spacex-uv.png", "spacex-yuv.png"]


def main(checkout):
    from PIL import Image
    reftests = os.path.join(checkout, "wrench", "reftests")
    out = {}
    for p in PNGS:
        a = np.array(Image.open(os.path.join(reftests, p)).convert("RGBA"))
        assert (a[..., 3] == 255).all(), p
        out[p] = a[YUV_ROWS, :, :3] if p == "image/yuv.png" else a[..., :3]
    buf = io.BytesIO()
    np.savez(buf, **out)
    open(IMAGES, "wb").write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
    os.makedirs(YUV_PLANES, exist_ok=True)
    n = YUV_ROWS.stop - YUV_ROWS.start
    for p in YUV_PLANE_PNGS:
        im = Image.open(os.path.join(reftests, "image", p))
        a = np.array(im)
        a[n:] = 0
        Image.fromarray(a, im.mode).save(os.path.join(YUV_PLANES, p), optimize=True)


if __name__ == "__main__":
    main(sys.argv[1])
