"""Helpers shared by the parity tests."""
import hashlib
import json
import os

import numpy as np
import pytest

from webrender_b200 import abi, draw_frame

REFERENCE_DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
# tests/golden/make_reference_digests.py sets this to a file: the reference build is then run and recorded
RECORD_ENV = "WRCU_RECORD_REFERENCE"
_digests = {}


def digest(arrays):
    """One digest over {name: uint8 array}: names, shapes and bytes."""
    h = hashlib.blake2b(digest_size=16)
    for n in sorted(arrays):
        a = np.ascontiguousarray(arrays[n])
        h.update(f"{n}:{a.shape}:".encode())
        h.update(a.tobytes())
    return h.hexdigest()


@pytest.fixture
def reference(request):
    """check(got, live, part=None) -> got.  `got` ({name: uint8 array}, drawn by a checker or by this
    repository's kernels) must be byte for byte what the unmodified reference rasteriser (oracle/_ref) drew
    for the same input: its digest is stored in golden/reference_digests.json.  `live()` draws the same
    with the reference build; it runs only when recording (RECORD_ENV names the file to append to), and
    then `got` must equal its result and a GPU test ends there."""
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
            _digests.update(json.load(open(REFERENCE_DIGESTS)))
        assert key in _digests, f"{key}: no stored reference digest (tests/golden/make_reference_digests.py)"
        assert digest(got) == _digests[key], f"{key}: differs from the reference rasteriser's output"
        return got
    return check


def render(device_cls, frame, targets=None, tile_lists=False):
    """Run `frame` through a device; return {name: uint8 array} of target contents."""
    d = device_cls()
    try:
        handles = draw_frame(d, frame, tile_lists=tile_lists)
        out = {}
        names = targets or sorted({t.texture for p in frame.passes for t in p})
        for n in names:
            desc = frame.textures[n]
            out[n] = d.read_pixels(handles[n], 0, 0, desc.width, desc.height, abi.FMT_BPP[desc.fmt])
        return out
    finally:
        d.close()


def assert_same(a, b, what=""):
    for k in a:
        diff = a[k] != b[k]
        if diff.any():
            ys, xs = np.nonzero(diff)
            raise AssertionError(f"{what} target {k}: {int(diff.sum())} bytes differ; first at "
                                 f"(byte x={xs[0]}, y={ys[0]}): {a[k][ys[0], xs[0]]} vs {b[k][ys[0], xs[0]]}")
