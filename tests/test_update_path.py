"""Update path (SURVEY.md §8f rank 3): batched texture-cache uploads, texture
copies and GPU-cache update lists — the reference's plumbing replayed against
SWGL, the oracle, the host emulation and (GPU tier) the CUDA backend."""
import numpy as np
import pytest

from oracle.backends import OracleDevice, SwglDevice

from common import reference  # noqa: F401 (fixture)

from update_path import run_sequence


def _run(cls, kind, seed):
    dev = cls()
    try:
        return run_sequence(dev, kind, seed)
    finally:
        dev.close()


@pytest.mark.parametrize("kind", ["text", "image"])
@pytest.mark.parametrize("seed", [1, 2])
def test_oracle_matches_reference_plumbing(kind, seed, reference):
    def frames(cls):
        return {f"frame{i}": x for i, x in enumerate(_run(cls, kind, seed))}
    b = reference(frames(OracleDevice), lambda: frames(SwglDevice))
    assert not np.array_equal(b["frame0"], b["frame1"])   # frame 2 really differs (patched cache / moved tile)


@pytest.mark.parametrize("kind", ["text", "image"])
def test_emu_matches_oracle(kind):
    from emu import EmuDevice
    a = _run(EmuDevice, kind, 1)
    b = _run(OracleDevice, kind, 1)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["text", "image"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_cuda_matches_oracle(kind, seed):
    from webrender_b200.device import CudaDevice
    a = _run(CudaDevice, kind, seed)
    b = _run(OracleDevice, kind, seed)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_cuda_upload_batch_bad_rect_is_rejected():
    from webrender_b200.device import CudaDevice, WrcuError
    from webrender_b200 import abi
    dev = CudaDevice(0)
    try:
        t = dev.texture_create(abi.FMT_RGBA8, 64, 64)
        with pytest.raises(WrcuError):
            dev.texture_upload_batch(t, [(32, 32, 64, 8, 0, 256)], np.zeros(4096, np.uint8))
        with pytest.raises(WrcuError):
            dev.texture_upload_batch(t, [(0, 0, 16, 16, 0, 64)], np.zeros(512, np.uint8))   # blob too small
    finally:
        dev.close()
