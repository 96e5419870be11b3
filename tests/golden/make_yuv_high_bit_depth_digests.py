"""Regenerates tests/golden/yuv_high_bit_depth_digests.json: for every check of the `reference` fixture of
tests/test_yuv_high_bit_depth.py, the digest of what the UNMODIFIED reference rasteriser (oracle/_ref/libswgl_ref.so,
built by oracle/Makefile from a WebRender checkout) draws.

Needs oracle/_ref:  python tests/golden/make_yuv_high_bit_depth_digests.py
The CPU tests fail where the host emulation differs from the reference build; the GPU tests stop once their
reference is recorded, so no GPU is needed.
"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MODULE = os.path.join(ROOT, "tests", "test_yuv_high_bit_depth.py")
# the GPU tests that draw through the `reference` fixture
GPU_TESTS = ["test_cuda_high_bit_depth_frames", "test_cuda_high_bit_depth_full_size", "test_gl_shim_composite_yuv_r16",
             "test_host_renderer_p010"]


def main():
    from common import RECORD_ENV
    from oracle.backends import have_swgl
    if not have_swgl():
        raise SystemExit("oracle/_ref/libswgl_ref.so is not built (oracle/Makefile, target ref)")
    with tempfile.TemporaryDirectory() as tmp:
        rec = os.path.join(tmp, "digests.jsonl")
        env = dict(os.environ, **{RECORD_ENV: rec})
        pytest = [sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider"] + sys.argv[1:]
        subprocess.run(pytest + ["-m", "not gpu", MODULE], check=True, cwd=ROOT, env=env)
        subprocess.run(pytest + ["-m", "gpu", "-k", " or ".join(GPU_TESTS), MODULE], check=True, cwd=ROOT, env=env)
        out = {}
        for line in open(rec):
            out.update(json.loads(line))
    json.dump(out, open(os.path.join(HERE, "yuv_high_bit_depth_digests.json"), "w"), indent=0, sort_keys=True)
    print(len(out), "digests")


if __name__ == "__main__":
    main()
