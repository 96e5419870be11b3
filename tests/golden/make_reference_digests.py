"""Regenerates tests/golden/reference_digests.json: for every check of the `reference` fixture
(tests/common.py), the digest of what the UNMODIFIED reference rasteriser (oracle/_ref/libswgl_ref.so,
built by oracle/Makefile from a WebRender checkout) draws.  The tests then compare against the stored
digests and need no reference build.

Needs oracle/_ref:  python tests/golden/make_reference_digests.py
Recording runs the tests below with the reference build beside the checker they pin and fails where
the two differ; the GPU tests among them stop once their reference is recorded.
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

CPU_MODULES = ["test_oracle_vs_swgl.py", "test_emu_parity.py", "test_update_path.py"]
GPU_TESTS = ["test_cuda_parity.py::test_perspective_brushes", "test_cuda_parity.py::test_perspective_picture_brushes",
             "test_cuda_parity.py::test_perspective_full_size", "test_cuda_parity.py::test_split_composite",
             "test_gl_shim.py::test_sw_compositor_composite_yuv", "test_gl_shim.py::test_sw_compositor_composite"]


def main():
    from common import RECORD_ENV, REFERENCE_DIGESTS
    from oracle.backends import have_swgl
    if not have_swgl():
        raise SystemExit("oracle/_ref/libswgl_ref.so is not built (oracle/Makefile, target ref)")
    with tempfile.TemporaryDirectory() as tmp:
        rec = os.path.join(tmp, "digests.jsonl")
        env = dict(os.environ, **{RECORD_ENV: rec})
        pytest = [sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider"] + sys.argv[1:]
        tests = os.path.join(ROOT, "tests")
        subprocess.run(pytest + ["-m", "not gpu"] + [os.path.join(tests, m) for m in CPU_MODULES],
                       check=True, cwd=ROOT, env=env)
        subprocess.run(pytest + [os.path.join(tests, t) for t in GPU_TESTS], check=True, cwd=ROOT, env=env)
        out = {}
        for line in open(rec):
            out.update(json.loads(line))
    json.dump(out, open(REFERENCE_DIGESTS, "w"), indent=0, sort_keys=True)
    print(len(out), "digests")


if __name__ == "__main__":
    main()
