"""High-bit-depth video against the 8-bit control, on one GPU, in one process.

Each workload is timed the way bench.py --workload times a frame: the frame is built once, every step is
wr::Renderer::render of the C++ host mirror (or one wrcu_composite_blit_yuv call for the CompositeYUV rows), the
126 MB L2 is flushed between steps, CUDA events around each step, the median of --steps after --warmup.  The
workloads are run round-robin (--rounds times) so that drift on a shared machine falls on all of them alike.
One JSON line per workload: ms, launches, target pixels, the card's name and power limit read in this run, and
SWGL on one core on the same frame when the reference build (oracle/_ref) is there.

    python tools/bench_hdr_video.py [--steps 50] [--warmup 10] [--rounds 3] [--no-cpu-baseline]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H = 3840, 2160


def frame_workloads():
    from workloads import scenes
    return {
        "nv12_1080p_to_4k": lambda: scenes.video_frame(W, H, 1920, 1080, "nv12"),
        "p010_1080p_to_4k": lambda: scenes.hdr_video_frame(W, H, 1920, 1080, "p010", 10),
        "planar10_1080p_to_4k": lambda: scenes.hdr_video_frame(W, H, 1920, 1080, "planar", 10),
        "p010_4k_1to1": lambda: scenes.hdr_video_frame(W, H, W, H, "p010", 10),
    }


BLIT_WORKLOADS = {"composite_yuv_8bit_1080p_to_4k": 8, "composite_yuv_10bit_1080p_to_4k": 10}


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        power = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        power = None
    return {"gpu": name, "power_limit_w": power}


def blit_planes(depth):
    """a seeded 1920x1080 4:2:0 frame: R8 planes at depth 8, LSB-aligned R16 planes otherwise"""
    rng = np.random.RandomState(depth)
    top, dt = (256, np.uint8) if depth == 8 else (1 << depth, np.uint16)
    return [rng.randint(0, top, s).astype(dt) for s in ((1080, 1920), (540, 960), (540, 960))]


class Blit:
    """CompositeYUV of a 1080p frame into a 4K destination (wrcu_composite_blit_yuv, SwCompositor's hook)"""

    def __init__(self, dev, depth):
        from webrender_b200 import abi
        self.dev, self.depth = dev, depth
        fmt = abi.FMT_R8 if depth == 8 else abi.FMT_R16
        self.planes = blit_planes(depth)
        self.tex = []
        for p in self.planes:
            t = dev.texture_create(fmt, p.shape[1], p.shape[0])
            dev.texture_upload(t, 0, 0, p.shape[1], p.shape[0], p)
            self.tex.append(t)
        self.dst = dev.texture_create(abi.FMT_RGBA8, W, H)
        I4 = C.c_int32 * 4
        self.rects = (I4(0, 0, 1920, 1080), I4(0, 0, W, H), I4(0, 0, W, H))
        self.f = dev.lib.wrcu_composite_blit_yuv
        self.f.argtypes = [C.c_void_p] + [C.c_uint32] * 4 + [C.c_int, C.c_uint32, C.POINTER(C.c_int32),
                                                             C.POINTER(C.c_int32), C.c_int, C.c_int, C.POINTER(C.c_int32)]

    def step(self):
        sr, dr, cr = self.rects
        self.dev._check(self.f(self.dev.ctx, self.dst, *self.tex, 2, self.depth, sr, dr, 0, 0, cr))


def swgl_baseline(name, frame, depth):
    """SWGL (the unmodified reference, one core) on the same work: best of up to 5 runs within ~15 s"""
    from oracle.backends import SwglDevice, have_swgl
    from webrender_b200 import abi
    from webrender_b200.frame import draw_frame
    if not have_swgl():
        return None
    # R16 / RG16 storage and GL_RED / GL_RG + GL_UNSIGNED_SHORT transfers (gl.cc:257-285, 1755-1757)
    SwglDevice._IFMT.setdefault(abi.FMT_R16, 0x822A)
    SwglDevice._IFMT.setdefault(abi.FMT_RG16, 0x822C)
    SwglDevice._XFER.setdefault(abi.FMT_R16, (0x1903, 0x1403))
    SwglDevice._XFER.setdefault(abi.FMT_RG16, (0x8227, 0x1403))
    d = SwglDevice()
    try:
        if frame is not None:
            h = draw_frame(d, frame)
            run = lambda: draw_frame(d, frame, h)  # noqa: E731
        else:
            fmt = abi.FMT_R8 if depth == 8 else abi.FMT_R16
            planes = blit_planes(depth)
            tex = []
            for p in planes:
                t = d.texture_create(fmt, p.shape[1], p.shape[0])
                d.texture_upload(t, 0, 0, p.shape[1], p.shape[0], p)
                tex.append(t)
            dst = d.texture_create(abi.FMT_RGBA8, W, H)
            run = lambda: d.sw_composite_yuv(dst, *tex, 2, (0, 0, 1920, 1080), (0, 0, W, H), False, False,  # noqa: E731
                                             (0, 0, W, H), color_depth=depth)
            run()
        best, reps, t_end = None, 0, time.perf_counter() + 15.0
        while reps < 1 or (time.perf_counter() < t_end and reps < 5):
            t0 = time.perf_counter()
            run()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
            reps += 1
    finally:
        d.close()
    return {"ms": best * 1e3, "cores": 1, "kind": "reference", "sample": f"the same work, best of {reps}"}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_hdr_video.py: no CUDA device; the wrcu backend has no CPU path")
    from bench import l2_flush, _frame_pixels
    from webrender_b200.device import CudaDevice
    from webrender_b200.host import HostRenderer
    info = gpu_info()
    dev = CudaDevice(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    hr = HostRenderer(dev)
    runs, frames = {}, {}
    for name, make in frame_workloads().items():
        frames[name] = make()
        nf = hr.build(frames[name])
        runs[name] = (lambda nf=nf: hr.render_native(nf))
    for name, depth in BLIT_WORKLOADS.items():
        runs[name] = Blit(dev, depth).step
    ms = {n: [] for n in runs}
    launches = {n: 0 for n in runs}
    for name, run in runs.items():
        for _ in range(max(args.warmup, 3)):
            run()
    dev.finish()
    for _ in range(args.rounds):
        for name, run in runs.items():
            dev.finish()
            dev.reset_stats()
            for _ in range(args.steps):
                l2_flush(flush)
                dev.timer_begin()
                run()
                ms[name].append(dev.timer_end())
            launches[name] = dev.stats()["kernel_launches"] // args.steps
    control = {}
    for name in runs:
        t = sorted(ms[name])
        med = t[len(t) // 2]
        control[name] = med
        is_blit = name in BLIT_WORKLOADS
        line = {"workload": name, "ms": med, "ms_min": t[0], "ms_max": t[-1], "samples": len(t),
                "launches": int(launches[name]),
                "target_pixels": W * H if is_blit else _frame_pixels(frames[name]),
                **info, "l2": "flushed between steps", "host": "wrcu_composite_blit_yuv" if is_blit else
                "wr::Renderer::render (C++ host mirror)"}
        ctl = "composite_yuv_8bit_1080p_to_4k" if is_blit else "nv12_1080p_to_4k"
        if name != ctl and ctl in control:
            line["vs_8bit_control"] = med / control[ctl]
        if not args.no_cpu_baseline:
            base = swgl_baseline(name, None if is_blit else frames[name], BLIT_WORKLOADS.get(name, 8))
            if base is not None:
                line["cpu_baseline"] = base
        print(json.dumps(line), flush=True)
    hr.close()
    dev.close()


if __name__ == "__main__":
    main()
