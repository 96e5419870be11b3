#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its config B: Mpix/s composited at
3840x2160 (examples/alpha_perf.rs scene: 1000 overlapping alpha rects, one
batch), through the wrcu C ABI on N B200s (one process per GPU).

A "step" = one frame: clear + the alpha-blend batch.  `value` times the draw
path with inputs resident on the device; `e2e` times the public call sequence
with HOST buffers in and the framebuffer read back to the host every step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, N_RECTS = 3840, 2160, 1000
BYTES_PER_PIXEL_LAYER = 8  # SURVEY.md §8d: blended pass = 4 B dst read + 4 B dst write


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons)}


WORKLOAD_B = ("config B: examples/alpha_perf.rs scene, 1000 full-frame alpha=0.05 rects in one Quad(ColorOrTexture) "
              "batch at 3840x2160, premultiplied-alpha blend, clear each frame")


def usable_cores():
    """Host cores this process may actually run on: the affinity mask, further limited by the cgroup CPU
    quota (os.cpu_count() reports the machine's cores, which over-subscribed the reference arm in round 1)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:  # cgroup v2, then v1
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = min(n, max(1, int(float(q[0]) / float(q[1]))))
    except (OSError, ValueError, IndexError):
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0 and period > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return max(1, n)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on
    this box's host cores: the unmodified SWGL rasteriser (oracle/_ref) when it
    was built, else the C oracle port.  SWGL is single-threaded by design
    (swgl/README.md:6); all cores are used by running one process per core on
    disjoint horizontal bands of the frame (tiles are independent)."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.backends import have_swgl
    kind = "reference" if have_swgl() else "port"
    cores = min(usable_cores(), args.ref_cores) if args.ref_cores > 0 else usable_cores()
    n_rects = args.ref_rects
    band_h = max(8, H // cores)
    times = []
    ctxm = mp.get_context("spawn")
    # one persistent worker (= one SWGL context) per core; contexts, programs and
    # frames are created once, outside the timed region
    with ctxm.Pool(cores, initializer=_ref_init, initargs=(kind, W, band_h, n_rects)) as pool:
        pool.map(_ref_band, range(cores))  # untimed: first touch of every worker
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            layers = pool.map(_ref_band, range(cores), chunksize=1)
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append((dt, sum(layers)))
    tot_t = sum(t for t, _ in times)
    tot_px = sum(p for _, p in times)
    value = tot_px / tot_t / 1e6
    line = {
        "impl": "reference", "metric": "Mpix/s composited at 3840x2160 (alpha-blend brush pass)",
        "value": value, "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot_t / len(times) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD_B,
                   "sample": f"bounded per step: {n_rects} of the 1000 layers, the 3840x2160 frame cut into {cores} "
                             f"bands of {band_h} rows, one per core ({cores * band_h} of {H} rows); every layer is "
                             f"the same full-band rect, so Mpix/s is a rate on homogeneous work and compares "
                             f"directly with the wrcu arm's 1000-layer frame",
                   "cores": cores, "os_cpu_count": os.cpu_count()},
        "cpu_baseline": {"value": value, "unit": "Mpix/s", "cores": cores, "kind": kind,
                         "sample": f"{n_rects} full-band alpha rects on {cores} bands of {W}x{band_h} px per step "
                                   f"(one persistent SWGL context per core)"},
        "e2e": {"value": value, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


_REF = {}


def _ref_init(kind, w, h, n):
    sys.path.insert(0, ROOT)
    from oracle.backends import OracleDevice, SwglDevice
    from webrender_b200 import draw_frame
    from workloads import scenes
    _REF["frame"] = scenes.alpha_rects_frame(w, h, n)
    _REF["dev"] = (SwglDevice if kind == "reference" else OracleDevice)()
    _REF["handles"] = draw_frame(_REF["dev"], _REF["frame"])
    _REF["layers"] = w * h * n


def _ref_band(_):
    from webrender_b200 import draw_frame
    draw_frame(_REF["dev"], _REF["frame"], _REF["handles"])
    return _REF["layers"]


def cpu_baseline_sample():
    """1-core SWGL (or port) on a bounded sample of config B: timed beside the
    GPU number; reported, not a target."""
    from oracle.backends import OracleDevice, SwglDevice, have_swgl
    from webrender_b200 import draw_frame
    from workloads import scenes
    kind = "reference" if have_swgl() else "port"
    w, h, n = W, 270, 200  # 1/8 of the frame height, 200 layers
    f = scenes.alpha_rects_frame(w, h, n)
    d = (SwglDevice if kind == "reference" else OracleDevice)()
    handles = draw_frame(d, f)  # warm-up (allocations, program link)
    best = None
    t_end = time.perf_counter() + 12.0
    reps = 0
    while reps < 3 or (time.perf_counter() < t_end and reps < 10):
        t0 = time.perf_counter()
        draw_frame(d, f, handles)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
        reps += 1
    d.close()
    return {"value": w * h * n / best / 1e6, "unit": "Mpix/s", "cores": 1, "kind": kind,
            "sample": f"{n} full-frame alpha rects at {w}x{h} (1/8 of config B's rows), best of {reps}, "
                      f"includes table upload + clear; SWGL built with g++ -O2 (generic, non-SSE-intrinsic paths)"}


# ---- the other rows of SURVEY.md §8 (parity-test configurations and the §8f "next" rows), same bar:
# device-timed with the reference's CPU implementation beside it.  Not the contract's bench line
# (that is config B, the default); run with --workload NAME.
def other_workloads():
    from webrender_b200 import abi
    from workloads import scenes
    return {
        "b_prime": lambda: scenes.alpha_rects_frame(W, H, 1000, random_rects=True, seed=1, color=None),
        "text": lambda: scenes.text_frame(width=W, height=H, n_runs=68, glyphs_per_run=89, seed=2, atlas_size=2048),
        "gradients": lambda: scenes.gradient_frame(width=W, height=H, n_grad=10, full_frame=True),
        "box_shadow": lambda: scenes.box_shadow_frame(width=1024, height=1024, n_clips=1, full_size=(1024, 1024), seed=7),
        "clip_rects": lambda: scenes.clip_mask_frame(),
        "composite": lambda: scenes.composite_frame(W, H, 1024, 512, seed=4),
        "page": lambda: scenes.page_frame(W, H, 1024, 512, seed=1),
        "video_nv12": lambda: scenes.video_frame(W, H, 1920, 1080, "nv12"),
        "video_planar": lambda: scenes.video_frame(W, H, 1920, 1080, "planar"),
        "images": lambda: scenes.image_frame(width=W, height=H, seed=1),
        "blur": lambda: scenes.blur_frame(seed=1, color=True),
        "cache_linear_gradients": lambda: scenes.cached_gradient_frame(abi.KIND_LINEAR_GRADIENT, 2048, 2048, n_tasks=96, seed=1),
        "cache_radial_gradients": lambda: scenes.cached_gradient_frame(abi.KIND_RADIAL_GRADIENT, 2048, 2048, n_tasks=96, seed=1),
        "cache_conic_gradients": lambda: scenes.cached_gradient_frame(abi.KIND_CONIC_GRADIENT, 2048, 2048, n_tasks=96, seed=1),
        "quad_radial_gradients": lambda: scenes.quad_gradient_frame(abi.KIND_QUAD_RADIAL_GRADIENT, W, H, n_quads=24, seed=1),
        "borders_solid": lambda: scenes.border_frame(abi.KIND_BORDER_SOLID, 2048, 2048, n_borders=40, seed=1),
        "borders_complex": lambda: scenes.border_frame(abi.KIND_BORDER_SEGMENT, 2048, 2048, n_borders=40, seed=1, scale=1.5),
        "line_decorations": lambda: scenes.line_decoration_frame(1024, 1024, n_tasks=400, seed=1),
    }


def _frame_pixels(frame):
    """Σ over batches of instance-rect areas where the instance starts with a device rect; else target area."""
    t = frame.passes[-1][-1]
    d = frame.textures[t.texture]
    return d.width * d.height


def run_other_workload(args):
    import numpy as np
    import torch
    from webrender_b200 import abi
    from webrender_b200.device import CudaDevice
    from webrender_b200.frame import draw_frame
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the wrcu backend has no CPU path")
    dev = CudaDevice(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    if args.workload == "update_path":
        line = run_update_path(dev, flush, args)
        print(json.dumps(line))
        dev.close()
        return
    make = other_workloads()[args.workload]
    frame = make()
    # the frame is built once (the frame builder's job upstream); each step is Renderer::render of the C++
    # host mirror (webrender_b200/host/) on it: tables + instances from host memory through the C ABI
    from webrender_b200.host import HostRenderer
    hr = HostRenderer(dev)
    nf = hr.build(frame)
    handles = nf.handles
    for _ in range(max(args.warmup, 3)):
        hr.render_native(nf)
    dev.finish()
    dev.reset_stats()
    ms = []
    for _ in range(args.steps):
        l2_flush(flush)
        dev.timer_begin()
        hr.render_native(nf)
        ms.append(dev.timer_end())
    launches = dev.stats()["kernel_launches"] // max(1, args.steps)
    ms.sort()
    med = ms[len(ms) // 2]
    # the same frame back to back without the flush (what a running compositor sees: code, tables and small
    # targets still in the 126 MB L2) and pipelined (N frames queued, one pair of events): informational
    warm = []
    for _ in range(args.steps):
        dev.timer_begin()
        hr.render_native(nf)
        warm.append(dev.timer_end())
    warm.sort()
    dev.timer_begin()
    for _ in range(args.steps):
        hr.render_native(nf)
    piped = dev.timer_end() / args.steps
    line = {"metric": "frames/s of the named workload", "value": 1e3 / med, "unit": "frames/s", "n_gpus": 1,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": med, "higher_is_better": True,
            "data": "synthetic", "config": {"workload": args.workload, "l2": "flushed between iterations (256 MiB write, then read back: clean lines)",
                                            "host": "wr::Renderer::render (C++ host mirror) per step, CUDA events"},
            "gpu_launches": int(launches), "target_pixels": _frame_pixels(frame),
            "ms_warm_l2": warm[len(warm) // 2], "ms_pipelined": piped}
    if not args.no_cpu_baseline:
        # the reference's own CPU implementation (SWGL, 1 core) on the same frame; bounded to ~15 s
        from oracle.backends import OracleDevice, SwglDevice, have_swgl
        kind = "reference" if have_swgl() else "port"
        d = (SwglDevice if kind == "reference" else OracleDevice)()
        h = draw_frame(d, frame)
        best, reps, t_end = None, 0, time.perf_counter() + 15.0
        while reps < 1 or (time.perf_counter() < t_end and reps < 5):
            t0 = time.perf_counter()
            draw_frame(d, frame, h)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
            reps += 1
        d.close()
        line["cpu_baseline"] = {"value": 1.0 / best, "unit": "frames/s", "cores": 1, "kind": kind,
                                "sample": f"the same frame, best of {reps}"}
    print(json.dumps(line))
    dev.close()


def workloads_summary(local, flush, steps=5):
    """The other §8 rows in the default bench line (device-timed, L2 flushed, C++ host mirror per step): what a
    compositor's frame is made of besides the 1000-layer stress — many small batches (page), the tile composite,
    clip masks, a text page, a scaled video surface.  ms per frame and launches per frame."""
    from webrender_b200.device import CudaDevice
    from webrender_b200.host import HostRenderer
    out = {}
    makes = other_workloads()
    for name in ("page", "composite", "clip_rects", "text", "video_nv12", "images", "gradients"):
        dev = CudaDevice(local)
        try:
            hr = HostRenderer(dev)
            nf = hr.build(makes[name]())
            for _ in range(3):
                hr.render_native(nf)
            dev.finish()
            dev.reset_stats()
            ms = []
            for _ in range(steps):
                l2_flush(flush)
                dev.timer_begin()
                hr.render_native(nf)
                ms.append(dev.timer_end())
            ms.sort()
            out[name] = {"ms_per_frame": ms[len(ms) // 2], "launches": int(dev.stats()["kernel_launches"] // steps)}
            nf.destroy()
            hr.close()
        except Exception as e:   # informational: never lose the headline line
            out[name] = {"error": repr(e)[:160]}
        finally:
            dev.close()
    return out


def run_update_path(dev, flush, args):
    """§8f rank 3: a 2048^2 R8 glyph atlas arriving as 1024 tile uploads out of one staging blob, and a
    64K-block GPU cache arriving as ~5K Copy records; host memory in, device memory out, per step."""
    import numpy as np
    import torch
    from webrender_b200 import abi
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    rng = np.random.RandomState(1)
    size, tile = 2048, 64
    atlas = rng.randint(0, 256, (size, size)).astype(np.uint8)
    rects, off, blob = [], 0, []
    for y in range(0, size, tile):
        for x in range(0, size, tile):
            rects.append((x, y, tile, tile, off, tile))
            blob.append(np.ascontiguousarray(atlas[y:y + tile, x:x + tile]).reshape(-1))
            off += tile * tile
    staging = np.concatenate(blob)
    cache = rng.uniform(0, 1, (65536, 4)).astype(np.float32)
    updates, a = [], 0
    while a < len(cache):
        c = int(min(rng.randint(1, 25), len(cache) - a, 1024 - (a % 1024)))
        updates.append((a, c, a % 1024, a // 1024))
        a += c
    tex = dev.texture_create(abi.FMT_R8, size, size)
    # what a host holds between frames: #[repr(C)] arrays, and the pixels in page-locked memory (the PBO analogue)
    rect_arr, upd_arr = dev.upload_rects(rects), dev.gpu_cache_copies(updates)
    pinned = dev.host_alloc(staging.shape, np.uint8)
    pinned[:] = staging
    zero = dict(prim_headers_f=np.zeros((0, 4), np.float32), prim_headers_i=np.zeros((0, 4), np.int32),
                transforms=np.zeros((0, 4), np.float32), render_tasks=np.zeros((0, 4), np.float32),
                gpu_cache=None, gpu_buffer_f=np.zeros((0, 4), np.float32), gpu_buffer_i=np.zeros((0, 4), np.int32))

    def step():
        dev.gpu_cache_update(64, False, upd_arr, cache)
        dev.frame_begin(zero)
        dev.texture_upload_batch(tex, rect_arr, pinned)
        dev.frame_end()

    for _ in range(3):
        step()
    dev.finish()
    ms = []
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step()
        dev.finish()
        ms.append((time.perf_counter() - t0) * 1e3)
    ms.sort()
    med = ms[len(ms) // 2]
    got = dev.read_pixels(tex, 0, 0, size, size, 1)
    assert np.array_equal(got, atlas), "uploaded atlas differs"
    nbytes = staging.size + cache.nbytes
    line = {"metric": "update-path throughput (host memory in, device memory out)", "value": nbytes / (med * 1e-3) / 1e9,
            "unit": "GB/s", "n_gpus": 1, "steps": args.steps, "ms_per_step": med, "higher_is_better": True,
            "data": "synthetic", "gpu_launches": 2,
            "config": {"workload": "update_path", "atlas": "2048^2 R8 in 1024 64x64 rects", "gpu_cache_blocks": len(cache),
                       "gpu_cache_updates": len(updates), "timing": "host wall clock incl. ctypes marshalling, synchronised"}}
    if not args.no_cpu_baseline:
        from oracle.backends import OracleDevice, SwglDevice, have_swgl
        kind = "reference" if have_swgl() else "port"
        d = (SwglDevice if kind == "reference" else OracleDevice)()
        t = d.texture_create(abi.FMT_R8, size, size)
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            d.gpu_cache_update(64, False, updates, cache)
            d.texture_upload_batch(t, rects, staging)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        d.close()
        line["cpu_baseline"] = {"value": nbytes / best / 1e9, "unit": "GB/s", "cores": 1, "kind": kind,
                                "sample": "the same update lists through the reference's TexSubImage2D plumbing, best of 3"}
    return line


def l2_flush(flush):
    """Evict the 126 MB L2: write a 256 MiB buffer (the contract's flush), then READ it back once so the
    lines left in L2 are clean — otherwise the timed kernel's first misses also pay for writing the flush
    buffer's dirty lines back to DRAM, which a bandwidth-bound kernel sees as up to 2x its own traffic."""
    import torch
    flush.fill_(1)
    flush.view(torch.int64).sum()
    torch.cuda.synchronize()


def roofline_sweep(dev, flush, steps, peak):
    """Config B geometry (full-frame alpha rects in one batch at 3840x2160) at L layers, and B' (1000 seeded
    random rects): where the brush pass is memory-bound and where the on-chip layer loop takes over.
    Per entry: raster-kernel time (CUDA events around the raster kernel alone, L2 flushed), batch time
    (setup + raster), algorithmic GB/s (8 B per pixel-layer), and GB/s on the DRAM bytes the tile-resident
    kernel actually moves (target once in, once out = 2 x 33.2 MB; ncu-measured figures per L are in
    profiles/) with its fraction of the measured HBM peak."""
    import torch
    from webrender_b200 import abi
    from workloads import scenes
    from webrender_b200.frame import Batch, Clear
    from webrender_b200.gpu_types import ortho
    tgt = dev.texture_create(abi.FMT_RGBA8, W, H)
    proj = ortho(W, H)
    out = []
    dev.profile_enable(True)
    cases = [(str(L), lambda L=L: scenes.alpha_rects_frame(W, H, L)) for L in (1, 2, 4, 8, 16, 64, 256, 1000)]
    cases.append(("b_prime", lambda: scenes.alpha_rects_frame(W, H, 1000, random_rects=True, seed=1, color=None)))
    for name, make in cases:
        frame = make()
        layers = scenes.pixel_layers_of_quad_batch(frame)
        tdesc = frame.passes[0][0]
        clear_op = [op for op in tdesc.ops if isinstance(op, Clear)][0]
        batch = [op for op in tdesc.ops if isinstance(op, Batch)][0]
        inst = batch.instance_bytes()
        k_ms, b_ms = [], []
        for it in range(steps + 2):
            dev.frame_begin(frame.tables)
            dev.target_bind(tgt, 0, proj, (0, 0, W, H))
            dev.clear(None, clear_op.color, None)
            dev.finish()
            l2_flush(flush)  # the clear leaves the target in L2: evict it so the batch reads DRAM
            dev.timer_begin()
            dev.draw_batch(batch.kind, batch.features, batch.blend, batch.depth, [0, 0, 0], 0, None,
                           batch.blend_color, inst)
            t = dev.timer_end()
            dev.frame_end()
            if it >= 2:
                b_ms.append(t)
                k_ms.append(dev.last_raster_ms())
        k_ms.sort()
        b_ms.sort()
        km, bm = k_ms[len(k_ms) // 2], b_ms[len(b_ms) // 2]
        dram = 2 * W * H * 4 if name != "b_prime" else None
        e = {"layers": name, "pixel_layers": layers, "raster_kernel_ms": km, "batch_ms": bm,
             "Mpix_s": layers / (km * 1e-3) / 1e6,
             "algorithmic_GBs": layers * BYTES_PER_PIXEL_LAYER / (km * 1e-3) / 1e9}
        e["algorithmic_frac"] = e["algorithmic_GBs"] / peak
        if dram:
            e["dram_bytes_model"] = dram
            e["dram_GBs"] = dram / (km * 1e-3) / 1e9
            e["dram_frac_of_hbm"] = e["dram_GBs"] / peak
        out.append(e)
    dev.profile_enable(False)
    dev.texture_destroy(tgt)
    return out


def run_config_e(dev, rank, world, local, steps, barrier):
    """Config E (SURVEY.md §8e): ONE 8192x4096 frame = 64 picture-cache tiles of 1024x512 (the config-B'
    rect list cut per tile), tiles round-robin over the ranks.  No gather: every rank composites its own
    tiles straight into rank 0's exported framebuffer (bulk-tensor stores over NVLink), ordered by stream
    flags (webrender_b200/multi_gpu.py DirectShardedRenderer).  Strong scaling of a single frame: device
    time per frame (CUDA events on each rank's stream, max over ranks), with the same code on ONE GPU
    (rank 0, all 64 tiles) measured in the same run as the reference."""
    import zlib
    import torch
    import torch.distributed as dist
    from webrender_b200 import multi_gpu
    from webrender_b200.device import CudaDevice
    scene = multi_gpu.tiled_alpha_scene()
    sr = multi_gpu.DirectShardedRenderer(dev, scene, rank, world)
    blobs = [None] * world
    if world > 1:
        dist.all_gather_object(blobs, sr.blob)
    else:
        blobs = [sr.blob]
    sr.connect(blobs)
    for _ in range(3):
        sr.render()
    barrier()
    dev.timer_begin()
    for _ in range(steps):
        sr.render()
    ms = dev.timer_end() / steps
    barrier()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    out = None
    if rank == 0:
        crc = zlib.crc32(sr.read_framebuffer().tobytes())
        # the same frame on one GPU (a second context on this device)
        d1 = CudaDevice(local)
        single = multi_gpu.DirectShardedRenderer(d1, scene, 0, 1)
        single.connect([single.blob])
        for _ in range(3):
            single.render()
        d1.finish()
        d1.timer_begin()
        for _ in range(steps):
            single.render()
        ms1 = d1.timer_end() / steps
        crc1 = zlib.crc32(single.read_framebuffer().tobytes())
        single.close()
        d1.close()
        out = {"workload": "config E: 8192x4096 frame, 64 tiles of 1024x512, 1000 seeded alpha rects cut per tile",
               "scaling": "strong", "n_gpus": world, "ms_per_frame": ms, "fps": 1e3 / ms,
               "Mpix_s": scene.pixel_layers / (ms * 1e-3) / 1e6, "tiles_per_rank": (len(scene.tiles) + world - 1) // world,
               "one_gpu_ms_per_frame": ms1, "speedup_vs_one_gpu": ms1 / ms, "efficiency": ms1 / ms / world,
               "exchange": "none staged: each rank's composite kernel stores its tiles into rank 0's framebuffer "
                           "(CUDA IPC mapping, TMA bulk stores over NVLink); stream-ordered flags, no host sync per frame",
               "nvlink_bytes_per_frame": int(sum((x1 - x0) * (y1 - y0) * 4 for i, (x0, y0, x1, y1) in enumerate(scene.rects)
                                                 if i % world != 0)),
               "timing": "CUDA events on each rank's stream over %d frames, max over ranks" % steps,
               "framebuffer_crc32": crc, "matches_single_gpu": bool(crc == crc1)}
    sr.close()
    return out


def pin_to_gpu_numa_node(local):
    """Run this rank (and allocate its page-locked buffers) on the NUMA node its GPU hangs off: with 8 ranks
    on one host the e2e readbacks otherwise cross the socket interconnect (round 1: 0.74 e2e efficiency)."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


DUMP_PIXELS = 1 << 20   # 16 MiB as float32 BGRA


def dump_framebuffer(out_dir, fb):
    """The framebuffer a caller of the timed path reads back, as float32 BGRA values 0..255 of DUMP_PIXELS
    pixels drawn with a fixed seed (row-major order), so that two builds can be compared output for output."""
    import numpy as np
    px = fb.reshape(-1, 4)
    idx = np.sort(np.random.RandomState(0).choice(px.shape[0], DUMP_PIXELS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "framebuffer.npy"), px[idx].astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="wrcu", choices=["wrcu", "reference"])
    ap.add_argument("--ref-rects", type=int, default=400, help="layers per step for --impl reference")
    ap.add_argument("--ref-cores", type=int, default=0, help="--impl reference: use this many cores (default: all usable)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config-e", action="store_true", help="also run the sharded 8K frame (always on for --gpus > 1)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the layer-depth roofline sweep")
    ap.add_argument("--sweep-only", action="store_true", help="only the layer-depth sweep (for an ncu pass over its kernels)")
    ap.add_argument("--workload", default="config_b",
                    help="config_b (the contract's bench line) or one of the other §8 rows: see other_workloads(), update_path")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="config_b: write what the last timed step drew to DIR/framebuffer.npy (float32 BGRA of a fixed "
                         "seeded sample of 2^20 pixels) for output-for-output comparison of two builds")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "wrcu" or args.workload != "config_b" or args.sweep_only):
        ap.error("--dump-outputs writes the config_b frame of --impl wrcu")
    args.warmup = max(args.warmup, 3) if args.impl == "wrcu" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload != "config_b":
        run_other_workload(args)
        return
    if args.sweep_only:
        import torch
        from webrender_b200.device import CudaDevice
        dev = CudaDevice(0)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        peak, _ = load_peaks()
        print(json.dumps({"roofline_sweep": roofline_sweep(dev, flush, max(2, min(args.steps, 10)), peak)}))
        dev.close()
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the wrcu backend has no CPU path")
    torch.cuda.set_device(local)
    numa_node = pin_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from webrender_b200 import abi
    from workloads import scenes
    from webrender_b200.device import CudaDevice
    from webrender_b200.frame import Batch, Clear
    from webrender_b200.gpu_types import ortho

    # Every rank renders its own full config-B frame (weak scaling: frames are
    # independent render targets; no data-path collective).
    frame = scenes.alpha_rects_frame(W, H, N_RECTS)
    layers = scenes.pixel_layers_of_quad_batch(frame)
    dev = CudaDevice(local)
    tgt = dev.texture_create(abi.FMT_RGBA8, W, H)
    tdesc = frame.passes[0][0]
    clear_op = [op for op in tdesc.ops if isinstance(op, Clear)][0]
    batch = [op for op in tdesc.ops if isinstance(op, Batch)][0]
    inst = batch.instance_bytes()
    proj = ortho(W, H)

    def draw_step():
        dev.frame_begin(frame.tables)
        dev.target_bind(tgt, 0, proj, (0, 0, W, H))
        dev.clear(None, clear_op.color, None)
        dev.draw_batch(batch.kind, batch.features, batch.blend, batch.depth, [0, 0, 0], 0, None,
                       batch.blend_color, inst)
        dev.frame_end()

    def barrier():
        if world > 1:
            dist.barrier()
        dev.finish()
        torch.cuda.synchronize()

    # L2 flush between iterations: write a buffer larger than the 126 MB L2
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    for _ in range(args.warmup):
        draw_step()
    dev.finish()

    # ---- device-resident timing: CUDA events on the context's stream -------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dev.reset_stats()
    barrier()
    kernel_ms = []
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        dev.timer_begin()
        draw_step()
        kernel_ms.append(dev.timer_end())
    barrier()
    st = dev.stats()
    if rank == 0 and args.dump_outputs:
        dump_framebuffer(args.dump_outputs, dev.read_pixels(tgt, 0, 0, W, H, 4))
    if rank == 0 and not sampler.lines:
        # a short timed region can end before nvidia-smi's first 100 ms sample: keep the same load
        # running (untimed) until one arrives, so the clocks line still describes the GPU under this work
        t_lim = time.perf_counter() + 2.0
        while not sampler.lines and time.perf_counter() < t_lim:
            draw_step()
            dev.finish()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = float(sum(kernel_ms))

    # ---- the dominant kernel alone: CUDA events around the draw_batch region ------
    # (init + vertex-stage setup kernel + tile raster kernel; the raster kernel is
    # > 99 % of it, see profiles/)
    batch_ms = []
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        dev.frame_begin(frame.tables)
        dev.target_bind(tgt, 0, proj, (0, 0, W, H))
        dev.clear(None, clear_op.color, None)
        dev.timer_begin()
        dev.draw_batch(batch.kind, batch.features, batch.blend, batch.depth, [0, 0, 0], 0, None,
                       batch.blend_color, inst)
        batch_ms.append(dev.timer_end())
        dev.frame_end()
    kernel_avg_ms = float(sum(batch_ms)) / len(batch_ms)

    # ---- e2e: host buffers in, framebuffer read back to the host, every step -----
    # The call sequence a host makes per frame: tables + instances from host memory
    # (frame_begin / draw_batch copy them H2D), draws, then the framebuffer read back
    # into page-locked host memory.  Like the reference's PBO readback
    # (device/gl.rs:3160-3241) the read is queued behind the frame and overlaps the
    # NEXT frame's draws (two targets, two host buffers); every step's copies finish
    # inside the timed region.
    tgt2 = dev.texture_create(abi.FMT_RGBA8, W, H)
    targets = [tgt, tgt2]
    host_fb = [dev.host_alloc((H, W * 4)), dev.host_alloc((H, W * 4))]
    fences = [0, 0]

    def draw_step_to(t):
        dev.frame_begin(frame.tables)
        dev.target_bind(t, 0, proj, (0, 0, W, H))
        dev.clear(None, clear_op.color, None)
        dev.draw_batch(batch.kind, batch.features, batch.blend, batch.depth, [0, 0, 0], 0, None,
                       batch.blend_color, inst)
        dev.frame_end()

    def e2e_loop(n):
        checksum = 0
        for i in range(n):
            k = i & 1
            if fences[k]:
                dev.fence_wait(fences[k])            # result of step i-2 is in host memory
                checksum += int(host_fb[k][H // 2, W * 2])
            draw_step_to(targets[k])
            fences[k] = dev.read_pixels_async(targets[k], 0, 0, W, H, host_fb[k])
        for k in range(2):
            if fences[k]:
                dev.fence_wait(fences[k])
                checksum += int(host_fb[k][H // 2, W * 2])
                fences[k] = 0
        return checksum

    e2e_loop(2)
    barrier()
    dev.reset_stats()
    e0 = time.perf_counter()
    e2e_loop(args.steps)
    barrier()
    e2e_s = time.perf_counter() - e0
    st_e2e = dev.stats()
    # the same without overlap: synchronous read_pixels after every frame
    barrier()
    s0 = time.perf_counter()
    for _ in range(args.steps):
        draw_step()
        dev._check(dev.lib.wrcu_read_pixels(dev.ctx, tgt, 0, 0, W, H, host_fb[0].ctypes.data, host_fb[0].strides[0]))
    barrier()
    e2e_sync_s = time.perf_counter() - s0

    if world > 1:
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = float(t[0]), float(t[1])

    # ---- config E (SURVEY.md §8e), informational: ONE 8K frame whose 64 tiles are
    # sharded over the ranks, gathered to rank 0 over NCCL and composited there ----
    config_e = None
    if world > 1 or args.config_e:
        try:
            config_e = run_config_e(dev, rank, world, local, max(5, args.steps), barrier)
        except Exception as e:  # keep the headline line even if the extra fails
            config_e = {"error": repr(e)[:200]}

    if rank == 0:
        peak, peak_src = load_peaks()
        ms_per_step = total_ms / args.steps
        value = world * layers / (ms_per_step * 1e-3) / 1e6
        achieved = layers * BYTES_PER_PIXEL_LAYER / (kernel_avg_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        prof = os.path.join(ROOT, "profiles", "hot_kernel.json")
        if os.path.exists(prof):
            # ncu's DRAM bytes describe the kernel they were captured from: use them only while the source
            # that defines the kernel is unchanged (tools/hot_kernel.py stamps its SHA-1 into the record)
            import hashlib
            pj = json.load(open(prof))
            sha = hashlib.sha1(open(os.path.join(ROOT, "webrender_b200", "csrc", "raster.cuh"), "rb").read()).hexdigest()
            if pj.get("raster_cuh_sha1") == sha:
                traffic = pj["dram_bytes_read"] + pj["dram_bytes_write"]
                traffic_src = pj.get("source")
            else:
                traffic_src = "stale: profiles/hot_kernel.json was captured from another version of raster.cuh"
        line = {
            "metric": "Mpix/s composited at 3840x2160 (alpha-blend brush pass)",
            "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD_B,
                       "pixel_layers_per_step": layers, "frames_per_gpu_per_step": 1,
                       "l2": "flushed between timed iterations (256 MiB write)", "timing": "CUDA events on the wrcu stream",
                       "multi_gpu": "value: every rank renders its own config-B frame (independent render targets, no "
                                    "data-path collective: weak scaling); config_e: ONE 8K frame sharded by tile over the "
                                    "ranks into a shared framebuffer (strong scaling, its own one-GPU reference)",
                       "numa_node_rank0": numa_node},
            "clocks": clocks,
            "gpu_launches": int(st["kernel_launches"]),
            "e2e": {"value": world * layers * args.steps / e2e_s / 1e6, "unit": "Mpix/s",
                    "h2d_bytes_per_step": int(st_e2e["h2d_bytes"] // args.steps),
                    "d2h_bytes_per_step": int(st_e2e["d2h_bytes"] // args.steps),
                    "how": "wrcu C ABI per frame: frame_begin(tables) + clear + draw_batch(instances) from host memory, "
                           "read_pixels_async into page-locked host memory overlapping the next frame (2 targets), "
                           "fence_wait before the buffer is reused",
                    "sync_value": world * layers * args.steps / e2e_sync_s / 1e6},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "wr_raster_solid_premult", "kernel_ms": kernel_avg_ms,
                         "algorithmic_bytes_per_launch": layers * BYTES_PER_PIXEL_LAYER, "peak_source": peak_src,
                         "note": "algorithmic bytes = 8 B per pixel-layer (SURVEY.md §8d); the tile-resident kernel "
                                 "keeps layers on chip, so DRAM traffic is ~2 x 33 MB per launch and achieved may exceed peak"},
        }
        if not args.no_sweep:
            line["roofline_sweep"] = roofline_sweep(dev, flush, max(5, min(args.steps, 10)), peak)
        if config_e is not None:
            line["config_e"] = config_e
        if world == 1 and not args.no_sweep:
            line["workloads"] = workloads_summary(local, flush)
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_sample()
        print(json.dumps(line))
    dev.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
