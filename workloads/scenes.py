"""Synthetic frames for the configurations BASELINE.json names (SURVEY.md §8d).

Each builder returns a `Frame` holding exactly the binary tables and batches
the reference's frame builder would hand to `Renderer::draw_frame` for that
scene; deterministic (seeded numpy RNG), no file or network input.
"""
import numpy as np

from webrender_b200 import abi
from webrender_b200.frame import Batch, Clear, Frame, Target, TextureDesc
from webrender_b200.gpu_types import (FrameTables, INVALID_SEGMENT_INDEX, PART_ALL, QF_APPLY_DEVICE_CLIP, quad_instance)


def alpha_rects_frame(width=3840, height=2160, n_rects=1000, random_rects=False, seed=1,
                      color=(0.05, 0.05, 0.05, 0.05), clear_color=(0.3, 0.0, 0.0, 1.0),
                      blend=abi.BLEND_PREMULTIPLIED_ALPHA):
    """Config B — examples/alpha_perf.rs:35-49: N overlapping alpha rects in ONE
    batch of `Quad(ColorOrTexture)` instances (plain rects take the quad path,
    prepare.rs:216-259) over a cleared colour target.  `random_rects` gives the
    B' variant: seeded uniform origins, sizes in [64, 1024] px."""
    t = FrameTables()
    task = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    rng = np.random.RandomState(seed)
    inst = []
    for i in range(n_rects):
        if random_rects:
            w, h = rng.randint(64, 1025, size=2)
            x0 = int(rng.randint(0, max(1, width - 32)))
            y0 = int(rng.randint(0, max(1, height - 32)))
            rect = (float(x0), float(y0), float(min(width, x0 + w)), float(min(height, y0 + h)))
        else:
            rect = (0.0, 0.0, float(width), float(height))
        if color is None:
            a = rng.uniform(0.05, 1.0)
            c = tuple(float(v) for v in (rng.uniform(0, a), rng.uniform(0, a), rng.uniform(0, a), a))
        else:
            c = color
        prim_f = t.add_quad_prim(rect, rect, c)
        prim_i = t.add_quad_header(0, i + 1)
        inst.append(quad_instance(prim_i, prim_f, QF_APPLY_DEVICE_CLIP, 0, PART_ALL, INVALID_SEGMENT_INDEX, task))
    inst = np.stack(inst)
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    ops = [Clear(color=clear_color),
           Batch(abi.KIND_QUAD_TEXTURED, inst, blend=blend)]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def pixel_layers_of_quad_batch(frame: Frame):
    """Σ covered pixels over the quad instances of the first batch (axis-aligned,
    identity transform): the unit of work of the Mpix/s metric."""
    tgt = frame.passes[0][0]
    desc = frame.textures[tgt.texture]
    batch = [op for op in tgt.ops if isinstance(op, Batch)][0]
    gf = frame.tables["gpu_buffer_f"]
    total = 0
    for row in batch.instances:
        b = gf[row[1]]
        x0, y0 = max(0.0, b[0]), max(0.0, b[1])
        x1, y1 = min(float(desc.width), b[2]), min(float(desc.height), b[3])
        total += max(0, int(np.floor(x1 + 0.5)) - int(np.floor(x0 + 0.5))) * \
            max(0, int(np.floor(y1 + 0.5)) - int(np.floor(y0 + 0.5)))
    return total


def _rand_rect(rng, width, height, min_size=8, max_size=None, integer=True):
    max_size = max_size or max(width, height)
    w = rng.randint(min_size, max(min_size + 1, min(max_size, width)))
    h = rng.randint(min_size, max(min_size + 1, min(max_size, height)))
    x0 = rng.randint(-w // 4, max(1, width - w // 2))
    y0 = rng.randint(-h // 4, max(1, height - h // 2))
    if integer:
        return (float(x0), float(y0), float(x0 + w), float(y0 + h))
    fx, fy = rng.uniform(0, 1, 2)
    return (float(np.float32(x0 + fx)), float(np.float32(y0 + fy)),
            float(np.float32(x0 + w + fy)), float(np.float32(y0 + h + fx)))


def rotation_matrix(deg, cx, cy, sx=1.0, sy=1.0):
    """2D rotation by `deg` about (cx, cy), optionally with non-uniform scale, as a 4x4."""
    a = np.deg2rad(deg)
    c, s = float(np.cos(a)), float(np.sin(a))
    m = np.eye(4, dtype=np.float64)
    m[0, 0], m[0, 1], m[1, 0], m[1, 1] = c * sx, -s * sy, s * sx, c * sy
    m[0, 3] = cx - (m[0, 0] * cx + m[0, 1] * cy)
    m[1, 3] = cy - (m[1, 0] * cx + m[1, 1] * cy)
    return m.astype(np.float32)


def brush_solid_frame(width=640, height=360, n_opaque=12, n_alpha=24, seed=1, with_masks=True,
                      fractional=False, force_aa=False, device_pixel_scale=1.0, rotate=None, occlude_alpha=False):
    """Brush(Solid) batches the way draw_alpha_batch_container issues them
    (renderer/mod.rs:2804-2969): an opaque batch front-to-back with depth
    LEQUAL + write, then an alpha batch with premultiplied blending, depth test
    only, and per-instance clip masks sampled from an R8 alpha target."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), device_pixel_scale, (0.0, 0.0))
    mw, mh = 256, 256
    mask = rng.randint(0, 256, size=(mh, mw)).astype(np.uint8)
    mask[rng.randint(0, mh, 40)[:, None], :] = 255
    mask[:, rng.randint(0, mw, 40)] = 0
    z = 1
    opaque, alpha = [], []
    # a rotated (non-axis-aligned) spatial node: transform id carries the "complex" bit
    # (TransformPaletteId, gpu_types.rs:730-760), which turns edge AA on (brush.glsl:118-134)
    xf = 0
    if rotate is not None:
        xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0, 1.0, 0.9), axis_aligned=False)

    def add(rect, clip_rect, color, opacity, clip_task, flags=0, edge=0):
        nonlocal z
        addr = t.push_gpu_cache([color])
        hdr = t.add_prim_header(rect, clip_rect, z, addr, xf, pic, (int(opacity * 65535), 0, 0, 0))
        z += 1
        return brush_instance(hdr, clip_task, 0xFFFF, edge, flags, 0)

    s = 1.0 / device_pixel_scale
    # occlude_alpha: the opaque prims sit IN FRONT of the alpha prims (larger z ids), so alpha spans are cut
    # into passing depth runs by them (an opaque box over translucent content)
    if occlude_alpha:
        z = 10000
    for _ in range(n_opaque):
        r = _rand_rect(rng, width, height, 16, integer=not fractional)
        r = tuple(v * s for v in r)
        c = tuple(float(v) for v in rng.uniform(0, 1, 3)) + (1.0,)
        opaque.append(add(r, (-1e9, -1e9, 1e9, 1e9), c, 1.0, CLIP_TASK_EMPTY))
    if occlude_alpha:
        z = 1
    for i in range(n_alpha):
        r = _rand_rect(rng, width, height, 16, integer=not fractional)
        a = rng.uniform(0.1, 1.0)
        c = tuple(float(v * a) for v in rng.uniform(0, 1, 3)) + (float(a),)
        clip_task = CLIP_TASK_EMPTY
        if with_masks and i % 2 == 0:
            # mask region: device rect (sx,sy,w,h) stored in the mask texture at (mx,my)
            w_ = int(min(r[2] - r[0], 120))
            h_ = int(min(r[3] - r[1], 100))
            sx, sy = int(np.floor(r[0])) + rng.randint(0, 8), int(np.floor(r[1])) + rng.randint(0, 8)
            mx, my = rng.randint(0, mw - w_), rng.randint(0, mh - h_)
            clip_task = t.add_render_task((float(mx), float(my), float(mx + w_), float(my + h_)), 1.0,
                                          (float(sx), float(sy)))
        clip = (-1e9, -1e9, 1e9, 1e9)
        if i % 3 == 0:
            clip = (r[0] + 3.0, r[1] + 2.0, r[2] - 5.0, r[3] - 1.0)
        r = tuple(v * s for v in r)
        clip = tuple(v * s for v in clip)
        flags = 1024 if force_aa else 0
        edge = (i % 16) if force_aa else 0
        alpha.append(add(r, clip, c, rng.uniform(0.3, 1.0), clip_task, flags, edge))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "depth": TextureDesc(abi.FMT_DEPTH24, width, height),
                "mask": TextureDesc(abi.FMT_R8, mw, mh, mask)}
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0), depth=1.0)]
    if opaque:
        ops.append(Batch(abi.KIND_BRUSH_SOLID, np.stack(opaque[::-1]), blend=abi.BLEND_NONE,
                         depth=abi.DEPTH_TEST_WRITE))
    if alpha:
        ops.append(Batch(abi.KIND_BRUSH_SOLID, np.stack(alpha), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                         depth=abi.DEPTH_TEST, features=abi.FEAT_ALPHA_PASS, clip_mask="mask"))
    return Frame(t.arrays(), textures, [[Target("target", depth="depth", ops=ops)]])


def clip_mask_frame(width=512, height=384, n_clips=10, seed=1, fractional=False, scale=1.0):
    """An alpha (R8) target filled the way draw_alpha_target does it
    (renderer/mod.rs:3754-3929): clear to one, primary rounded-rect clips with
    blending off, then secondary clips multiplied in (ZERO, SRC_COLOR).  Mixes
    the FAST_PATH (uniform radius) and general (per-corner elliptical radii)
    programs and both clip modes."""
    from webrender_b200.gpu_types import clip_rect_instance
    rng = np.random.RandomState(seed)
    t = FrameTables()
    xf = t.add_transform(scale_matrix(scale)) if scale != 1.0 else 0
    fast, slow, fast2, slow2 = [], [], [], []
    for i in range(n_clips):
        # mask task region inside the R8 target
        w, h = int(rng.randint(24, 200)), int(rng.randint(24, 160))
        tx, ty = int(rng.randint(0, width - w)), int(rng.randint(0, height - h))
        sx, sy = int(rng.randint(0, 500)), int(rng.randint(0, 500))
        # the clip rect in local space roughly covering the task's screen rect
        off = rng.uniform(-6, 6, 4) if fractional else rng.randint(-6, 7, 4).astype(np.float64)
        rect = ((sx + off[0]) / scale, (sy + off[1]) / scale, (sx + w + off[2]) / scale, (sy + h + off[3]) / scale)
        rw, rh = rect[2] - rect[0], rect[3] - rect[1]
        mode = float(i % 3 == 2)
        uniform = i % 2 == 0
        if uniform:
            r = float(rng.uniform(2, min(rw, rh) / 2)) if fractional else float(rng.randint(2, max(3, int(min(rw, rh) / 2))))
            radii = ((r, r),) * 4
        else:
            radii = tuple((float(rng.uniform(1, rw / 2)), float(rng.uniform(1, rh / 2))) for _ in range(4))
        inst = clip_rect_instance((0.0, 0.0, float(w), float(h)), (float(tx), float(ty)), (float(sx), float(sy)),
                                  scale, xf, xf, (rect[0], rect[1]), rect, mode, radii)
        primary = i < n_clips * 2 // 3
        (fast if uniform else slow).append(inst) if primary else (fast2 if uniform else slow2).append(inst)
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0))]
    for lst, feat, blend in ((slow, 0, abi.BLEND_NONE), (fast, abi.FEAT_FAST_PATH, abi.BLEND_NONE),
                             (slow2, 0, abi.BLEND_MULTIPLY), (fast2, abi.FEAT_FAST_PATH, abi.BLEND_MULTIPLY)):
        if lst:
            ops.append(Batch(abi.KIND_CLIP_RECTANGLE, np.stack(lst), blend=blend, features=feat))
    textures = {"mask": TextureDesc(abi.FMT_R8, width, height)}
    return Frame(t.arrays(), textures, [[Target("mask", ops=ops)]])


def scale_matrix(s):
    m = np.eye(4, dtype=np.float32)
    m[0, 0] = m[1, 1] = s
    return m


def rounded_rects_frame(width=640, height=400, n_rects=6, seed=1, fractional=False, device_pixel_scale=1.0,
                        filter=abi.LINEAR, spec=None, surface=(512, 512), rotate=None):
    """Config A flavour (wrench/reftests/aa/rounded-rects.yaml): solid rects with
    rounded-rect clips drawn the Indirect way (quad.rs:722-792, 239-264):
      pass 0, off-screen colour target: each rect as an untextured Quad with
        blending off (handle_prims, mod.rs:2199), then its clip multiplied in with
        ps_quad_mask (FAST_PATH for a uniform radius) (handle_clips, mod.rs:2278);
      pass 1, picture-cache tile: one textured Quad per rect sampling the
        off-screen task, premultiplied-alpha blended."""
    from webrender_b200.gpu_types import mask_instance, QF_IS_MASK
    rng = np.random.RandomState(seed)
    t = FrameTables()
    sw, sh = surface
    tile_task = t.add_render_task((0.0, 0.0, float(width), float(height)), device_pixel_scale, (0.0, 0.0))
    prims, masks_fast, masks_slow, composites = [], [], [], []
    # `rotate`: the textured quads that composite the off-screen tasks into the tile sit under a transformed spatial
    # node (a rotation, or via with_transform any 4x4 — a perspective one sends them through draw_perspective)
    cxf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0), axis_aligned=False) if rotate is not None else 0
    cursor_x, cursor_y, row_h = 0, 0, 0
    s = device_pixel_scale
    if spec is not None:
        n_rects = len(spec)
    for i in range(n_rects):
        if spec is not None:
            (sx0, sy0, sx1, sy1), scolor, sradii = spec[i][:3]
            smode = float(spec[i][3]) if len(spec[i]) > 3 else 0.0
            w, h = int(sx1 - sx0), int(sy1 - sy0)
        else:
            w, h = int(rng.randint(40, 220)), int(rng.randint(30, 160))
        if cursor_x + w > sw:
            cursor_x, cursor_y, row_h = 0, cursor_y + row_h, 0
        tx, ty = cursor_x, cursor_y
        cursor_x += w
        row_h = max(row_h, h)
        # device-space rect of the primitive, local = device / scale
        if spec is not None:
            dx, dy = int(sx0), int(sy0)
            rect = (float(sx0), float(sy0), float(sx1), float(sy1))
            color = scolor
        else:
            dx, dy = int(rng.randint(0, width - w)), int(rng.randint(0, height - h))
            fo = rng.uniform(0, 1, 2) if fractional else (0.0, 0.0)
            rect = ((dx + fo[0]) / s, (dy + fo[1]) / s, (dx + w - fo[1]) / s, (dy + h - fo[0]) / s)
            a = rng.uniform(0.3, 1.0)
            color = tuple(float(v * a) for v in rng.uniform(0, 1, 3)) + (float(a),)
        task = t.add_render_task((float(tx), float(ty), float(tx + w), float(ty + h)), s, (float(dx), float(dy)))
        prim_f = t.add_quad_prim(rect, rect, color)
        prim_i = t.add_quad_header(0, i + 1)
        qi = quad_instance(prim_i, prim_f, QF_APPLY_DEVICE_CLIP, 0, PART_ALL, INVALID_SEGMENT_INDEX, task)
        prims.append(qi)
        rw, rh = rect[2] - rect[0], rect[3] - rect[1]
        uniform = i % 2 == 0
        mode = float(i % 5 == 4)
        if spec is not None:
            mode = smode
            uniform = not isinstance(sradii, (list, tuple))
        if spec is not None and uniform:
            r = float(sradii)
            clip_addr = t.push_gpu_buffer_f([rect, (r, r, r, r), (mode, 0, 0, 0)])
        elif spec is not None:
            (tl, tr, bl, br) = sradii   # radii_top = (tl, tr), radii_bottom = (bl, br): ps_quad_mask.glsl:55-60
            clip_addr = t.push_gpu_buffer_f([rect, (tl[0], tl[1], tr[0], tr[1]), (bl[0], bl[1], br[0], br[1]),
                                             (mode, 0, 0, 0)])
        elif uniform:
            r = float(rng.uniform(2, min(rw, rh) / 2)) if fractional else float(rng.randint(2, max(3, int(min(rw, rh) / 2))))
            clip_addr = t.push_gpu_buffer_f([rect, (r, r, r, r), (mode, 0, 0, 0)])
        else:
            rad = [float(rng.uniform(1, rw / 2)) if k % 2 == 0 else float(rng.uniform(1, rh / 2)) for k in range(8)]
            clip_addr = t.push_gpu_buffer_f([rect, rad[0:4], rad[4:8], (mode, 0, 0, 0)])
        mprim_f = t.add_quad_prim(rect, rect, (1.0, 1.0, 1.0, 1.0))
        mqi = quad_instance(prim_i, mprim_f, QF_APPLY_DEVICE_CLIP | QF_IS_MASK, 0, PART_ALL, INVALID_SEGMENT_INDEX, task)
        (masks_fast if uniform else masks_slow).append(mask_instance(mqi, 0, clip_addr, 0))
        # further clips of the same primitive (spec[i][4] = [(clip rect, uniform radius, mode), ...]): one more
        # ps_quad_mask instance each, multiplied into the same task (build_mask_tasks, render_target.rs:1192-1442)
        for crect, cradius, cmode in (spec[i][4] if spec is not None and len(spec[i]) > 4 else []):
            r = float(cradius)
            caddr = t.push_gpu_buffer_f([tuple(float(v) for v in crect), (r, r, r, r), (float(cmode), 0, 0, 0)])
            masks_fast.append(mask_instance(mqi, 0, caddr, 0))
        # composite: textured quad, uv rect = the task rect in the off-screen surface
        cprim_f = t.add_quad_prim(rect, rect, (1.0, 1.0, 1.0, 1.0),
                                  uv_rect=(float(tx), float(ty), float(tx + w), float(ty + h)))
        cprim_i = t.add_quad_header(cxf, 100 + i)
        composites.append(quad_instance(cprim_i, cprim_f, QF_APPLY_DEVICE_CLIP, 0, PART_ALL, INVALID_SEGMENT_INDEX,
                                        tile_task))
    textures = {"surface": TextureDesc(abi.FMT_RGBA8, sw, sh, filter=filter),
                "target": TextureDesc(abi.FMT_RGBA8, width, height)}
    p0 = [Clear(color=(0.0, 0.0, 0.0, 0.0)), Batch(abi.KIND_QUAD_TEXTURED, np.stack(prims), blend=abi.BLEND_NONE)]
    if masks_fast:
        p0.append(Batch(abi.KIND_QUAD_MASK, np.stack(masks_fast), blend=abi.BLEND_MULTIPLY, features=abi.FEAT_FAST_PATH))
    if masks_slow:
        p0.append(Batch(abi.KIND_QUAD_MASK, np.stack(masks_slow), blend=abi.BLEND_MULTIPLY))
    p1 = [Clear(color=(1.0, 1.0, 1.0, 1.0)),
          Batch(abi.KIND_QUAD_TEXTURED, np.stack(composites), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                color=("surface", "", ""))]
    return Frame(t.arrays(), textures, [[Target("surface", ops=p0)], [Target("target", ops=p1)]])


def image_frame(width=640, height=360, n_opaque=8, n_alpha=20, seed=1, filter=abi.LINEAR, one_to_one=False,
                fractional=False, rotate=None, occlude_alpha=False):
    """Brush(Image) batches: an opaque batch (depth write, blending off) and an
    alpha batch (premultiplied over, depth test) sampling one RGBA8 atlas, with
    colour modes Image / ColorBitmap / Alpha(drop-shadow override), 1:1 and
    scaled mappings, plus segment-relative texel-rect (nine-patch style) instances."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    aw, ah = 256, 192
    atlas = rng.randint(0, 256, size=(ah, aw, 4)).astype(np.uint8)
    # premultiply so colours are valid
    a = atlas[..., 3:4].astype(np.uint16)
    atlas[..., :3] = (atlas[..., :3].astype(np.uint16) * a // 255).astype(np.uint8)
    z = 1
    opaque, alpha = [], []
    xf = 0
    if rotate is not None:
        xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0, 0.95, 1.0), axis_aligned=False)

    def add(rect, uv, color, color_mode, opacity, flags=0, segment=None, stretch=(-1.0, -1.0)):
        nonlocal z
        blocks = [color, (0.0, 0.0, 0.0, 0.0), (stretch[0], stretch[1], 0.0, 0.0)]
        seg_index = 0xFFFF
        if segment is not None:
            blocks += [segment[0], segment[1]]
            seg_index = 0
        addr = t.push_gpu_cache(blocks)
        res = t.push_gpu_cache([uv, (0.0, 0.0, 0.0, 0.0)])
        hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), z, addr, xf, pic,
                                (color_mode | (1 << 16), 0, int(opacity * 65535), 0))
        z += 1
        return brush_instance(hdr, CLIP_TASK_EMPTY, seg_index, 0, flags, res)

    def rand_uv(w, h):
        if one_to_one:
            uw, uh = int(w), int(h)
        else:
            uw, uh = int(rng.randint(4, 120)), int(rng.randint(4, 100))
        uw, uh = min(uw, aw - 1), min(uh, ah - 1)
        u0, v0 = int(rng.randint(0, aw - uw)), int(rng.randint(0, ah - uh))
        return (float(u0), float(v0), float(u0 + uw), float(v0 + uh))

    if occlude_alpha:  # opaque prims in front of the alpha prims: alpha spans split into depth runs
        z = 10000
    for _ in range(n_opaque):
        r = _rand_rect(rng, width, height, 16, 200, integer=not fractional)
        opaque.append(add(r, rand_uv(r[2] - r[0], r[3] - r[1]), (1.0, 1.0, 1.0, 1.0), 4, 1.0))
    if occlude_alpha:
        z = 1
    for i in range(n_alpha):
        r = _rand_rect(rng, width, height, 16, 200, integer=not fractional)
        mode = [4, 4, 3, 0, 4][i % 5]
        col = (1.0, 1.0, 1.0, 1.0) if i % 4 == 0 else tuple(float(v) for v in rng.uniform(0.2, 1.0, 4))
        if i % 7 == 6:
            # segment-relative texel rect: the middle ninth of the uv rect on the middle of the prim
            rw, rh = r[2] - r[0], r[3] - r[1]
            seg = ((float(int(rw / 4)), float(int(rh / 4)), float(int(rw * 3 / 4)), float(int(rh * 3 / 4))),
                   (0.25, 0.25, 0.75, 0.75))
            alpha.append(add(r, rand_uv(rw, rh), col, mode, rng.uniform(0.4, 1.0), flags=2 | 512, segment=seg))
        else:
            alpha.append(add(r, rand_uv(r[2] - r[0], r[3] - r[1]), col, mode, rng.uniform(0.4, 1.0)))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "depth": TextureDesc(abi.FMT_DEPTH24, width, height),
                "atlas": TextureDesc(abi.FMT_RGBA8, aw, ah, atlas.reshape(ah, aw * 4), filter=filter)}
    ops = [Clear(color=(0.2, 0.3, 0.4, 1.0), depth=1.0)]
    if opaque:
        ops.append(Batch(abi.KIND_BRUSH_IMAGE, np.stack(opaque[::-1]), blend=abi.BLEND_NONE, depth=abi.DEPTH_TEST_WRITE,
                         features=abi.FEAT_TEXTURE_2D, color=("atlas", "", "")))
    if alpha:
        ops.append(Batch(abi.KIND_BRUSH_IMAGE, np.stack(alpha), blend=abi.BLEND_PREMULTIPLIED_ALPHA, depth=abi.DEPTH_TEST,
                         features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D, color=("atlas", "", "")))
    return Frame(t.arrays(), textures, [[Target("target", depth="depth", ops=ops)]])


def page_frame(width=3840, height=2160, tile_w=1024, tile_h=512, seed=1, clips=12):
    """What a page costs a compositor: MANY SMALL batches.  Three passes as draw_frame issues them
    (renderer/mod.rs:4525-4841): (1) an alpha target of rounded-rect clip masks (cs_clip_rectangle, primary and
    secondary, fast and general programs); (2) every picture-cache tile of the 4K page (1024x512 tiles) as its own
    target: clear, opaque solids and images front to back with depth write, then alpha batches in order — masked /
    anti-aliased solids, images, a linear gradient, two text runs; (3) the tile list composited into the framebuffer.
    ~7 batches per tile x 20 tiles + masks + composite = ~150 draws of 2-60 instances each."""
    from webrender_b200.gpu_types import (brush_instance, glyph_instance, clip_rect_instance, composite_instance,
                            build_gradient_table, CLIP_TASK_EMPTY)
    rng = np.random.RandomState(seed)
    t = FrameTables()
    textures = {}
    # ---- pass 1: clip masks into an R8 alpha target ------------------------------------------------------
    mw, mh = 1024, 512
    fast, slow, fast2 = [], [], []
    mask_tasks = []   # (render task address of the mask region, w, h)
    for i in range(clips):
        w, h = int(rng.randint(60, 200)), int(rng.randint(40, 140))
        tx, ty = (i % 4) * 256 + int(rng.randint(0, 40)), (i // 4) * 160 + int(rng.randint(0, 16))
        sx, sy = int(rng.randint(0, tile_w - w)), int(rng.randint(0, tile_h - h))
        rect = (float(sx + 2), float(sy + 2), float(sx + w - 2), float(sy + h - 2))
        uniform = i % 2 == 0
        if uniform:
            r = float(rng.randint(4, 20))
            radii = ((r, r),) * 4
        else:
            radii = tuple((float(rng.uniform(3, 28)), float(rng.uniform(3, 20))) for _ in range(4))
        inst = clip_rect_instance((0.0, 0.0, float(w), float(h)), (float(tx), float(ty)), (float(sx), float(sy)),
                                  1.0, 0, 0, (rect[0], rect[1]), rect, 0.0, radii)
        (fast if uniform else slow).append(inst)
        if i % 4 == 0:   # a secondary clip multiplied into the same region
            r2 = (rect[0] + 10.0, rect[1] + 6.0, rect[2] - 14.0, rect[3] - 8.0)
            fast2.append(clip_rect_instance((0.0, 0.0, float(w), float(h)), (float(tx), float(ty)), (float(sx), float(sy)),
                                            1.0, 0, 0, (r2[0], r2[1]), r2, 0.0, ((8.0, 8.0),) * 4))
        mask_tasks.append((t.add_render_task((float(tx), float(ty), float(tx + w), float(ty + h)), 1.0,
                                             (float(sx), float(sy))), sx, sy, w, h))
    mops = [Clear(color=(1.0, 1.0, 1.0, 1.0))]
    for lst, feat, blend in ((slow, 0, abi.BLEND_NONE), (fast, abi.FEAT_FAST_PATH, abi.BLEND_NONE),
                             (fast2, abi.FEAT_FAST_PATH, abi.BLEND_MULTIPLY)):
        if lst:
            mops.append(Batch(abi.KIND_CLIP_RECTANGLE, np.stack(lst), blend=blend, features=feat))
    textures["mask"] = TextureDesc(abi.FMT_R8, mw, mh)
    # ---- shared inputs: an image atlas and a glyph atlas --------------------------------------------------
    aw, ah = 512, 512
    atlas = rng.randint(0, 256, size=(ah, aw, 4)).astype(np.uint8)
    al = atlas[..., 3:4].astype(np.uint16)
    atlas[..., :3] = (atlas[..., :3].astype(np.uint16) * al // 255).astype(np.uint8)
    textures["atlas"] = TextureDesc(abi.FMT_RGBA8, aw, ah, atlas.reshape(ah, aw * 4))
    gsz = 512
    cells = gsz // 16
    gtex = np.zeros((gsz, gsz), dtype=np.uint8)
    glyph_res = []
    for gy in range(cells):
        for gx in range(cells):
            gw, gh = int(rng.randint(4, 17)), int(rng.randint(4, 17))
            gtex[gy * 16: gy * 16 + gh, gx * 16: gx * 16 + gw] = rng.randint(0, 256, size=(gh, gw)).astype(np.uint8)
            glyph_res.append((gx * 16, gy * 16, gw, gh))
    textures["glyphs"] = TextureDesc(abi.FMT_R8, gsz, gsz, gtex)
    glyph_addr = {}
    # ---- pass 2: the picture-cache tiles ------------------------------------------------------------------
    cols, rows = (width + tile_w - 1) // tile_w, (height + tile_h - 1) // tile_h
    tile_targets, comp = [], []
    ti = 0
    for ry in range(rows):
        for cx in range(cols):
            name, dname = "tile%d" % ti, "tile%d_depth" % ti
            textures[name] = TextureDesc(abi.FMT_RGBA8, tile_w, tile_h, filter=abi.NEAREST)
            textures[dname] = TextureDesc(abi.FMT_DEPTH24, tile_w, tile_h)
            ox, oy = float(cx * tile_w), float(ry * tile_h)
            pic = t.add_render_task((0.0, 0.0, float(tile_w), float(tile_h)), 1.0, (ox, oy))
            z = 1

            def prim(rect, clip, blocks, user=(65535, 0, 0, 0), res=None, flags=0, edge=0, clip_task=CLIP_TASK_EMPTY):
                nonlocal z
                addr = t.push_gpu_cache(blocks)
                hdr = t.add_prim_header(rect, clip, z, addr, 0, pic, user)
                z += 1
                return brush_instance(hdr, clip_task, 0xFFFF, edge, flags, 0 if res is None else res)

            def local(r):  # a rect inside this tile, in page space
                return (r[0] + ox, r[1] + oy, r[2] + ox, r[3] + oy)
            noclip = (-1e9, -1e9, 1e9, 1e9)
            z = 1000
            osolid = [prim(local(_rand_rect(rng, tile_w, tile_h, 40, 400)), noclip,
                           [tuple(float(v) for v in rng.uniform(0, 1, 3)) + (1.0,)]) for _ in range(6)]
            oimg = []
            for _ in range(3):
                r = _rand_rect(rng, tile_w, tile_h, 40, 300)
                uw, uh = min(int(r[2] - r[0]), aw - 1), min(int(r[3] - r[1]), ah - 1)
                u0, v0 = int(rng.randint(0, aw - uw)), int(rng.randint(0, ah - uh))
                res = t.push_gpu_cache([(float(u0), float(v0), float(u0 + uw), float(v0 + uh)), (0.0, 0.0, 0.0, 0.0)])
                oimg.append(prim(local(r), noclip, [(1.0, 1.0, 1.0, 1.0), (0.0, 0.0, 0.0, 0.0), (-1.0, -1.0, 0.0, 0.0)],
                                 user=(4 | (1 << 16), 0, 65535, 0), res=res))
            z = 1
            asolid = []
            for i in range(8):
                r = _rand_rect(rng, tile_w, tile_h, 30, 300)
                a = float(rng.uniform(0.2, 0.9))
                c = tuple(float(v * a) for v in rng.uniform(0, 1, 3)) + (a,)
                ct = CLIP_TASK_EMPTY
                if i % 3 == 0:
                    task, sx, sy, w, h = mask_tasks[int(rng.randint(0, len(mask_tasks)))]
                    r = (float(sx), float(sy), float(sx + w), float(sy + h))
                    ct = task
                asolid.append(prim(local(r), noclip, [c], user=(int(rng.uniform(0.4, 1.0) * 65535), 0, 0, 0),
                                   flags=1024 if i % 2 else 0, edge=(i % 16) if i % 2 else 0, clip_task=ct))
            aimg = []
            for i in range(6):
                r = _rand_rect(rng, tile_w, tile_h, 30, 260)
                uw, uh = int(rng.randint(16, 200)), int(rng.randint(16, 160))
                u0, v0 = int(rng.randint(0, aw - uw)), int(rng.randint(0, ah - uh))
                res = t.push_gpu_cache([(float(u0), float(v0), float(u0 + uw), float(v0 + uh)), (0.0, 0.0, 0.0, 0.0)])
                col = tuple(float(v) for v in rng.uniform(0.3, 1.0, 4))
                aimg.append(prim(local(r), noclip, [col, (0.0, 0.0, 0.0, 0.0), (-1.0, -1.0, 0.0, 0.0)],
                                 user=(4 | (1 << 16), 0, int(rng.uniform(0.5, 1.0) * 65535), 0), res=res))
            grads = []
            for i in range(2):
                r = _rand_rect(rng, tile_w, tile_h, 100, 500)
                stops = [(0.0, tuple(float(v * 0.8) for v in rng.uniform(0, 1, 3)) + (0.8,)),
                         (1.0, tuple(float(v * 0.5) for v in rng.uniform(0, 1, 3)) + (0.5,))]
                if (len(t.gpu_buffer_f) % 1024) + 260 > 1024:
                    t.push_gpu_buffer_f([(0, 0, 0, 0)] * ((-len(t.gpu_buffer_f)) % 1024))
                lut = t.push_gpu_buffer_f(list(build_gradient_table(stops)))
                grads.append(prim(local(r), noclip, [(0.0, 0.0, float(r[2] - r[0]), float(r[3] - r[1])),
                                                     (0.0, float(r[2] - r[0]), float(r[3] - r[1]), 0.0)], user=(lut, 0, 0, 0)))
            glyphs = []
            for run in range(2):
                a = float(rng.uniform(0.6, 1.0))
                color = tuple(float(v * a) for v in rng.uniform(0, 0.4, 3)) + (a,)
                bx, by = float(rng.randint(0, tile_w - 500)) + ox, float(rng.randint(20, tile_h - 8)) + oy
                pen, offs, gids = 0.0, [], []
                for g in range(30):
                    gid = int(rng.randint(0, len(glyph_res)))
                    gids.append(gid)
                    offs.append((pen, 0.0))
                    pen += glyph_res[gid][2] + 1.0
                blocks = [color] + [(offs[k][0], offs[k][1], offs[k + 1][0], offs[k + 1][1]) for k in range(0, 30, 2)]
                addr = t.push_gpu_cache(blocks)
                hdr = t.add_prim_header((bx, by, 0.0, 0.0), noclip, z, addr, 0, pic, (65535, 0, 0, 0))
                z += 1
                for g, gid in enumerate(gids):
                    if gid not in glyph_addr:
                        gx, gy, gw, gh = glyph_res[gid]
                        glyph_addr[gid] = t.push_gpu_cache([(float(gx), float(gy), float(gx + gw), float(gy + gh)),
                                                            (0.0, float(-gh), 1.0, 0.0)])
                    glyphs.append(glyph_instance(hdr, CLIP_TASK_EMPTY, 0, 0, g, glyph_addr[gid]))
            PM = abi.BLEND_PREMULTIPLIED_ALPHA
            ops = [Clear(color=(1.0, 1.0, 1.0, 1.0), depth=1.0),
                   Batch(abi.KIND_BRUSH_SOLID, np.stack(osolid[::-1]), blend=abi.BLEND_NONE, depth=abi.DEPTH_TEST_WRITE),
                   Batch(abi.KIND_BRUSH_IMAGE, np.stack(oimg[::-1]), blend=abi.BLEND_NONE, depth=abi.DEPTH_TEST_WRITE,
                         features=abi.FEAT_TEXTURE_2D, color=("atlas", "", "")),
                   Batch(abi.KIND_BRUSH_SOLID, np.stack(asolid), blend=PM, depth=abi.DEPTH_TEST, features=abi.FEAT_ALPHA_PASS,
                         clip_mask="mask"),
                   Batch(abi.KIND_BRUSH_IMAGE, np.stack(aimg), blend=PM, depth=abi.DEPTH_TEST,
                         features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D, color=("atlas", "", "")),
                   Batch(abi.KIND_BRUSH_LINEAR_GRADIENT, np.stack(grads), blend=PM, depth=abi.DEPTH_TEST,
                         features=abi.FEAT_ALPHA_PASS),
                   Batch(abi.KIND_TEXT_RUN, np.stack(glyphs), blend=PM, depth=abi.DEPTH_TEST,
                         features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D, color=("glyphs", "", ""))]
            tile_targets.append(Target(name, depth=dname, ops=ops))
            rect = (ox, oy, ox + tile_w, oy + tile_h)
            clip = (ox, oy, min(ox + tile_w, float(width)), min(oy + tile_h, float(height)))
            comp.append(Batch(abi.KIND_COMPOSITE, composite_instance(rect, clip)[None, :], blend=abi.BLEND_NONE,
                              features=abi.FEAT_FAST_PATH | abi.FEAT_TEXTURE_2D, color=(name, "", "")))
            ti += 1
    # ---- pass 3: the tile list into the framebuffer ---------------------------------------------------------
    textures["fb"] = TextureDesc(abi.FMT_RGBA8, width, height)
    fb = Target("fb", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0))] + comp)
    return Frame(t.arrays(), textures, [[Target("mask", ops=mops)], tile_targets, [fb]])


def perspective_matrix(width, height, d=800.0, ry=35.0, rx=0.0):
    """A CSS-style perspective transform about the page centre: perspective(d) rotateX(rx) rotateY(ry).
    With a small `d` and a steep angle part of the page lies behind the eye (w <= 0): the near-plane
    clipping of draw_perspective (rasterize.h:1467-1521)."""
    cx, cy = width / 2.0, height / 2.0
    t1 = np.eye(4)
    t1[0, 3], t1[1, 3] = -cx, -cy
    a, b = np.deg2rad(ry), np.deg2rad(rx)
    rym = np.array([[np.cos(a), 0, np.sin(a), 0], [0, 1, 0, 0], [-np.sin(a), 0, np.cos(a), 0], [0, 0, 0, 1]])
    rxm = np.array([[1, 0, 0, 0], [0, np.cos(b), -np.sin(b), 0], [0, np.sin(b), np.cos(b), 0], [0, 0, 0, 1]])
    pm = np.eye(4)
    pm[3, 2] = -1.0 / d
    t2 = np.eye(4)
    t2[0, 3], t2[1, 3] = cx, cy
    return (t2 @ pm @ rxm @ rym @ t1).astype(np.float32)


def with_transform(make_frame, matrix, **kw):
    """Build one of the `rotate=` scenes with an arbitrary 4x4 (e.g. perspective_matrix) in place of the rotation."""
    global rotation_matrix
    saved = rotation_matrix
    rotation_matrix = lambda *a, **k: matrix  # noqa: E731
    try:
        return make_frame(rotate=0.0, **kw)
    finally:
        rotation_matrix = saved


def perspective_frame(kind="solid", width=640, height=360, d=800.0, ry=35.0, rx=0.0, **kw):
    """Brush batches under a perspective spatial node (w differs between the vertices: draw_perspective,
    rasterize.h:1422-1545): kind = "solid" (brush_solid_frame: opaque + alpha with masks / AA) or "image"
    (image_frame: opaque + alpha pass sampling an atlas)."""
    m = perspective_matrix(width, height, d, ry, rx)
    make = {"solid": brush_solid_frame, "image": image_frame, "quad": rounded_rects_frame, "opacity": opacity_frame,
            "blend": blend_frame, "mix_blend": mix_blend_frame}[kind]
    return with_transform(make, m, width=width, height=height, **kw)


def split_composite_frame(width=640, height=360, n_polys=10, seed=1, d=600.0, ry=40.0, rx=-15.0,
                          perspective_interpolate=0, with_masks=True, filter=abi.LINEAR):
    """BatchKind::SplitComposite (batch.rs:74, 2040-2080): the polygons a plane-split preserve-3d picture is cut
    into, each drawn by ps_split_composite from the picture's surface with premultiplied blending under the
    depth test, behind a few opaque Brush(Solid) prims.  Polygon points are in the picture's local space; the
    prim header carries the picture rect and its (perspective) transform, user_data = [ImageSource address,
    perspective_interpolate, 0, clip task]; the ImageSource has the UvRectKind::Quad corner block."""
    from webrender_b200.gpu_types import brush_instance, split_composite_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    sw, sh = 256, 192
    surf = rng.randint(0, 256, size=(sh, sw, 4)).astype(np.uint8)
    al = surf[..., 3:4].astype(np.uint16)
    surf[..., :3] = (surf[..., :3].astype(np.uint16) * al // 255).astype(np.uint8)
    mw, mh = 256, 256
    mask = rng.randint(0, 256, size=(mh, mw)).astype(np.uint8)
    xf = t.add_transform(perspective_matrix(width, height, d, ry, rx), axis_aligned=False)
    # opaque solids in front (larger z), some under the same transform
    opaque = []
    z = 5000
    for i in range(4):
        r = _rand_rect(rng, width, height, 30, 160)
        c = tuple(float(v) for v in rng.uniform(0, 1, 3)) + (1.0,)
        addr = t.push_gpu_cache([c])
        hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), z, addr, xf if i % 2 else 0, pic, (65535, 0, 0, 0))
        z += 1
        opaque.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
    polys = []
    z = 1
    for i in range(n_polys):
        # the picture: a local rect, its surface region, and a convex quad inside it
        r = _rand_rect(rng, width, height, 60, 300)
        rw, rh = r[2] - r[0], r[3] - r[1]
        uw, uh = int(rng.randint(20, 200)), int(rng.randint(20, 150))
        u0, v0 = int(rng.randint(0, sw - uw)), int(rng.randint(0, sh - uh))
        j = lambda s: float(rng.uniform(0.0, 0.3) * s)  # noqa: E731
        pts = [(r[0] + j(rw), r[1] + j(rh)), (r[2] - j(rw), r[1] + j(rh)), (r[2] - j(rw), r[3] - j(rh)), (r[0] + j(rw), r[3] - j(rh))]
        poly_addr = t.push_gpu_cache([(pts[0][0], pts[0][1], pts[1][0], pts[1][1]), (pts[2][0], pts[2][1], pts[3][0], pts[3][1])])
        k = float(rng.uniform(0.8, 1.25))
        res = t.push_gpu_cache([(float(u0), float(v0), float(u0 + uw), float(v0 + uh)), (0.0, 0.0, 0.0, 0.0),
                                (0.0, 0.0, 0.0, 1.0), (k, 0.0, 0.0, k), (0.0, 1.0, 0.0, 1.0), (1.0, 1.0, 0.0, 1.0)])
        clip_task = CLIP_TASK_EMPTY
        if with_masks and i % 3 == 1:
            w_, h_ = 100, 80
            mx, my = int(rng.randint(0, mw - w_)), int(rng.randint(0, mh - h_))
            sx, sy = int(rng.randint(0, width - w_)), int(rng.randint(0, height - h_))
            clip_task = t.add_render_task((float(mx), float(my), float(mx + w_), float(my + h_)), 1.0, (float(sx), float(sy)))
        hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), z, 0, xf, pic, (res, perspective_interpolate, 0, clip_task))
        polys.append(split_composite_instance(hdr, poly_addr, z, pic))
        z += 1
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "depth": TextureDesc(abi.FMT_DEPTH24, width, height),
                "surface": TextureDesc(abi.FMT_RGBA8, sw, sh, surf.reshape(sh, sw * 4), filter=filter),
                "mask": TextureDesc(abi.FMT_R8, mw, mh, mask)}
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0), depth=1.0),
           Batch(abi.KIND_BRUSH_SOLID, np.stack(opaque[::-1]), blend=abi.BLEND_NONE, depth=abi.DEPTH_TEST_WRITE),
           Batch(abi.KIND_SPLIT_COMPOSITE, np.stack(polys), blend=abi.BLEND_PREMULTIPLIED_ALPHA, depth=abi.DEPTH_TEST,
                 color=("surface", "", ""), clip_mask="mask")]
    return Frame(t.arrays(), textures, [[Target("target", depth="depth", ops=ops)]])


def image_repeat_frame(width=640, height=360, n_opaque=6, n_alpha=14, seed=1, filter=abi.LINEAR, fractional=False,
                       device_pixel_scale=1.0, occlude_alpha=False):
    """Tiled images and border-image segments: Brush(Image) with BatchFeatures::REPETITION
    (shade.rs:985-1000 "ANTIALIASING,REPETITION"): stretch sizes smaller than the primitive
    (background-repeat), segment-relative REPEAT_X / REPEAT_Y with ROUND and CENTERED flags and
    texel-rect nine-patch middles (border-image-repeat), small (few-texel) tiles and 1:1 tiles."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), device_pixel_scale, (0.0, 0.0))
    aw, ah = 256, 192
    atlas = rng.randint(0, 256, size=(ah, aw, 4)).astype(np.uint8)
    a = atlas[..., 3:4].astype(np.uint16)
    atlas[..., :3] = (atlas[..., :3].astype(np.uint16) * a // 255).astype(np.uint8)
    z = 1
    opaque, alpha = [], []

    def add(rect, uv, color, color_mode, opacity, flags=0, segment=None, stretch=(-1.0, -1.0)):
        nonlocal z
        blocks = [color, (0.0, 0.0, 0.0, 0.0), (stretch[0], stretch[1], 0.0, 0.0)]
        seg_index = 0xFFFF
        if segment is not None:
            blocks += [segment[0], segment[1]]
            seg_index = 0
        addr = t.push_gpu_cache(blocks)
        res = t.push_gpu_cache([uv, (0.0, 0.0, 0.0, 0.0)])
        hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), z, addr, 0, pic,
                                (color_mode | (1 << 16), 0, int(opacity * 65535), 0))
        z += 1
        return brush_instance(hdr, CLIP_TASK_EMPTY, seg_index, 0, flags, res)

    def tile_uv(i):
        if i % 5 == 4:
            uw, uh = int(rng.randint(1, 4)), int(rng.randint(1, 4))       # a few texels: the solid-span test
        else:
            uw, uh = int(rng.randint(8, 64)), int(rng.randint(8, 48))
        u0, v0 = int(rng.randint(0, aw - uw)), int(rng.randint(0, ah - uh))
        return (float(u0), float(v0), float(u0 + uw), float(v0 + uh)), uw, uh

    lw, lh = int(width / device_pixel_scale), int(height / device_pixel_scale)
    if occlude_alpha:
        z = 10000
    for i in range(n_opaque):
        r = _rand_rect(rng, lw, lh, 40, 260, integer=not fractional)
        uv, uw, uh = tile_uv(i)
        st = (float(uw), float(uh)) if i % 2 == 0 else (float(rng.uniform(6, 70)), float(rng.uniform(6, 50)))
        opaque.append(add(r, uv, (1.0, 1.0, 1.0, 1.0), 4, 1.0, stretch=st))
    if occlude_alpha:
        z = 1
    for i in range(n_alpha):
        r = _rand_rect(rng, lw, lh, 40, 260, integer=not fractional)
        uv, uw, uh = tile_uv(i)
        mode = [4, 4, 3, 0, 4][i % 5]
        col = (1.0, 1.0, 1.0, 1.0) if i % 3 == 0 else tuple(float(v) for v in rng.uniform(0.2, 1.0, 4))
        rw, rh = r[2] - r[0], r[3] - r[1]
        k = i % 4
        if k == 0:      # plain tiling by stretch size
            alpha.append(add(r, uv, col, mode, rng.uniform(0.5, 1.0),
                             stretch=(float(rng.uniform(7, 80)), float(rng.uniform(7, 60)))))
        elif k == 1:    # segment-relative, repeat both axes with explicit sizes, rounded
            seg = ((float(int(rw / 5)), float(int(rh / 5)), float(int(rw * 4 / 5)), float(int(rh * 4 / 5))),
                   (0.0, 0.0, float(rng.uniform(9, 40)), float(rng.uniform(9, 30))))
            alpha.append(add(r, uv, col, mode, rng.uniform(0.5, 1.0), flags=2 | 4 | 8 | 16 | 32, segment=seg))
        elif k == 2:    # nine-patch middle with texel rect, repeat x centred
            seg = ((float(int(rw / 4)), float(int(rh / 4)), float(int(rw * 3 / 4)), float(int(rh * 3 / 4))),
                   (0.25, 0.25, 0.75, 0.75))
            alpha.append(add(r, uv, col, mode, rng.uniform(0.5, 1.0), flags=2 | 512 | 256 | 4 | 64, segment=seg))
        else:           # edge segment with texel rect, repeat y centred + rounded
            seg = ((0.0, float(int(rh / 4)), float(int(rw / 4)), float(int(rh * 3 / 4))), (0.0, 0.25, 0.25, 0.75))
            alpha.append(add(r, uv, col, mode, rng.uniform(0.5, 1.0), flags=2 | 512 | 8 | 32 | 128, segment=seg))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "depth": TextureDesc(abi.FMT_DEPTH24, width, height),
                "atlas": TextureDesc(abi.FMT_RGBA8, aw, ah, atlas.reshape(ah, aw * 4), filter=filter)}
    feats = abi.FEAT_TEXTURE_2D | abi.FEAT_REPETITION | abi.FEAT_ANTIALIASING
    ops = [Clear(color=(0.2, 0.3, 0.4, 1.0), depth=1.0)]
    if opaque:
        ops.append(Batch(abi.KIND_BRUSH_IMAGE, np.stack(opaque[::-1]), blend=abi.BLEND_NONE, depth=abi.DEPTH_TEST_WRITE,
                         features=feats, color=("atlas", "", "")))
    if alpha:
        ops.append(Batch(abi.KIND_BRUSH_IMAGE, np.stack(alpha), blend=abi.BLEND_PREMULTIPLIED_ALPHA, depth=abi.DEPTH_TEST,
                         features=feats | abi.FEAT_ALPHA_PASS, color=("atlas", "", "")))
    return Frame(t.arrays(), textures, [[Target("target", depth="depth", ops=ops)]])


def text_frame(width=960, height=540, n_runs=12, glyphs_per_run=40, seed=2, atlas_size=512, atlas="r8",
               device_pixel_scale=1.0, fractional=False, color_modes=(0,), with_masks=False, glyph_transform=None,
               clip_runs=False):
    """Config C flavour (wrench/benchmarks/text-rendering.yaml): text runs as
    TextRun(Alpha) glyph instances blitting from a glyph atlas.  The atlas is
    synthetic (seeded coverage cells, w,h in [4,16]) — glyph rasterisation is
    FreeType's job upstream and out of scope; the blit is what is under test.
    glyph_transform = (degrees, sx, sy): runs under a rotated / scaled 2-D transform drawn with
    BatchFeatures::GLYPH_TRANSFORM (glyphs rasterised in the transformed space, quads trimmed to the
    glyph rect by gl_ClipDistance); clip_runs gives every other run a local clip rect that cuts
    through its glyphs (the non-"inside" branch of ps_text_run.glsl:160-167)."""
    from webrender_b200.gpu_types import glyph_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), device_pixel_scale, (0.0, 0.0))
    xf = 0
    if glyph_transform is not None:
        deg, gsx, gsy = glyph_transform
        xf = t.add_transform(rotation_matrix(deg, width / (2.0 * device_pixel_scale), height / (2.0 * device_pixel_scale),
                                             gsx, gsy), axis_aligned=(deg == 0))
    # atlas: grid of 16x16 cells each holding one glyph of random size
    cells = atlas_size // 16
    bpp = 1 if atlas == "r8" else 4
    tex = np.zeros((atlas_size, atlas_size, bpp), dtype=np.uint8)
    glyph_res = []
    for gy in range(cells):
        for gx in range(cells):
            gw, gh = int(rng.randint(4, 17)), int(rng.randint(4, 17))
            cov = rng.randint(0, 256, size=(gh, gw, bpp)).astype(np.uint8)
            if bpp == 4:
                a = cov[..., 3:4].astype(np.uint16)
                cov[..., :3] = (cov[..., :3].astype(np.uint16) * a // 255).astype(np.uint8)
            tex[gy * 16: gy * 16 + gh, gx * 16: gx * 16 + gw] = cov
            glyph_res.append((gx * 16, gy * 16, gw, gh))
    res_addr = {}
    inst_by_mode = {}
    z = 1
    mask = None
    mw = mh = 256
    if with_masks:
        mask = rng.randint(0, 256, size=(mh, mw)).astype(np.uint8)
    for r in range(n_runs):
        color_mode = color_modes[r % len(color_modes)]
        a = rng.uniform(0.5, 1.0)
        color = tuple(float(v * a) for v in rng.uniform(0, 1, 3)) + (float(a),)
        base_x, base_y = float(rng.randint(0, width - 100)), float(rng.randint(16, height - 16))
        if fractional:
            base_x += float(rng.uniform(0, 1)); base_y += float(rng.uniform(0, 1))
        offsets = []
        pen = 0.0
        gids = []
        for g in range(glyphs_per_run):
            gid = int(rng.randint(0, len(glyph_res)))
            gids.append(gid)
            offsets.append((pen + (float(rng.uniform(0, 1)) if fractional else 0.0), 0.0))
            pen += glyph_res[gid][2] + 1.0
        blocks = [color]
        for k in range(0, len(offsets), 2):
            o0 = offsets[k]
            o1 = offsets[k + 1] if k + 1 < len(offsets) else (0.0, 0.0)
            blocks.append((o0[0], o0[1], o1[0], o1[1]))
        addr = t.push_gpu_cache(blocks)
        s = 1.0 / device_pixel_scale
        # local_rect.p0 = run origin (added to glyph offsets), local_rect.p1 = text_offset (batch.rs:1109-1340)
        lclip = (-1e9, -1e9, 1e9, 1e9)
        if clip_runs and r % 2 == 1:
            lclip = (base_x * s + 7.3, base_y * s - 9.6, base_x * s + pen * 0.6, base_y * s - 2.2)
        hdr = t.add_prim_header((base_x * s, base_y * s, 0.0, 0.0), lclip, z, addr, xf, pic,
                                (65535, 0, 0, 0))
        z += 1
        clip_task = CLIP_TASK_EMPTY
        if with_masks and r % 2 == 0:
            mx, my = int(rng.randint(0, mw - 200)), int(rng.randint(0, mh - 40))
            clip_task = t.add_render_task((float(mx), float(my), float(mx + 200), float(my + 40)), 1.0,
                                          (float(int(base_x)), float(int(base_y) - 12)))
        for g, gid in enumerate(gids):
            if gid not in res_addr:
                gx, gy, gw, gh = glyph_res[gid]
                # GlyphResource: uv_rect (px), offset.xy, scale (ps_text_run.glsl:56-65)
                res_addr[gid] = t.push_gpu_cache([(float(gx), float(gy), float(gx + gw), float(gy + gh)),
                                                  (0.0, float(-gh), 1.0, 0.0)])
            inst_by_mode.setdefault(color_mode, []).append(
                glyph_instance(hdr, clip_task, 0, color_mode, g, res_addr[gid]))
    fmt = abi.FMT_R8 if atlas == "r8" else abi.FMT_RGBA8
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "atlas": TextureDesc(fmt, atlas_size, atlas_size, tex.reshape(atlas_size, atlas_size * bpp))}
    if mask is not None:
        textures["mask"] = TextureDesc(abi.FMT_R8, mw, mh, mask)
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0))]
    for mode, lst in sorted(inst_by_mode.items()):
        ops.append(Batch(abi.KIND_TEXT_RUN, np.stack(lst), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                         features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D |
                         (abi.FEAT_GLYPH_TRANSFORM if glyph_transform is not None else 0), color=("atlas", "", ""),
                         clip_mask="mask" if mask is not None else ""))
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def gradient_frame(width=640, height=360, n_grad=6, seed=1, fractional=False, full_frame=False, repeat=False,
                   blend=abi.BLEND_NONE, rotate=None):
    """Config D flavour (wrench/benchmarks/aligned-gradient.yaml / unaligned-gradient.yaml):
    Brush(LinearGradient) instances; under is_software non-tiled linear gradients
    stay uncached brushes (scene_building.rs:3392-3396).  Each has its own
    130-entry two-colour LUT in gpu_buffer_f."""
    from webrender_b200.gpu_types import brush_instance, build_gradient_table, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    inst = []
    gxf = 0
    if rotate is not None:
        gxf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0), axis_aligned=False)
    for i in range(n_grad):
        if full_frame:
            r = (0.0, 0.0, float(width), float(height))
            start, end = (0.0, -2000.0), (float(i % 2), 4000.0)   # aligned / unaligned-gradient.yaml
            stops = [(0.0, (1.0, 0.0, 0.0, 1.0)), (1.0, (0.0, 1.0, 0.0, 1.0))]
        else:
            r = _rand_rect(rng, width, height, 24, 400, integer=not fractional)
            start = (float(rng.uniform(-20, 60)), float(rng.uniform(-20, 60)))
            end = (float(rng.uniform(80, 300)), float(rng.uniform(-50, 200)))
            ns = int(rng.randint(2, 5))
            offs = [0.0] + sorted(float(v) for v in rng.uniform(0.05, 0.95, ns - 2)) + [1.0]
            stops = []
            for o in offs:
                a = float(rng.uniform(0.3, 1.0)) if blend != abi.BLEND_NONE else 1.0
                stops.append((o, tuple(float(v * a) for v in rng.uniform(0, 1, 3)) + (a,)))
        # keep the 260-texel table inside one 1024-texel row (swgl_validateGradient)
        pad = (-len(t.gpu_buffer_f)) % 1024
        if (len(t.gpu_buffer_f) % 1024) + 260 > 1024:
            t.push_gpu_buffer_f([(0, 0, 0, 0)] * pad)
        lut = t.push_gpu_buffer_f(list(build_gradient_table(stops)))
        rw, rh = r[2] - r[0], r[3] - r[1]
        stretch = (rw, rh) if not repeat else (rw / 2.5, rh / 1.5)
        addr = t.push_gpu_cache([(start[0], start[1], end[0], end[1]),
                                 (1.0 if (repeat and i % 2) else 0.0, stretch[0], stretch[1], 0.0)])
        hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), i + 1, addr, gxf, pic, (lut, 0, 0, 0))
        inst.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    feats = abi.FEAT_ALPHA_PASS if blend != abi.BLEND_NONE else 0
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0)),
           Batch(abi.KIND_BRUSH_LINEAR_GRADIENT, np.stack(inst), blend=blend, features=feats)]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def _random_stops(rng, premultiplied_alpha=True, hard=False):
    ns = int(rng.randint(2, 6))
    offs = [0.0] + sorted(float(v) for v in rng.uniform(0.05, 0.95, ns - 2)) + [1.0]
    if hard and ns >= 4:
        offs[2] = offs[1]   # a hard stop
    stops = []
    for o in offs:
        a = float(rng.uniform(0.3, 1.0)) if premultiplied_alpha else 1.0
        stops.append((o, tuple(float(v * a) for v in rng.uniform(0, 1, 3)) + (a,)))
    return stops


def cached_gradient_frame(kind, width=1024, height=512, n_tasks=6, seed=1, repeat=False, hard=False,
                          big=None):
    """Gradient render tasks the way draw_texture_cache_target draws them
    (renderer/mod.rs:4085-4183): blending off, one instance per cached task rect
    in a texture-cache RGBA8 target.  kind = KIND_{FAST_LINEAR,LINEAR,RADIAL,CONIC}_GRADIENT.
    Parameters follow the task builders in prim_store/gradient/{linear,radial,conic}.rs:
    points/radii in task-local device pixels, `scale` = prim size / task size."""
    from webrender_b200 import gpu_types as G
    rng = np.random.RandomState(seed)
    t = FrameTables()
    inst = []
    x_cursor, y_cursor, row_h = 3, 2, 0
    for i in range(n_tasks):
        if big:
            w, h = big
            x0, y0 = 0, 0
        else:
            w, h = int(rng.randint(17, 330)), int(rng.randint(9, 200))
            if x_cursor + w > width - 2:
                x_cursor, y_cursor, row_h = 3, y_cursor + row_h + 3, 0
            x0, y0 = x_cursor, y_cursor
            x_cursor += w + 5
            row_h = max(row_h, h)
        rect = (float(x0), float(y0), float(x0 + w), float(y0 + h))
        sc = (float(rng.uniform(1.0, 2.5)), float(rng.uniform(1.0, 2.5))) if i % 3 else (1.0, 1.0)
        pw, ph = w * sc[0], h * sc[1]
        ext = 1 if (repeat or (i % 4 == 3)) else 0
        if kind == abi.KIND_FAST_LINEAR_GRADIENT:
            c0 = tuple(float(v) for v in rng.uniform(0, 1, 4))
            c1 = tuple(float(v) for v in rng.uniform(0, 1, 4))
            inst.append(G.fast_linear_gradient_instance(rect, c0, c1, float(i % 2)))
            continue
        if (len(t.gpu_buffer_f) % 1024) + 260 > 1024:
            t.push_gpu_buffer_f([(0, 0, 0, 0)] * ((-len(t.gpu_buffer_f)) % 1024))
        lut = t.push_gpu_buffer_f(list(G.build_gradient_table(_random_stops(rng, True, hard))))
        if kind == abi.KIND_LINEAR_GRADIENT:
            start = (float(rng.uniform(-0.2, 0.6) * pw), float(rng.uniform(-0.2, 0.6) * ph))
            end = (float(rng.uniform(0.3, 1.2) * pw), float(rng.uniform(-0.3, 1.2) * ph))
            if i % 5 == 4:
                end = (start[0], end[1] + 1.0)       # vertical: constant offset along a row
            if ext:
                end = (start[0] + (end[0] - start[0]) * 0.3, start[1] + (end[1] - start[1]) * 0.3)
            inst.append(G.linear_gradient_instance(rect, start, end, sc, ext, lut))
        elif kind == abi.KIND_RADIAL_GRADIENT:
            center = (float(rng.uniform(-0.1, 1.1) * pw), float(rng.uniform(-0.1, 1.1) * ph))
            r0 = float(rng.uniform(0, 0.2) * pw) if i % 2 else 0.0
            r1 = r0 + float(rng.uniform(0.1, 0.9) * pw) * (0.3 if ext else 1.0)
            ratio = float(rng.uniform(0.5, 2.0)) if i % 3 == 1 else 1.0
            inst.append(G.radial_gradient_instance(rect, center, sc, r0, r1, ratio, ext, lut))
        else:
            center = (float(rng.uniform(0.1, 0.9) * pw), float(rng.uniform(0.1, 0.9) * ph))
            so = float(rng.uniform(0.0, 0.3)) if i % 2 else 0.0
            eo = so + (float(rng.uniform(0.2, 0.5)) if ext else 1.0 - so)
            ang = float(rng.uniform(0, 2 * np.pi)) if i % 3 else 0.0
            inst.append(G.conic_gradient_instance(rect, center, sc, so, eo, ang, ext, lut))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    ops = [Clear(color=(0.0, 0.0, 0.0, 0.0)), Batch(kind, np.stack(inst), blend=abi.BLEND_NONE)]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


class _ShelfPacker:
    """Places render-task rects in a texture-cache target, shelf by shelf."""

    def __init__(self, width, height, pad=2):
        self.w, self.h, self.pad = width, height, pad
        self.x, self.y, self.row_h = pad, pad, 0

    def place(self, w, h):
        if self.x + w > self.w - self.pad:
            self.x, self.y, self.row_h = self.pad, self.y + self.row_h + self.pad, 0
        if self.y + h > self.h - self.pad:
            return None
        x0, y0 = self.x, self.y
        self.x += w + self.pad
        self.row_h = max(self.row_h, h)
        return x0, y0


def line_decoration_frame(width=512, height=256, n_tasks=24, seed=1):
    """cs_line_decoration tasks (renderer/mod.rs:4059-4083): premultiplied-alpha
    blending on, one LineDecorationJob per cached tile: solid / dotted / dashed /
    wavy, horizontal and vertical, at device scales 1, 1.5 and 2 (the task rect is
    the local size times the device scale, so the AA range varies)."""
    from webrender_b200 import gpu_types as G
    rng = np.random.RandomState(seed)
    pack = _ShelfPacker(width, height)
    inst = []
    for i in range(n_tasks):
        style = i % 4
        vertical = (i // 4) % 2
        t = float(rng.choice([1.0, 1.5, 2.0, 3.0, 5.0, 8.0]))
        scale = float(rng.choice([1.0, 1.5, 2.0]))
        if style == 2:      # dashed: period x thickness
            size = (6.0 * t, t)
        elif style == 1:    # dotted: two diameters x diameter
            size = (2.0 * t, t)
        elif style == 3:    # wavy
            lt = max(t, 1.0)
            h = float(np.ceil(lt * 3.0 + rng.randint(0, 4)))
            slope, flat = h - lt, max((lt - 1.0) * 2.0, 1.0)
            size = (2.0 * (slope + flat), h)
        else:
            size = (float(rng.randint(8, 40)), t)
        if vertical:
            size = (size[1], size[0])
        tw, th = int(np.ceil(size[0] * scale)), int(np.ceil(size[1] * scale))
        at = pack.place(tw, th)
        if at is None:
            break
        rect = (float(at[0]), float(at[1]), float(at[0] + tw), float(at[1] + th))
        inst.append(G.line_decoration_instance(rect, size, t, style, float(vertical)))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    ops = [Clear(color=(0.0, 0.0, 0.0, 0.0)),
           Batch(abi.KIND_LINE_DECORATION, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA)]
    return Frame(FrameTables().arrays(), textures, [[Target("target", ops=ops)]])


def wrench_checkerboard(border, tile, count):
    """wrench's `checkerboard(border, tile size, tile count)` image (yaml_frame_reader.rs:195-240, BlackGrey kind):
    BGRA bytes, a `border`-pixel frame of (0, 0, 255, 255) around 0xff / 0x7f squares."""
    n = 2 * border + tile * count
    yy, xx = np.mgrid[0:n, 0:n]
    inner = (xx >= border) & (xx < n - border) & (yy >= border) & (yy < n - border)
    xon = ((xx - border) % (2 * tile)) < tile
    yon = ((yy - border) % (2 * tile)) < tile
    v = np.where(xon ^ yon, 0xFF, 0x7F).astype(np.uint8)
    img = np.zeros((n, n, 4), dtype=np.uint8)
    img[..., 0] = np.where(inner, v, 0)
    img[..., 1] = np.where(inner, v, 0)
    img[..., 2] = np.where(inner, v, 0xFF)
    img[..., 3] = 0xFF
    return img.reshape(n, n * 4)


def reftest_image_segments_frame():
    """wrench/reftests/image/segments.yaml (== segments.png, fuzzy-if(platform(swgl),1,20)): a 260x260 checkerboard image
    drawn 1:1 twice — at (10,10) under a rounded clip of radius 32, at (10,290) unclipped.  The frame builder segments
    the clipped image and masks only its corners; the pixels are those of the whole image under the clip's coverage
    mask, which is how it is drawn here: cs_clip_rectangle into an R8 mask task, then Brush(Image) alpha pass with the
    mask; the second image is an opaque Brush(Image).  Reference image 290x583."""
    from webrender_b200.gpu_types import brush_instance, clip_rect_instance, CLIP_TASK_EMPTY
    W, H = 290, 583
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    rect = (10.0, 10.0, 270.0, 270.0)
    mask_task = t.add_render_task((0.0, 0.0, 260.0, 260.0), 1.0, (10.0, 10.0))
    clip = clip_rect_instance((0.0, 0.0, 260.0, 260.0), (0.0, 0.0), (10.0, 10.0), 1.0, 0, 0, (rect[0], rect[1]), rect, 0.0,
                              ((32.0, 32.0),) * 4)
    uv = t.push_gpu_cache([(0.0, 0.0, 260.0, 260.0), (0.0, 0.0, 0.0, 0.0)])
    blocks = [(1.0, 1.0, 1.0, 1.0), (0.0, 0.0, 0.0, 0.0), (-1.0, -1.0, 0.0, 0.0)]
    h1 = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), 2, t.push_gpu_cache(blocks), 0, pic, (4 | (1 << 16), 0, 65535, 0))
    h2 = t.add_prim_header((10.0, 290.0, 270.0, 550.0), (-1e9, -1e9, 1e9, 1e9), 1, t.push_gpu_cache(blocks), 0, pic,
                           (4 | (1 << 16), 0, 65535, 0))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H),
                "mask": TextureDesc(abi.FMT_R8, 512, 512),
                "image": TextureDesc(abi.FMT_RGBA8, 260, 260, data=wrench_checkerboard(2, 16, 16), filter=abi.LINEAR)}
    p0 = [Target("mask", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                              Batch(abi.KIND_CLIP_RECTANGLE, clip[None, :], blend=abi.BLEND_NONE, features=abi.FEAT_FAST_PATH)])]
    p1 = [Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                                Batch(abi.KIND_BRUSH_IMAGE, brush_instance(h2, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, uv)[None, :],
                                      blend=abi.BLEND_NONE, features=abi.FEAT_TEXTURE_2D, color=("image", "", "")),
                                Batch(abi.KIND_BRUSH_IMAGE, brush_instance(h1, mask_task, 0xFFFF, 0, 0, uv)[None, :],
                                      blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D,
                                      color=("image", "", ""), clip_mask="mask")])]
    return Frame(t.arrays(), textures, [p0, p1])


def reftest_gradient_border_radius_frame(repeat=False):
    """wrench/reftests/gradient/linear-aligned-border-radius.yaml (== linear-aligned-border-radius.png on GL; `repeat`
    sets the extend mode of repeat-border-radius.yaml's first row): three 100x100 vertical red -> yellow gradients under a rounded
    clip of radius 32 — on the white page, on a blue and on a black 120x120 rect.  Brush(LinearGradient) in the alpha
    pass with a cs_clip_rectangle mask each (the uncached brush path an `is_software` frame builder keeps).
    Reference images 395x151."""
    from webrender_b200.gpu_types import brush_instance, build_gradient_table, clip_rect_instance, CLIP_TASK_EMPTY
    W, H = 395, 151
    red, yellow = (1.0, 0.0, 0.0, 1.0), (1.0, 1.0, 0.0, 1.0)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    lut = t.push_gpu_buffer_f(list(build_gradient_table([(0.0, red), (1.0, yellow)])))
    solids, grads, clips = [], [], []
    z = 1
    for i, (x, bg) in enumerate(((20, None), (140, (0.0, 0.0, 1.0, 1.0)), (270, (0.0, 0.0, 0.0, 1.0)))):
        if bg is not None:
            addr = t.push_gpu_cache([bg])
            hdr = t.add_prim_header((float(x - 10), 10.0, float(x + 110), 130.0), (-1e9, -1e9, 1e9, 1e9), z, addr, 0, pic, (65535, 0, 0, 0))
            z += 1
            solids.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
        rect = (float(x), 20.0, float(x + 100), 120.0)
        mask_task = t.add_render_task((float(128 * i), 0.0, float(128 * i + 100), 100.0), 1.0, (rect[0], rect[1]))
        clips.append(clip_rect_instance((0.0, 0.0, 100.0, 100.0), (float(128 * i), 0.0), (rect[0], rect[1]), 1.0, 0, 0,
                                        (rect[0], rect[1]), rect, 0.0, ((32.0, 32.0),) * 4))
        # gradient brush data: start / end points relative to the prim, extend mode, stretch size
        addr = t.push_gpu_cache([(50.0, 0.0, 50.0, 100.0), (1.0 if repeat else 0.0, 100.0, 100.0, 0.0)])
        hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), z, addr, 0, pic, (lut, 0, 0, 0))
        z += 1
        grads.append(brush_instance(hdr, mask_task, 0xFFFF, 0, 0, 0))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H), "mask": TextureDesc(abi.FMT_R8, 512, 128)}
    p0 = [Target("mask", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                              Batch(abi.KIND_CLIP_RECTANGLE, np.stack(clips), blend=abi.BLEND_NONE, features=abi.FEAT_FAST_PATH)])]
    p1 = [Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                                Batch(abi.KIND_BRUSH_SOLID, np.stack(solids), blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS),
                                Batch(abi.KIND_BRUSH_LINEAR_GRADIENT, np.stack(grads), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                      features=abi.FEAT_ALPHA_PASS, clip_mask="mask")])]
    return Frame(t.arrays(), textures, [p0, p1])


def composited_through_tile(frame, tile=(1024, 1024)):
    """A single-target frame drawn the way the compositor path draws a page: "target" becomes a picture-cache tile (a
    power-of-two texture, same content, same render task) and an extra pass composites it into the framebuffer "fb" of
    the page's size — clear, one opaque FAST_PATH tile instance clipped to the page (composite_simple / draw_tile_list,
    renderer/mod.rs:3126-3484).  The tile maps 1:1, so it takes the copy class on the GPU (§4.7 of DESIGN.md)."""
    from webrender_b200.gpu_types import composite_instance
    d = frame.textures["target"]
    W, H = d.width, d.height
    textures = dict(frame.textures)
    textures["target"] = TextureDesc(d.fmt, tile[0], tile[1], filter=abi.NEAREST)
    textures["fb"] = TextureDesc(abi.FMT_RGBA8, W, H)
    inst = composite_instance((0.0, 0.0, float(tile[0]), float(tile[1])), (0.0, 0.0, float(W), float(H)))
    fb = Target("fb", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0)),
                           Batch(abi.KIND_COMPOSITE, inst[None, :], blend=abi.BLEND_NONE,
                                 features=abi.FEAT_FAST_PATH | abi.FEAT_TEXTURE_2D, color=("target", "", ""))])
    return Frame(frame.tables, textures, list(frame.passes) + [[fb]])


def reftest_box_shadow_suite_composited_frame():
    """reftest_box_shadow_suite_no_blur_frame through a picture-cache tile and the composite pass."""
    return composited_through_tile(reftest_box_shadow_suite_no_blur_frame())


def reftest_line_decorations_frame():
    """The first eight items of wrench/reftests/text/decorations-suite.yaml (rows 0-99 of decorations-suite.png; the
    reftest allows SWGL 3 on 13 540 pixels over the whole suite): horizontal lines 200 long, 1 / 2 / 3 / 6 thick —
    solid (black), dashed (blue), dotted (green), wavy (red).  Draw list (scene_building.rs add_line, prim_store/
    line_dec.rs:195-241 get_line_decoration_size, prepare.rs:345-425, batch.rs:1338-1420): a solid line is a
    Brush(Solid) rect; the others are a cs_line_decoration task of ceil(size) — dashed (2 * min(3h, 64), 4), dotted
    (2h, h), wavy (2 * (h - t + max(2(t - 1), 1)), h) — in the texture cache, repeated along the line by Brush(Image)
    REPETITION with the stretch size = the task's local size and the line colour, premultiplied blending."""
    from webrender_b200 import gpu_types as G
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    W, H = 495, 439
    black, blue, green, red = (0.0, 0.0, 0.0, 1.0), (0.0, 0.0, 1.0, 1.0), (0.0, 1.0, 0.0, 1.0), (1.0, 0.0, 0.0, 1.0)
    lines = [(10, 10, 210, 1, 0, black, 0.0), (20, 10, 210, 1, 2, blue, 0.0), (30, 10, 210, 1, 1, green, 0.0),
             (40, 10, 210, 3, 3, red, 1.0), (50, 10, 210, 2, 0, black, 0.0), (65, 10, 210, 2, 2, blue, 0.0),
             (80, 10, 207, 2, 1, green, 0.0), (95, 10, 210, 6, 3, red, 2.0)]   # style: 0 solid, 1 dotted, 2 dashed, 3 wavy
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    pack = _ShelfPacker(256, 64)
    tasks, solids, images = [], [], []
    for i, (base, x0, x1, h, style, col, thick) in enumerate(lines):
        rect = (float(x0), float(base), float(x1), float(base + h))
        if style == 0:
            addr = t.push_gpu_cache([col])
            hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), i + 1, addr, 0, pic, (65535, 0, 0, 0))
            solids.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
            continue
        hf = float(h)
        if style == 2:
            size = (2.0 * max(min(3.0 * hf, 64.0), 1.0), 4.0)
        elif style == 1:
            d = max(min(hf, 64.0), 1.0)
            size = (2.0 * d, d)
        else:
            lt = max(thick, 1.0)
            size = (2.0 * ((hf - lt) + max((lt - 1.0) * 2.0, 1.0)), hf)
        tw, th = int(np.ceil(size[0])), int(np.ceil(size[1]))
        at = pack.place(tw, th)
        trect = (float(at[0]), float(at[1]), float(at[0] + tw), float(at[1] + th))
        tasks.append(G.line_decoration_instance(trect, size, thick, style, 0.0))
        addr = t.push_gpu_cache([col, (1.0, 1.0, 1.0, 1.0), (size[0], size[1], 0.0, 0.0)])
        res = t.push_gpu_cache([trect, (0.0, 0.0, 0.0, 0.0)])
        hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), i + 1, addr, 0, pic, (4 | (1 << 16), 0, 65535, 0))
        images.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, res))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H),
                "cache": TextureDesc(abi.FMT_RGBA8, 256, 64, filter=abi.LINEAR)}
    p0 = [Target("cache", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0)),
                               Batch(abi.KIND_LINE_DECORATION, np.stack(tasks), blend=abi.BLEND_PREMULTIPLIED_ALPHA)])]
    p1 = [Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                                Batch(abi.KIND_BRUSH_SOLID, np.stack(solids), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                      features=abi.FEAT_ALPHA_PASS),
                                Batch(abi.KIND_BRUSH_IMAGE, np.stack(images), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                      features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D | abi.FEAT_REPETITION | abi.FEAT_ANTIALIASING,
                                      color=("cache", "", ""))])]
    return Frame(t.arrays(), textures, [p0, p1])


def _ellipse_point_tangent(rx, ry, theta):
    c, s = float(np.cos(theta)), float(np.sin(theta))
    return (rx * c, ry * s), (-rx * s, ry * c)


def border_frame(kind, width=1024, height=512, n_borders=6, seed=1, scale=1.0):
    """Border render tasks (renderer/mod.rs:4015-4057): premultiplied-alpha blending
    on; per border four corner tasks and four edge tasks as border.rs:904-1243
    builds them (task-local rects, adjacent-corner clips, dash/dot clip
    parameters).  kind = KIND_BORDER_SOLID (solid styles, optional AA) or
    KIND_BORDER_SEGMENT (double/dotted/dashed/groove/ridge/inset/outset).
    Dash and dot positions along a corner use uniform ellipse angles where the
    reference solves for arc length (the frame builder is outside this path)."""
    from webrender_b200 import gpu_types as G
    rng = np.random.RandomState(seed)
    pack = _ShelfPacker(width, height)
    inst = []
    f32 = np.float32
    solid = kind == abi.KIND_BORDER_SOLID
    styles = [G.BORDER_STYLE_DOUBLE, G.BORDER_STYLE_DOTTED, G.BORDER_STYLE_DASHED, G.BORDER_STYLE_GROOVE,
              G.BORDER_STYLE_RIDGE, G.BORDER_STYLE_INSET, G.BORDER_STYLE_OUTSET]

    def rcolor(black=False):
        a = float(rng.uniform(0.4, 1.0))
        rgb = (0.0, 0.0, 0.0) if black else tuple(float(v) for v in rng.uniform(0, 1, 3))
        return tuple(float(f32(c * a)) for c in rgb) + (a,)

    for b in range(n_borders):
        wl, wt, wr, wb = [float(f32(rng.choice([1.0, 2.0, 3.0, 4.5, 6.0, 9.0, 14.0]) * scale)) for _ in range(4)]
        box_w, box_h = float(rng.randint(120, 260)) * scale, float(rng.randint(90, 200)) * scale
        radii = {}
        for c in range(4):
            if b % 3 == 2:
                radii[c] = (0.0, 0.0)
            else:
                radii[c] = (float(f32(rng.uniform(4, 50) * scale)), float(f32(rng.uniform(4, 50) * scale)))
        do_aa = bool(b % 4 != 3) if solid else True
        if solid:
            st = [G.BORDER_STYLE_SOLID] * 4            # left, top, right, bottom
        else:
            st = [int(styles[(b + k * (1 if b % 2 else 0)) % len(styles)]) for k in range(4)]
        col = [rcolor(black=(not solid and b % 5 == 4 and k == 0)) for k in range(4)]
        side_w = [wl, wt, wr, wb]
        # corner: (segment, side0 = horizontal-adjacent edge index, side1, widths (x, y), radius)
        corners = [(G.SEGMENT_TOP_LEFT, 0, 1, (wl, wt), radii[0]), (G.SEGMENT_TOP_RIGHT, 1, 2, (wr, wt), radii[1]),
                   (G.SEGMENT_BOTTOM_RIGHT, 2, 3, (wr, wb), radii[2]), (G.SEGMENT_BOTTOM_LEFT, 3, 0, (wl, wb), radii[3])]
        corner_size = {}
        for seg, s0, s1, wd, rad in corners:
            corner_size[seg] = (max(rad[0], wd[0]), max(rad[1], wd[1]))
        # outer corner points of the box, per corner segment
        outer_pt = {0: (0.0, 0.0), 1: (box_w, 0.0), 2: (box_w, box_h), 3: (0.0, box_h)}
        corner_org = {0: (0.0, 0.0), 1: (box_w - corner_size[1][0], 0.0),
                      2: (box_w - corner_size[2][0], box_h - corner_size[2][1]), 3: (0.0, box_h - corner_size[3][1])}
        h_adj = {0: 1, 1: 0, 2: 3, 3: 2}
        v_adj = {0: 3, 1: 2, 2: 1, 3: 0}
        for seg, s0, s1, wd, rad in corners:
            cw, ch = corner_size[seg]
            tw, th = int(np.ceil(cw)), int(np.ceil(ch))
            at = pack.place(tw, th)
            if at is None:
                continue
            org = corner_org[seg]
            rect = (0.0, 0.0, float(f32(cw)), float(f32(ch)))
            base = dict(task_origin=(float(at[0]), float(at[1])), local_rect=rect, color0=col[s0], color1=col[s1],
                        segment=seg, style0=st[s0], style1=st[s1], do_aa=do_aa, widths=wd, radius=rad)
            hseg, vseg = h_adj[seg], v_adj[seg]
            adj = (outer_pt[hseg][0] - org[0], outer_pt[hseg][1] - org[1]) + radii[hseg] + \
                  (outer_pt[vseg][0] - org[0], outer_pt[vseg][1] - org[1]) + radii[vseg]
            adj = tuple(float(f32(v)) for v in adj)
            os_ = {0: (0.0, 0.0), 1: (1.0, 0.0), 2: (1.0, 1.0), 3: (0.0, 1.0)}[seg]
            outer = (os_[0] * rad[0], os_[1] * rad[1])
            sign = (1.0 - 2.0 * os_[0], 1.0 - 2.0 * os_[1])
            if not solid and st[s0] == G.BORDER_STYLE_DASHED and rad[0] > 0 and rad[1] > 0:
                n_dash = 3
                for k in range(n_dash):
                    th0 = (np.pi / 2) * (2 * k) / (2 * n_dash - 1) if k else 0.0
                    th0 = (np.pi / 2) * max(0.0, (2 * k - 0.5)) / (2 * n_dash - 1)
                    th1 = (np.pi / 2) * (2 * k + 1.0) / (2 * n_dash - 1)
                    pts = []
                    for th_ in (th0, th1):
                        p, t = _ellipse_point_tangent(rad[0], rad[1], th_)
                        pts += [outer[0] + sign[0] * (rad[0] - p[0]), outer[1] + sign[1] * (rad[1] - p[1]),
                                -t[0] * sign[0], -t[1] * sign[1]]
                    inst.append(G.border_instance(clip_kind=G.BORDER_CLIP_DASH_CORNER,
                                                  clip_params=tuple(float(f32(v)) for v in pts), **base))
            elif not solid and st[s0] == G.BORDER_STYLE_DOTTED:
                if rad[0] < wd[0] / 2 or rad[1] < wd[1] / 2:
                    dd = 0.5 * (wd[0] + wd[1])
                    inst.append(G.border_instance(clip_kind=G.BORDER_CLIP_DOT,
                                                  clip_params=(wd[0] / 2, wd[1] / 2, 0.5 * dd, 0, 0, 0, 0, 0), **base))
                else:
                    irx, iry = abs(rad[0] - wd[0] * 0.5), abs(rad[1] - wd[1] * 0.5)
                    n_dot = 4
                    for k in range(n_dot):
                        th_ = (np.pi / 2) * k / (n_dot - 1)
                        p, _ = _ellipse_point_tangent(irx, iry, th_)
                        cx = outer[0] + sign[0] * (rad[0] - p[0])
                        cy = outer[1] + sign[1] * (rad[1] - p[1])
                        dia = wd[0] + (wd[1] - wd[0]) * k / (n_dot - 1)
                        inst.append(G.border_instance(clip_kind=G.BORDER_CLIP_DOT,
                                                      clip_params=(float(f32(cx)), float(f32(cy)), float(f32(0.5 * dia)),
                                                                   0, 0, 0, 0, 0), **base))
            else:
                inst.append(G.border_instance(clip_params=adj, **base))
        # edges: (segment, side index, vertical)
        for seg, side, vertical in ((G.SEGMENT_LEFT, 0, True), (G.SEGMENT_TOP, 1, False),
                                    (G.SEGMENT_RIGHT, 2, True), (G.SEGMENT_BOTTOM, 3, False)):
            wdt = side_w[side]
            style = st[side]
            if style == G.BORDER_STYLE_DASHED:
                length = 6.0 * wdt          # task = one dash period (border.rs get_edge_info)
            elif style == G.BORDER_STYLE_DOTTED:
                length = 2.0 * wdt
            else:
                length = 8.0
            size = (wdt, length) if vertical else (length, wdt)
            tw, th = int(np.ceil(size[0])), int(np.ceil(size[1]))
            at = pack.place(tw, th)
            if at is None:
                continue
            rect = (0.0, 0.0, float(f32(size[0])), float(f32(size[1])))
            base = dict(task_origin=(float(at[0]), float(at[1])), local_rect=rect, color0=col[side], color1=col[side],
                        segment=seg, style0=style, style1=style, do_aa=do_aa, widths=(wdt, wdt), radius=(0.0, 0.0))
            if not solid and style == G.BORDER_STYLE_DASHED:
                half = (size[1] if vertical else size[0]) * 0.25
                cp = (0.0, half) if vertical else (half, 0.0)
                inst.append(G.border_instance(clip_kind=G.BORDER_CLIP_DASH_EDGE, clip_params=cp + (0,) * 6, **base))
            elif not solid and style == G.BORDER_STYLE_DOTTED:
                cp = (wdt * 0.5, wdt, wdt * 0.5) if vertical else (wdt, wdt * 0.5, wdt * 0.5)
                inst.append(G.border_instance(clip_kind=G.BORDER_CLIP_DOT, clip_params=cp + (0,) * 5, **base))
            else:
                inst.append(G.border_instance(**base))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    ops = [Clear(color=(0.0, 0.0, 0.0, 0.0)), Batch(kind, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA)]
    return Frame(FrameTables().arrays(), textures, [[Target("target", ops=ops)]])


def texture_cache_frame(seed=1, width=1024, height=1024):
    """One texture-cache target carrying every task list draw_texture_cache_target
    walks (renderer/mod.rs:3931-4200), in its order: clears, solid borders, complex
    borders, line decorations (premultiplied-alpha blending), then fast-linear and
    radial gradients (blending off).  Built from the per-kind scenes, each moved to
    its own band of the target."""
    bands = [(abi.KIND_BORDER_SOLID, border_frame(abi.KIND_BORDER_SOLID, width=width, height=300, n_borders=3, seed=seed), 0),
             (abi.KIND_BORDER_SEGMENT, border_frame(abi.KIND_BORDER_SEGMENT, width=width, height=300, n_borders=4,
                                                    seed=seed + 1, scale=1.5), 300),
             (abi.KIND_LINE_DECORATION, line_decoration_frame(width=width, height=100, n_tasks=16, seed=seed), 600),
             (abi.KIND_FAST_LINEAR_GRADIENT, cached_gradient_frame(abi.KIND_FAST_LINEAR_GRADIENT, width=width, height=150,
                                                                    n_tasks=4, seed=seed), 700),
             (abi.KIND_RADIAL_GRADIENT, cached_gradient_frame(abi.KIND_RADIAL_GRADIENT, width=width, height=170,
                                                               n_tasks=4, seed=seed), 850)]
    ops = [Clear(color=(0.0, 0.0, 0.0, 0.0))]
    tables = None
    for kind, f, dy in bands:
        b = [op for op in f.passes[0][0].ops if isinstance(op, Batch)][0]
        rows = np.ascontiguousarray(b.instance_bytes()).copy()
        fl = rows.view(np.float32)
        if kind in (abi.KIND_BORDER_SOLID, abi.KIND_BORDER_SEGMENT):
            fl[:, 1] += dy                    # task_origin.y
        else:
            fl[:, 1] += dy                    # task_rect.y0 / y1
            fl[:, 3] += dy
        keep = fl[:, 3] <= height if kind not in (abi.KIND_BORDER_SOLID, abi.KIND_BORDER_SEGMENT) else np.ones(len(fl), bool)
        ops.append(Batch(kind, rows[keep], blend=b.blend))
        if kind == abi.KIND_RADIAL_GRADIENT:
            tables = f.tables
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    return Frame(tables, textures, [[Target("target", ops=ops)]])


def quad_gradient_frame(kind, width=640, height=360, n_quads=8, seed=1, fractional=False, blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                        rotate=None, device_pixel_scale=1.0):
    """Quad(RadialGradient) / Quad(ConicGradient) primitives through the quad path
    (prim_store/gradient/{radial,conic}.rs `write_prim_gpu_blocks` → ps_quad_*_gradient):
    pattern_input = (gradient parameter blocks, stops LUT) in gpu_buffer_f."""
    from webrender_b200 import gpu_types as G
    rng = np.random.RandomState(seed)
    t = FrameTables()
    task = t.add_render_task((0.0, 0.0, float(width), float(height)), device_pixel_scale, (0.0, 0.0))
    xf = 0
    if rotate is not None:
        xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0), axis_aligned=False)
    inst = []
    for i in range(n_quads):
        r = _rand_rect(rng, int(width / device_pixel_scale), int(height / device_pixel_scale), 24, 300,
                       integer=not fractional)
        rw, rh = r[2] - r[0], r[3] - r[1]
        ext = 1.0 if i % 3 == 2 else 0.0
        if (len(t.gpu_buffer_f) % 1024) + 260 > 1024:
            t.push_gpu_buffer_f([(0, 0, 0, 0)] * ((-len(t.gpu_buffer_f)) % 1024))
        lut = t.push_gpu_buffer_f(list(G.build_gradient_table(_random_stops(rng, True, hard=(i % 4 == 3)))))
        sc = (1.0, 1.0) if i % 2 == 0 else (float(rng.uniform(0.5, 2.0)), float(rng.uniform(0.5, 2.0)))
        center = (float(rng.uniform(0.1, 0.9) * rw * sc[0]), float(rng.uniform(0.1, 0.9) * rh * sc[1]))
        if kind == abi.KIND_QUAD_RADIAL_GRADIENT:
            r0 = float(rng.uniform(0, 0.2) * rw) if i % 2 else 0.0
            r1 = r0 + float(rng.uniform(0.15, 0.9) * rw) * (0.35 if ext else 1.0)
            ratio = float(rng.uniform(0.5, 2.0)) if i % 3 == 1 else 1.0
            params = t.push_gpu_buffer_f([center + sc, (r0, r1, ratio, ext)])
        else:
            so = float(rng.uniform(0.0, 0.3)) if i % 2 else 0.0
            eo = so + (float(rng.uniform(0.2, 0.5)) if ext else 1.0 - so)
            ang = float(rng.uniform(0, 2 * np.pi)) if i % 3 else 0.0
            params = t.push_gpu_buffer_f([center + sc, (so, eo, ang, ext)])
        a = float(rng.uniform(0.4, 1.0)) if i % 2 else 1.0
        prim_f = t.add_quad_prim(r, r, (a, a, a, a))
        prim_i = t.add_quad_header(xf, i + 1, pattern_input=(params, lut))
        inst.append(quad_instance(prim_i, prim_f, QF_APPLY_DEVICE_CLIP, 0, PART_ALL, INVALID_SEGMENT_INDEX, task))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0)), Batch(kind, np.stack(inst), blend=blend)]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def reftest_cached_gradient_frame(which="premultiplied-radial"):
    """wrench/reftests/gradient/premultiplied-radial.yaml, premultiplied-conic.yaml and
    conic-center.yaml the way the frame builder draws them (prim_store/gradient/{radial,conic}.rs):
    pass 0 renders the gradient as a cached 200x200 render task (cs_radial_gradient /
    cs_conic_gradient, task size = stretch size, scale 1) into a texture-cache target; pass 1
    composites the task 1:1 with Brush(Image) (premultiplied-alpha blend, white colour) onto
    the white 300x300 page at (50,50)."""
    from webrender_b200 import gpu_types as G
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    W = H = 300
    red, green, blue, black = (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0), (0.0, 0.0, 1.0, 1.0), (0.0, 0.0, 0.0, 1.0)
    clear = (0.0, 0.0, 0.0, 0.0)
    t = FrameTables()
    task_rect = (0.0, 0.0, 200.0, 200.0)
    if which == "conic-center":
        stops = [(0.0, red), (0.25, red), (0.25, green), (0.5, green), (0.5, blue), (0.75, blue), (0.75, black), (1.0, black)]
        center = (50.0, 50.0)
    else:
        stops = [(0.0, red), (0.5, clear), (1.0, green)]
        center = (100.0, 100.0)
    lut = t.push_gpu_buffer_f(list(G.build_gradient_table(stops)))
    if which == "premultiplied-radial":
        kind = abi.KIND_RADIAL_GRADIENT
        inst = G.radial_gradient_instance(task_rect, center, (1.0, 1.0), 0.0, 100.0, 1.0, 0, lut)
    else:
        kind = abi.KIND_CONIC_GRADIENT
        inst = G.conic_gradient_instance(task_rect, center, (1.0, 1.0), 0.0, 1.0, 0.0, 0, lut)
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    addr = t.push_gpu_cache([(1.0, 1.0, 1.0, 1.0), (1.0, 1.0, 1.0, 1.0), (200.0, 200.0, 0.0, 0.0)])
    res = t.push_gpu_cache([task_rect, (0.0, 0.0, 0.0, 0.0)])
    hdr = t.add_prim_header((50.0, 50.0, 250.0, 250.0), (-1e9, -1e9, 1e9, 1e9), 1, addr, 0, pic,
                            (4 | (1 << 16), 0, 65535, 0))
    img = np.stack([brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, res)])
    textures = {"cache": TextureDesc(abi.FMT_RGBA8, 256, 256, filter=abi.LINEAR),
                "target": TextureDesc(abi.FMT_RGBA8, W, H)}
    opaque = which == "conic-center"
    p0 = Target("cache", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0)), Batch(kind, np.stack([inst]), blend=abi.BLEND_NONE)])
    p1 = Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                               Batch(abi.KIND_BRUSH_IMAGE, img,
                                     blend=abi.BLEND_NONE if opaque else abi.BLEND_PREMULTIPLIED_ALPHA,
                                     features=abi.FEAT_TEXTURE_2D | (0 if opaque else abi.FEAT_ALPHA_PASS),
                                     color=("cache", "", ""))])
    return Frame(t.arrays(), textures, [[p0], [p1]])


CACHED_GRADIENT_REFTESTS = {
    # wrench/reftests/gradient/<name>.yaml against its reference image, drawn as a cached gradient task + Brush(Image)
    # like reftest_cached_gradient_frame: (image size, bounds x y w h, kind, centre, radius (rx, ry) | angle, stops with
    # 0-255 colours + alpha, allowed (max diff, pixels))
    "radial-circle": ((400, 400), (50, 50, 300, 300), "radial", (150, 150), (200, 200),
                      [(0.0, (255, 0, 0, 1.0)), (1.0, (0, 0, 255, 1.0))], (1, 80000)),
    "radial-ellipse": ((400, 400), (50, 50, 300, 300), "radial", (150, 150), (100, 200),
                       [(0.0, (255, 0, 0, 1.0)), (1.0, (0, 0, 255, 1.0))], (1, 80000)),
    "conic-simple": ((400, 400), (50, 50, 300, 300), "conic", (150, 150), 0.0,
                     [(0.0, (255, 0, 0, 1.0)), (1.0, (255, 255, 0, 1.0))], (1, 300)),
}


def reftest_cached_gradient_frame2(name):
    """One of CACHED_GRADIENT_REFTESTS: the gradient as a cached render task of its own size (cs_radial_gradient /
    cs_conic_gradient; prim_store/gradient/{radial,conic}.rs: start radius 0, end radius rx, ratio_xy = rx / ry), then
    Brush(Image) 1:1 onto the white page, premultiplied blending."""
    from webrender_b200 import gpu_types as G
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    (W, H), (bx, by, bw, bh), kind, center, param, stops, _ = CACHED_GRADIENT_REFTESTS[name]
    t = FrameTables()
    task_rect = (0.0, 0.0, float(bw), float(bh))
    pm = [(o, (c[0] / 255.0 * c[3], c[1] / 255.0 * c[3], c[2] / 255.0 * c[3], c[3])) for o, c in stops]
    lut = t.push_gpu_buffer_f(list(G.build_gradient_table(pm)))
    if kind == "radial":
        rx, ry = param
        inst = G.radial_gradient_instance(task_rect, (float(center[0]), float(center[1])), (1.0, 1.0), 0.0, float(rx),
                                          float(rx) / float(ry), 0, lut)
        k = abi.KIND_RADIAL_GRADIENT
    else:
        inst = G.conic_gradient_instance(task_rect, (float(center[0]), float(center[1])), (1.0, 1.0), 0.0, 1.0, float(param), 0, lut)
        k = abi.KIND_CONIC_GRADIENT
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    addr = t.push_gpu_cache([(1.0, 1.0, 1.0, 1.0), (1.0, 1.0, 1.0, 1.0), (float(bw), float(bh), 0.0, 0.0)])
    res = t.push_gpu_cache([task_rect, (0.0, 0.0, 0.0, 0.0)])
    hdr = t.add_prim_header((float(bx), float(by), float(bx + bw), float(by + bh)), (-1e9, -1e9, 1e9, 1e9), 1, addr, 0, pic,
                            (4 | (1 << 16), 0, 65535, 0))
    img = np.stack([brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, res)])
    textures = {"cache": TextureDesc(abi.FMT_RGBA8, 512, 512, filter=abi.LINEAR),
                "target": TextureDesc(abi.FMT_RGBA8, W, H)}
    p0 = Target("cache", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0)), Batch(k, np.stack([inst]), blend=abi.BLEND_NONE)])
    p1 = Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                               Batch(abi.KIND_BRUSH_IMAGE, img, blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                     features=abi.FEAT_TEXTURE_2D | abi.FEAT_ALPHA_PASS, color=("cache", "", ""))])
    return Frame(t.arrays(), textures, [[p0], [p1]])


def shadow_mask_texture(size=256, seed=5):
    """A seeded stand-in for the blurred box-shadow masks cs_blur produces
    (render_task.rs BlurTask): soft-edged blobs plus a little noise, R8."""
    rng = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:size, 0:size].astype(np.float64)
    img = np.zeros((size, size))
    for _ in range(6):
        cx, cy = rng.uniform(0, size, 2)
        sx, sy = rng.uniform(size / 10, size / 3, 2)
        img += np.exp(-(((xx - cx) / sx) ** 2 + ((yy - cy) / sy) ** 2))
    img = img / img.max() * 255.0 + rng.uniform(-6, 6, img.shape)
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def box_shadow_frame(width=512, height=384, n_clips=8, seed=1, fractional=False, scale=1.0, atlas=256,
                     full_size=None):
    """Box-shadow clip masks the way draw_alpha_target issues them
    (renderer/mod.rs:3754-3929, batch.rs:3816-3838): a cs_clip_box_shadow batch
    with blending off for first clips, then one multiplied in.  Each instance
    nine-patches (Stretch) or scales (Simple) a blurred R8 mask into its task
    rect; every other one is ClipOut."""
    from webrender_b200.gpu_types import box_shadow_instance
    rng = np.random.RandomState(seed)
    t = FrameTables()
    xf = t.add_transform(scale_matrix(scale)) if scale != 1.0 else 0
    prim, sec = [], []
    for i in range(n_clips):
        if full_size:
            w, h = full_size
            tx = ty = 0
        else:
            w, h = int(rng.randint(48, 240)), int(rng.randint(40, 200))
            tx, ty = int(rng.randint(0, width - w)), int(rng.randint(0, height - h))
        sx, sy = int(rng.randint(0, 400)), int(rng.randint(0, 400))
        # shadow mask cell inside the atlas
        cw, ch = int(rng.randint(24, 96)), int(rng.randint(24, 96))
        cx, cy = int(rng.randint(0, atlas - cw)), int(rng.randint(0, atlas - ch))
        res = t.push_gpu_cache([(float(cx), float(cy), float(cx + cw), float(cy + ch)), (0.0, 0.0, 0.0, 0.0)])
        # destination rect in local space: a bit inside / outside the task rect
        off = rng.uniform(-10, 30, 4) if fractional else rng.randint(-10, 31, 4).astype(np.float64)
        dest = ((sx + off[0]) / scale, (sy + off[1]) / scale, (sx + w - off[2]) / scale, (sy + h - off[3]) / scale)
        stretch = (int(rng.randint(0, 2)), int(rng.randint(0, 2)))
        src_size = (float(cw) / scale, float(ch) / scale)
        if fractional:
            src_size = (src_size[0] * float(rng.uniform(0.8, 1.3)), src_size[1] * float(rng.uniform(0.8, 1.3)))
        inst = box_shadow_instance((0.0, 0.0, float(w), float(h)), (float(tx), float(ty)), (float(sx), float(sy)),
                                   scale, xf, xf, res, src_size, i % 2, stretch, dest)
        (prim if i < max(1, n_clips * 2 // 3) else sec).append(inst)
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0))]
    for lst, blend in ((prim, abi.BLEND_NONE), (sec, abi.BLEND_MULTIPLY)):
        if lst:
            ops.append(Batch(abi.KIND_CLIP_BOX_SHADOW, np.stack(lst), blend=blend, features=abi.FEAT_TEXTURE_2D,
                             color=("shadow", "", "")))
    textures = {"mask": TextureDesc(abi.FMT_R8, width, height),
                "shadow": TextureDesc(abi.FMT_R8, atlas, atlas, data=shadow_mask_texture(atlas, seed + 10),
                                      filter=abi.LINEAR)}
    return Frame(t.arrays(), textures, [[Target("mask", ops=ops)]])


def tile_texture(w, h, seed, opaque=True):
    """Seeded picture-cache tile content: smooth colour ramps plus noise, BGRA
    premultiplied."""
    rng = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    img = np.zeros((h, w, 4))
    ph = rng.uniform(0, 6.28, 6)
    for ch in range(3):
        img[..., ch] = 0.5 + 0.5 * np.sin(xx / (17.0 + 9 * ch) + ph[ch]) * np.cos(yy / (23.0 - 5 * ch) + ph[3 + ch])
    img[..., :3] += rng.uniform(-0.08, 0.08, (h, w, 3))
    a = np.ones((h, w)) if opaque else np.clip(0.5 + 0.5 * np.sin(xx / 31.0 + yy / 19.0), 0, 1)
    img = np.clip(img, 0, 1)
    img[..., :3] *= a[..., None]
    img[..., 3] = a
    return np.clip(np.rint(img * 255.0), 0, 255).astype(np.uint8).reshape(h, w * 4)


def composite_frame(width=640, height=384, tile_w=256, tile_h=128, seed=1, external=False, fractional=False):
    """composite_simple / draw_tile_list (renderer/mod.rs:3340-3484, 3126-3334):
    the framebuffer is cleared, opaque picture-cache tiles are copied front to
    back with blending off (FAST_PATH program: whole-texture uv, white), clear
    tiles punch holes with premultiplied dest-out, alpha tiles and solid-colour
    tiles (1x1 dummy texture) go over back to front.  `external` adds RGB
    external surfaces: unnormalised uv sub-rects, linear filter, scaling, flips."""
    from webrender_b200.gpu_types import composite_instance
    rng = np.random.RandomState(seed)
    textures = {"fb": TextureDesc(abi.FMT_RGBA8, width, height),
                "dummy": TextureDesc(abi.FMT_RGBA8, 1, 1, data=np.full((1, 4), 255, dtype=np.uint8),
                                     filter=abi.NEAREST)}
    ops = [Clear(color=(0.0, 0.0, 0.0, 0.0))]
    cols, rows = (width + tile_w - 1) // tile_w, (height + tile_h - 1) // tile_h
    jit = (lambda: float(rng.uniform(-0.4, 0.4))) if fractional else (lambda: 0.0)
    ti = 0
    alpha_ops = []
    for ry in range(rows):
        for cx in range(cols):
            name = "tile%d" % ti
            opaque = (ti % 3) != 2
            textures[name] = TextureDesc(abi.FMT_RGBA8, tile_w, tile_h, data=tile_texture(tile_w, tile_h, seed * 100 + ti, opaque),
                                         filter=abi.NEAREST)
            x0, y0 = cx * tile_w + jit(), ry * tile_h + jit()
            rect = (x0, y0, x0 + tile_w, y0 + tile_h)
            clip = (max(rect[0], 0.0) + (float(rng.randint(0, 40)) if ti % 4 == 1 else 0.0), max(rect[1], 0.0),
                    min(rect[2], float(width)), min(rect[3], float(height)) - (float(rng.randint(0, 30)) if ti % 5 == 2 else 0.0))
            inst = composite_instance(rect, clip)
            b = Batch(abi.KIND_COMPOSITE, inst[None, :], blend=abi.BLEND_NONE if opaque else abi.BLEND_PREMULTIPLIED_ALPHA,
                      features=abi.FEAT_FAST_PATH | abi.FEAT_TEXTURE_2D, color=(name, "", ""))
            (ops if opaque else alpha_ops).append(b)
            ti += 1
    # a clear tile (dest-out with black through the dummy texture) and solid colour tiles
    r = _rand_rect(rng, width, height, 40, 200, integer=not fractional)
    ops.append(Batch(abi.KIND_COMPOSITE, composite_instance(r, r, (0.0, 0.0, 0.0, 1.0))[None, :],
                     blend=abi.BLEND_PREMULTIPLIED_DEST_OUT, features=abi.FEAT_TEXTURE_2D, color=("dummy", "", "")))
    ops += alpha_ops
    solid = []
    for i in range(3):
        r = _rand_rect(rng, width, height, 30, 220, integer=not fractional)
        a = float(rng.uniform(0.3, 1.0))
        col = tuple(float(v * a) for v in rng.uniform(0, 1, 3)) + (a,)
        solid.append(composite_instance(r, r, col))
    ops.append(Batch(abi.KIND_COMPOSITE, np.stack(solid), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                     features=abi.FEAT_TEXTURE_2D, color=("dummy", "", "")))
    if external:
        textures["ext"] = TextureDesc(abi.FMT_RGBA8, 320, 200, data=tile_texture(320, 200, seed + 77, False),
                                      filter=abi.LINEAR)
        ext = []
        for i in range(4):
            r = _rand_rect(rng, width, height, 60, 300, integer=not fractional)
            ux, uy = float(rng.randint(0, 100)), float(rng.randint(0, 60))
            if i == 0:
                uw, uh = r[2] - r[0], r[3] - r[1]          # 1:1
                uw, uh = min(uw, 320 - ux), min(uh, 200 - uy)
                r = (r[0], r[1], r[0] + uw, r[1] + uh)
            else:
                uw, uh = float(rng.randint(40, 200)), float(rng.randint(30, 130))
            clip = (r[0] + 3.0, r[1] + 2.0, r[2] - 5.0, r[3] - 1.0)
            ext.append(composite_instance(r, clip, (1.0, 1.0, 1.0, 1.0) if i % 2 == 0 else (0.5, 0.5, 0.5, 0.5),
                                          (ux, uy, ux + uw, uy + uh), normalized=False, flip=(i == 2, i == 3)))
        ops.append(Batch(abi.KIND_COMPOSITE, np.stack(ext), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                         features=abi.FEAT_TEXTURE_2D, color=("ext", "", "")))
    return Frame(FrameTables().arrays(), textures, [[Target("fb", ops=ops)]])


def yuv_planes(w, h, seed, fmt):
    """Seeded 8-bit video frame: full-resolution luma, 4:2:0 chroma (interleaved: one BGRA
    texture holding Cb, Y, Cr in its B, G, R bytes — APPLE_rgb_422 mapping, yuv.glsl:223-229)."""
    rng = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    ph = rng.uniform(0, 6.28, 6)

    def plane(pw, ph_, k, lo, hi):
        y2, x2 = np.mgrid[0:ph_, 0:pw].astype(np.float64)
        v = 0.5 + 0.5 * np.sin(x2 / (11.0 + 7 * k) + ph[k]) * np.cos(y2 / (13.0 + 5 * k) + ph[3 + k])
        v += rng.uniform(-0.06, 0.06, (ph_, pw))
        return np.clip(np.rint(lo + np.clip(v, 0, 1) * (hi - lo)), 0, 255).astype(np.uint8)
    # the full byte range, so out-of-gamut / out-of-range samples exercise the saturating adds
    if fmt == "interleaved":
        y, u, v = plane(w, h, 0, 0, 255), plane(w, h, 1, 0, 255), plane(w, h, 2, 0, 255)
        img = np.stack([u, y, v, np.full_like(y, 255)], axis=2)
        return [img.reshape(h, w * 4)]
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y, u, v = plane(w, h, 0, 0, 255), plane(cw, ch, 1, 0, 255), plane(cw, ch, 2, 0, 255)
    if fmt == "nv12":
        return [y, np.stack([u, v], axis=2).reshape(ch, cw * 2)]
    return [y, u, v]


def yuv_composite_frame(fmt="planar", color_space=2, seed=1, width=512, height=320, linear=True,
                        opaque=True, fractional=False):
    """External YUV video surfaces through `composite` with WR_FEATURE_YUV
    (composite.glsl:14-33, 83-130, 163-176, 197-214; draw_tile_list renderer/mod.rs:3126-3334 with
    CompositeSurfaceFormat::Yuv): 8-bit PLANAR (three R8 planes), NV12 (R8 + RG8) or INTERLEAVED
    (one BGRA plane); 1:1, up- and down-scaled, flipped and clipped surfaces with texel-space uv
    sub-rects, chroma at half resolution."""
    from webrender_b200.gpu_types import (composite_yuv_instance, YUV_FORMAT_PLANAR, YUV_FORMAT_NV12, YUV_FORMAT_INTERLEAVED)
    rng = np.random.RandomState(seed * 31 + color_space)
    vw, vh = 192, 128
    planes = yuv_planes(vw, vh, seed + 5, fmt)
    filt = abi.LINEAR if linear else abi.NEAREST
    textures = {"fb": TextureDesc(abi.FMT_RGBA8, width, height)}
    if fmt == "planar":
        names, yuv_format = ("vy", "vu", "vv"), YUV_FORMAT_PLANAR
        fmts = (abi.FMT_R8, abi.FMT_R8, abi.FMT_R8)
    elif fmt == "nv12":
        names, yuv_format = ("vy", "vuv", ""), YUV_FORMAT_NV12
        fmts = (abi.FMT_R8, abi.FMT_RG8)
    else:
        names, yuv_format = ("vyuv", "", ""), YUV_FORMAT_INTERLEAVED
        fmts = (abi.FMT_RGBA8,)
    for nm, f, pl in zip(names, fmts, planes):
        textures[nm] = TextureDesc(f, pl.shape[1] // abi.FMT_BPP[f], pl.shape[0], data=pl, filter=filt)
    chroma = 1.0 if fmt == "interleaved" else 0.5
    insts = []
    for i in range(6):
        r = _rand_rect(rng, width, height, 40, 260, integer=not fractional)
        ux, uy = float(2 * rng.randint(0, 30)), float(2 * rng.randint(0, 20))
        if i == 0:      # 1:1
            uw, uh = min(r[2] - r[0], vw - ux), min(r[3] - r[1], vh - uy)
            uw, uh = float(int(uw) & ~1), float(int(uh) & ~1)
            r = (r[0], r[1], r[0] + uw, r[1] + uh)
        elif i == 1:    # the whole frame, scaled
            ux, uy, uw, uh = 0.0, 0.0, float(vw), float(vh)
        else:
            uw, uh = float(2 * rng.randint(10, 60)), float(2 * rng.randint(8, 40))
        clip = r if i == 1 else (r[0] + 3.0, r[1] + 2.0, r[2] - 5.0, r[3] - 1.0)
        ry = (ux, uy, ux + uw, uy + uh)
        rc = tuple(v * chroma for v in ry)
        insts.append(composite_yuv_instance(r, clip, color_space, yuv_format, 8, (ry, rc, rc), flip=(i == 3, i == 4)))
    ops = [Clear(color=(0.1, 0.2, 0.3, 1.0)),
           Batch(abi.KIND_COMPOSITE, np.stack(insts), blend=abi.BLEND_NONE if opaque else abi.BLEND_PREMULTIPLIED_ALPHA,
                 features=abi.FEAT_TEXTURE_2D | abi.FEAT_YUV, color=names)]
    return Frame(FrameTables().arrays(), textures, [[Target("fb", ops=ops)]])


def yuv_image_frame(fmt="planar", color_space=2, seed=1, width=512, height=320, linear=True, alpha_pass=True,
                    fractional=False, with_masks=True, rotate=None):
    """Brush(YuvImage) batch (BrushBatchKind::YuvImage, batch.rs:60-86; prim_store/image.rs
    YuvImageData::write_prim_gpu_blocks): video frames drawn as primitives inside a picture — prim data
    [channel_bit_depth, colour space, format, 0], user data = the gpu-cache addresses of the planes'
    ImageSource entries.  Opaque pass (blend off) or alpha pass (premultiplied blend; AA edges, clip
    masks, optionally a rotated spatial node)."""
    from webrender_b200.gpu_types import (brush_instance, CLIP_TASK_EMPTY, YUV_FORMAT_PLANAR, YUV_FORMAT_NV12,
                            YUV_FORMAT_INTERLEAVED)
    rng = np.random.RandomState(seed * 17 + color_space)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    vw, vh = 192, 128
    planes = yuv_planes(vw, vh, seed + 9, fmt)
    filt = abi.LINEAR if linear else abi.NEAREST
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height)}
    if fmt == "planar":
        names, yuv_format, fmts = ("vy", "vu", "vv"), YUV_FORMAT_PLANAR, (abi.FMT_R8,) * 3
    elif fmt == "nv12":
        names, yuv_format, fmts = ("vy", "vuv", ""), YUV_FORMAT_NV12, (abi.FMT_R8, abi.FMT_RG8)
    else:
        names, yuv_format, fmts = ("vyuv", "", ""), YUV_FORMAT_INTERLEAVED, (abi.FMT_RGBA8,)
    for nm, f, pl in zip(names, fmts, planes):
        textures[nm] = TextureDesc(f, pl.shape[1] // abi.FMT_BPP[f], pl.shape[0], data=pl, filter=filt)
    chroma = 1.0 if fmt == "interleaved" else 0.5
    xf = 0
    if rotate is not None:
        xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0, 1.0, 0.9), axis_aligned=False)
    if with_masks and alpha_pass:
        mask = rng.randint(0, 256, size=(256, 256)).astype(np.uint8)
        mask[rng.randint(0, 256, 40)[:, None], :] = 255
        mask[:, rng.randint(0, 256, 40)] = 0
        textures["mask"] = TextureDesc(abi.FMT_R8, 256, 256, data=mask, filter=abi.NEAREST)
    inst = []
    for i in range(7):
        r = _rand_rect(rng, width, height, 40, 240, integer=not fractional)
        ux, uy = float(2 * rng.randint(0, 30)), float(2 * rng.randint(0, 20))
        if i == 0:
            uw, uh = float(int(min(r[2] - r[0], vw - ux)) & ~1), float(int(min(r[3] - r[1], vh - uy)) & ~1)
            r = (r[0], r[1], r[0] + uw, r[1] + uh)
        else:
            uw, uh = float(2 * rng.randint(10, 60)), float(2 * rng.randint(8, 40))
        ry = (ux, uy, ux + uw, uy + uh)
        rc = tuple(v * chroma for v in ry)
        srcs = [t.push_gpu_cache([rr, (0.0, 0.0, 0.0, 0.0)]) for rr in (ry, rc, rc)]
        spec = t.push_gpu_cache([(8.0, float(color_space), float(yuv_format), 0.0)])
        clip = r if i % 3 else (r[0] + 4.0, r[1] + 3.0, r[2] - 6.0, r[3] - 2.0)
        clip_task = CLIP_TASK_EMPTY
        if with_masks and alpha_pass and i % 3 == 1:
            w_, h_ = int(min(r[2] - r[0], 120)), int(min(r[3] - r[1], 100))
            mx, my = int(rng.randint(0, 256 - w_)), int(rng.randint(0, 256 - h_))
            clip_task = t.add_render_task((float(mx), float(my), float(mx + w_), float(my + h_)), 1.0,
                                          (float(int(r[0])), float(int(r[1]))))
        hdr = t.add_prim_header(r, clip, i + 1, spec, xf, pic, (srcs[0], srcs[1], srcs[2], 0))
        edge = 0xF if (alpha_pass and (fractional or rotate is not None)) else 0
        inst.append(brush_instance(hdr, clip_task, 0xFFFF, edge, 0, 0))
    feats = abi.FEAT_TEXTURE_2D | abi.FEAT_YUV | (abi.FEAT_ALPHA_PASS if alpha_pass else 0)
    ops = [Clear(color=(0.2, 0.3, 0.1, 1.0)),
           Batch(abi.KIND_BRUSH_YUV_IMAGE, np.stack(inst),
                 blend=abi.BLEND_PREMULTIPLIED_ALPHA if alpha_pass else abi.BLEND_NONE,
                 features=feats, color=names, clip_mask="mask" if (with_masks and alpha_pass) else "")]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def reftest_yuv_frame(ref_dir):
    """wrench/reftests/image/yuv.yaml the way the frame builder draws it: three `yuv-image` items of 427x640 at
    1:1 — planar (three R8 planes), interleaved (one BGRA image: Cb, Y, Cr in B, G, R) and NV12 with the CbCr
    plane loaded as a BGRA image (wrench turns RGB PNGs into BGRA8: Cb in R, Cr in G — sampleYUV's RGBA8 branch,
    swgl_ext.h:1069-1075) — Color8, Rec709, limited range (yaml_frame_reader.rs:1203-1206), as opaque
    Brush(YuvImage) primitives on the white 1323x658 page.  Reads the reference's own plane PNGs from `ref_dir`
    (wrench/reftests/image of a WebRender checkout)."""
    from PIL import Image
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY, YUV_FORMAT_PLANAR, YUV_FORMAT_NV12, YUV_FORMAT_INTERLEAVED
    import os

    def load(name):
        im = Image.open(os.path.join(ref_dir, name))
        if im.mode == "L":
            return abi.FMT_R8, np.array(im, dtype=np.uint8)
        rgb = np.array(im.convert("RGB"), dtype=np.uint8)
        bgra = np.concatenate([rgb[..., ::-1], np.full(rgb.shape[:2] + (1,), 255, np.uint8)], axis=2)
        return abi.FMT_RGBA8, bgra.reshape(rgb.shape[0], rgb.shape[1] * 4)
    from webrender_b200.gpu_types import composite_instance
    W, H = 1323, 658
    t = FrameTables()
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H)}
    for nm, fn in (("y", "spacex-y.png"), ("u", "spacex-u.png"), ("v", "spacex-v.png"), ("uv", "spacex-uv.png"),
                   ("yuv", "spacex-yuv.png")):
        f, data = load(fn)
        textures[nm] = TextureDesc(f, 427, 640, data=data, filter=abi.LINEAR)
    items = [(10.0, YUV_FORMAT_PLANAR, ("y", "u", "v")), (447.0, YUV_FORMAT_INTERLEAVED, ("yuv", "", "")),
             (887.0, YUV_FORMAT_NV12, ("y", "uv", ""))]
    src = t.push_gpu_cache([(0.0, 0.0, 427.0, 640.0), (0.0, 0.0, 0.0, 0.0)])
    # the page is a picture cache: 1024x512 tiles, each its own target with its own picture task (content origin =
    # the tile's page position), every primitive drawn into every tile it touches — the edge walks restart per tile
    tile_targets, comp = [], []
    for ty in range(2):
        for tx in range(2):
            name = "tile%d%d" % (ty, tx)
            textures[name] = TextureDesc(abi.FMT_RGBA8, 1024, 512)
            pic = t.add_render_task((0.0, 0.0, 1024.0, 512.0), 1.0, (1024.0 * tx, 512.0 * ty))
            ops = [Clear(color=(1.0, 1.0, 1.0, 1.0))]
            for i, (x0, fmt, names) in enumerate(items):
                r = (x0, 10.0, x0 + 427.0, 650.0)
                if r[2] <= 1024.0 * tx or r[0] >= 1024.0 * (tx + 1):
                    continue
                spec = t.push_gpu_cache([(8.0, 2.0, float(fmt), 0.0)])   # Color8, Rec709Narrow
                hdr = t.add_prim_header(r, r, i + 1, spec, 0, pic, (src, src, src, 0))
                inst = brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)
                ops.append(Batch(abi.KIND_BRUSH_YUV_IMAGE, inst[None, :], blend=abi.BLEND_NONE,
                                 features=abi.FEAT_TEXTURE_2D | abi.FEAT_YUV, color=names))
            tile_targets.append(Target(name, ops=ops))
            rect = (1024.0 * tx, 512.0 * ty, 1024.0 * (tx + 1), 512.0 * (ty + 1))
            clip = (rect[0], rect[1], min(rect[2], float(W)), min(rect[3], float(H)))
            comp.append(Batch(abi.KIND_COMPOSITE, composite_instance(rect, clip)[None, :], blend=abi.BLEND_NONE,
                              features=abi.FEAT_FAST_PATH | abi.FEAT_TEXTURE_2D, color=(name, "", "")))
    final = Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0))] + comp)
    return Frame(t.arrays(), textures, [tile_targets, [final]])


def video_frame(width=3840, height=2160, vw=1920, vh=1080, fmt="nv12", color_space=2, seed=1):
    """One full-screen video surface: a vw x vh 8-bit YUV frame (NV12 by default, Rec.709 narrow
    range) scaled to the whole framebuffer by `composite` YUV — the compositor's video case."""
    from webrender_b200.gpu_types import (composite_yuv_instance, YUV_FORMAT_PLANAR, YUV_FORMAT_NV12, YUV_FORMAT_INTERLEAVED)
    planes = yuv_planes(vw, vh, seed, fmt)
    names = {"planar": ("vy", "vu", "vv"), "nv12": ("vy", "vuv", ""), "interleaved": ("vyuv", "", "")}[fmt]
    fmts = {"planar": (abi.FMT_R8,) * 3, "nv12": (abi.FMT_R8, abi.FMT_RG8), "interleaved": (abi.FMT_RGBA8,)}[fmt]
    yuv_format = {"planar": YUV_FORMAT_PLANAR, "nv12": YUV_FORMAT_NV12, "interleaved": YUV_FORMAT_INTERLEAVED}[fmt]
    textures = {"fb": TextureDesc(abi.FMT_RGBA8, width, height)}
    for nm, f, pl in zip(names, fmts, planes):
        textures[nm] = TextureDesc(f, pl.shape[1] // abi.FMT_BPP[f], pl.shape[0], data=pl, filter=abi.LINEAR)
    r = (0.0, 0.0, float(width), float(height))
    ry = (0.0, 0.0, float(vw), float(vh))
    ch = 1.0 if fmt == "interleaved" else 0.5
    rc = tuple(v * ch for v in ry)
    inst = composite_yuv_instance(r, r, color_space, yuv_format, 8, (ry, rc, rc))
    ops = [Clear(color=(0.0, 0.0, 0.0, 1.0)),
           Batch(abi.KIND_COMPOSITE, inst[None, :], blend=abi.BLEND_NONE,
                 features=abi.FEAT_TEXTURE_2D | abi.FEAT_YUV, color=names)]
    return Frame(FrameTables().arrays(), textures, [[Target("fb", ops=ops)]])


HDR_YUV_FORMATS = ("planar", "nv12", "p010")


def hdr_yuv_planes(w, h, seed, fmt, depth):
    """Seeded 10-, 12- or 16-bit video frame as 16-bit little-endian planes (uint8 rows): full-resolution luma,
    4:2:0 chroma.  "planar": three R16 planes; "nv12": R16 + RG16 (CbCr interleaved); both LSB-aligned (codes
    0 .. 2^depth - 1).  "p010": R16 + RG16 MSB-aligned (code << (16 - depth)), as P010 decoders write it."""
    rng = np.random.RandomState(seed)
    ph = rng.uniform(0, 6.28, 6)
    top = (1 << depth) - 1

    def plane(pw, ph_, k):
        y2, x2 = np.mgrid[0:ph_, 0:pw].astype(np.float64)
        v = 0.5 + 0.5 * np.sin(x2 / (11.0 + 7 * k) + ph[k]) * np.cos(y2 / (13.0 + 5 * k) + ph[3 + k])
        v += rng.uniform(-0.06, 0.06, (ph_, pw))
        # the full code range, so out-of-range samples exercise the saturating adds
        return np.rint(np.clip(v, 0, 1) * top).astype(np.uint16)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    y, u, v = plane(w, h, 0), plane(cw, ch, 1), plane(cw, ch, 2)
    if fmt == "p010":
        y, u, v = (p << (16 - depth) for p in (y, u, v))
    rows = lambda p: p.view(np.uint8).reshape(p.shape[0], -1)  # noqa: E731
    if fmt == "planar":
        return [rows(y), rows(u), rows(v)]
    return [rows(y), rows(np.ascontiguousarray(np.stack([u, v], axis=2)))]


def _hdr_yuv_textures(fmt, vw, vh, seed, depth, filt):
    """(plane names, YuvFormat, {name: TextureDesc}) of an hdr_yuv_planes frame"""
    from webrender_b200.gpu_types import YUV_FORMAT_PLANAR, YUV_FORMAT_NV12, YUV_FORMAT_P010
    planes = hdr_yuv_planes(vw, vh, seed, fmt, depth)
    if fmt == "planar":
        names, yuv_format, fmts = ("vy", "vu", "vv"), YUV_FORMAT_PLANAR, (abi.FMT_R16,) * 3
    else:
        names, yuv_format = ("vy", "vuv", ""), YUV_FORMAT_P010 if fmt == "p010" else YUV_FORMAT_NV12
        fmts = (abi.FMT_R16, abi.FMT_RG16)
    textures = {nm: TextureDesc(f, pl.shape[1] // abi.FMT_BPP[f], pl.shape[0], data=pl, filter=filt)
                for nm, f, pl in zip(names, fmts, planes)}
    return names, yuv_format, textures


def hdr_yuv_composite_frame(fmt="p010", depth=10, color_space=2, seed=1, width=512, height=320, linear=True,
                            opaque=True, fractional=False, right_edge=False):
    """yuv_composite_frame's surfaces (1:1, whole frame scaled, sub-rects; flips and clips) from a 10-, 12- or
    16-bit frame: PLANAR (three R16 planes), NV12 or P010 (R16 + RG16).  right_edge: every uv rect ends at the
    planes' last texel column, where the 16-bit fetches weight the last texel by 127/128."""
    from webrender_b200.gpu_types import composite_yuv_instance
    rng = np.random.RandomState(seed * 37 + color_space + 100 * depth)
    vw, vh = 192, 128
    names, yuv_format, textures = _hdr_yuv_textures(fmt, vw, vh, seed + 5, depth, abi.LINEAR if linear else abi.NEAREST)
    textures["fb"] = TextureDesc(abi.FMT_RGBA8, width, height)
    insts = []
    for i in range(6):
        r = _rand_rect(rng, width, height, 40, 260, integer=not fractional)
        ux, uy = float(2 * rng.randint(0, 30)), float(2 * rng.randint(0, 20))
        if i == 0:      # 1:1
            uw, uh = min(r[2] - r[0], vw - ux), min(r[3] - r[1], vh - uy)
            uw, uh = float(int(uw) & ~1), float(int(uh) & ~1)
            r = (r[0], r[1], r[0] + uw, r[1] + uh)
        elif i == 1:    # the whole frame, scaled
            ux, uy, uw, uh = 0.0, 0.0, float(vw), float(vh)
        else:
            uw, uh = float(2 * rng.randint(10, 60)), float(2 * rng.randint(8, 40))
        if right_edge:
            ux = float(vw) - uw
        clip = r if i == 1 else (r[0] + 3.0, r[1] + 2.0, r[2] - 5.0, r[3] - 1.0)
        ry = (ux, uy, ux + uw, uy + uh)
        rc = tuple(v * 0.5 for v in ry)
        insts.append(composite_yuv_instance(r, clip, color_space, yuv_format, depth, (ry, rc, rc), flip=(i == 3, i == 4)))
    ops = [Clear(color=(0.1, 0.2, 0.3, 1.0)),
           Batch(abi.KIND_COMPOSITE, np.stack(insts), blend=abi.BLEND_NONE if opaque else abi.BLEND_PREMULTIPLIED_ALPHA,
                 features=abi.FEAT_TEXTURE_2D | abi.FEAT_YUV, color=names)]
    return Frame(FrameTables().arrays(), textures, [[Target("fb", ops=ops)]])


def hdr_yuv_image_frame(fmt="p010", depth=10, color_space=2, seed=1, width=512, height=320, linear=True,
                        alpha_pass=True, fractional=False, with_masks=True, rotate=None):
    """yuv_image_frame's Brush(YuvImage) primitives (opaque or alpha pass; AA edges, clip masks, a rotated node)
    drawing a 10-, 12- or 16-bit frame: prim data [channel_bit_depth, colour space, format, 0]."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed * 41 + color_space + 100 * depth)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    vw, vh = 192, 128
    names, yuv_format, textures = _hdr_yuv_textures(fmt, vw, vh, seed + 9, depth, abi.LINEAR if linear else abi.NEAREST)
    textures["target"] = TextureDesc(abi.FMT_RGBA8, width, height)
    xf = 0
    if rotate is not None:
        xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0, 1.0, 0.9), axis_aligned=False)
    if with_masks and alpha_pass:
        mask = rng.randint(0, 256, size=(256, 256)).astype(np.uint8)
        mask[rng.randint(0, 256, 40)[:, None], :] = 255
        mask[:, rng.randint(0, 256, 40)] = 0
        textures["mask"] = TextureDesc(abi.FMT_R8, 256, 256, data=mask, filter=abi.NEAREST)
    inst = []
    for i in range(7):
        r = _rand_rect(rng, width, height, 40, 240, integer=not fractional)
        ux, uy = float(2 * rng.randint(0, 30)), float(2 * rng.randint(0, 20))
        if i == 0:
            uw, uh = float(int(min(r[2] - r[0], vw - ux)) & ~1), float(int(min(r[3] - r[1], vh - uy)) & ~1)
            r = (r[0], r[1], r[0] + uw, r[1] + uh)
        else:
            uw, uh = float(2 * rng.randint(10, 60)), float(2 * rng.randint(8, 40))
        ry = (ux, uy, ux + uw, uy + uh)
        rc = tuple(v * 0.5 for v in ry)
        srcs = [t.push_gpu_cache([rr, (0.0, 0.0, 0.0, 0.0)]) for rr in (ry, rc, rc)]
        spec = t.push_gpu_cache([(float(depth), float(color_space), float(yuv_format), 0.0)])
        clip = r if i % 3 else (r[0] + 4.0, r[1] + 3.0, r[2] - 6.0, r[3] - 2.0)
        clip_task = CLIP_TASK_EMPTY
        if with_masks and alpha_pass and i % 3 == 1:
            w_, h_ = int(min(r[2] - r[0], 120)), int(min(r[3] - r[1], 100))
            mx, my = int(rng.randint(0, 256 - w_)), int(rng.randint(0, 256 - h_))
            clip_task = t.add_render_task((float(mx), float(my), float(mx + w_), float(my + h_)), 1.0,
                                          (float(int(r[0])), float(int(r[1]))))
        hdr = t.add_prim_header(r, clip, i + 1, spec, xf, pic, (srcs[0], srcs[1], srcs[2], 0))
        edge = 0xF if (alpha_pass and (fractional or rotate is not None)) else 0
        inst.append(brush_instance(hdr, clip_task, 0xFFFF, edge, 0, 0))
    feats = abi.FEAT_TEXTURE_2D | abi.FEAT_YUV | (abi.FEAT_ALPHA_PASS if alpha_pass else 0)
    ops = [Clear(color=(0.2, 0.3, 0.1, 1.0)),
           Batch(abi.KIND_BRUSH_YUV_IMAGE, np.stack(inst),
                 blend=abi.BLEND_PREMULTIPLIED_ALPHA if alpha_pass else abi.BLEND_NONE,
                 features=feats, color=names, clip_mask="mask" if (with_masks and alpha_pass) else "")]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def hdr_video_frame(width=3840, height=2160, vw=1920, vh=1080, fmt="p010", depth=10, color_space=2, seed=1):
    """video_frame with a 10-, 12- or 16-bit source: one vw x vh surface (P010 by default, Rec.709 narrow range)
    scaled to the whole framebuffer by `composite` YUV."""
    from webrender_b200.gpu_types import composite_yuv_instance
    names, yuv_format, textures = _hdr_yuv_textures(fmt, vw, vh, seed, depth, abi.LINEAR)
    textures["fb"] = TextureDesc(abi.FMT_RGBA8, width, height)
    r = (0.0, 0.0, float(width), float(height))
    ry = (0.0, 0.0, float(vw), float(vh))
    rc = tuple(v * 0.5 for v in ry)
    inst = composite_yuv_instance(r, r, color_space, yuv_format, depth, (ry, rc, rc))
    ops = [Clear(color=(0.0, 0.0, 0.0, 1.0)),
           Batch(abi.KIND_COMPOSITE, inst[None, :], blend=abi.BLEND_NONE,
                 features=abi.FEAT_TEXTURE_2D | abi.FEAT_YUV, color=names)]
    return Frame(FrameTables().arrays(), textures, [[Target("fb", ops=ops)]])


def _picture_source(t, rng, aw, ah, w, h, one_to_one):
    """gpu-cache entry of an off-screen picture's uv rect the way
    RenderTaskCache/resolve_location publishes it: uv rect, user data, and the
    four homogeneous corner coordinates get_image_quad_uv reads
    (gpu_cache.glsl:103-135)."""
    if one_to_one:
        uw, uh = int(w), int(h)
    else:
        uw, uh = int(rng.randint(16, 160)), int(rng.randint(16, 120))
    uw, uh = min(uw, aw - 1), min(uh, ah - 1)
    u0, v0 = int(rng.randint(0, aw - uw)), int(rng.randint(0, ah - uh))
    return t.push_gpu_cache([(float(u0), float(v0), float(u0 + uw), float(v0 + uh)), (0.0, 0.0, 0.0, 0.0),
                             (0.0, 0.0, 0.0, 1.0), (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0), (1.0, 1.0, 0.0, 1.0)])


def opacity_frame(width=640, height=360, n_prims=14, seed=1, fractional=False, one_to_one=False, filter=abi.LINEAR,
                  rotate=None, brush_flags=0):
    """Brush(Opacity) batch (batch.rs:1671-1712): pictures with a filter:
    opacity() drawn from their off-screen surface, premultiplied-alpha blended;
    prim user data = [uv_rect_address, amount * 65536, 0, 0]."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    aw, ah = 320, 200
    inst = []
    # `rotate`: the pictures sit under a transformed spatial node (with_transform: any 4x4, e.g. a perspective one)
    xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0), axis_aligned=False) if rotate is not None else 0
    for i in range(n_prims):
        r = _rand_rect(rng, width, height, 24, 220, integer=not fractional)
        src = _picture_source(t, rng, aw, ah, r[2] - r[0], r[3] - r[1], one_to_one)
        spec = t.push_gpu_cache([(0.0, 0.0, 0.0, 0.0)] * 3)
        amount = 1.0 if i % 5 == 0 else float(rng.uniform(0.05, 1.0))
        hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), i + 1, spec, xf, pic, (src, int(amount * 65536.0), 0, 0))
        inst.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, brush_flags if i % 2 else 0, 0))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "surface": TextureDesc(abi.FMT_RGBA8, aw, ah, data=tile_texture(aw, ah, seed + 31, opaque=False), filter=filter)}
    ops = [Clear(color=(0.9, 0.9, 0.9, 1.0)),
           Batch(abi.KIND_BRUSH_OPACITY, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                 features=abi.FEAT_ALPHA_PASS, color=("surface", "", ""))]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def clear_frame(width=512, height=320, seed=1, r8=False):
    """Quad-based clears (ps_clear; renderer/mod.rs:2714-2744, 3795-3833,
    3971-3994): rects cleared by ClearInstance quads with depth forced to the
    far plane (so a depth-writing clear also resets depth), between batches of
    opaque depth-tested solid brushes."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))

    def solids(n, z0):
        out = []
        for i in range(n):
            r = _rand_rect(rng, width, height, 30, 260)
            addr = t.push_gpu_cache([tuple(float(v) for v in rng.uniform(0, 1, 3)) + (1.0,)])
            hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), z0 + i, addr, 0, pic, (65535, 0, 0, 0))
            out.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
        return np.stack(out[::-1])

    def clears(n, colors):
        out = np.zeros((n, 8), dtype=np.float32)
        for i in range(n):
            out[i, 0:4] = _rand_rect(rng, width, height, 40, 220)
            out[i, 4:8] = colors[i % len(colors)]
        return out

    if r8:
        textures = {"target": TextureDesc(abi.FMT_R8, width, height)}
        ops = [Clear(color=(0.5, 0.5, 0.5, 0.5)),
               Batch(abi.KIND_CLEAR, clears(6, [(0.0, 0.0, 0.0, 0.0), (1.0, 1.0, 1.0, 1.0)]))]
        return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "depth": TextureDesc(abi.FMT_DEPTH24, width, height)}
    ops = [Clear(color=(0.1, 0.2, 0.3, 1.0), depth=1.0),
           Batch(abi.KIND_BRUSH_SOLID, solids(8, 10), depth=abi.DEPTH_TEST_WRITE),
           Batch(abi.KIND_CLEAR, clears(3, [(0.0, 0.0, 0.0, 0.0), (0.25, 0.5, 0.75, 1.0)]), depth=abi.DEPTH_TEST_WRITE),
           Batch(abi.KIND_BRUSH_SOLID, solids(8, 1), depth=abi.DEPTH_TEST_WRITE),
           Batch(abi.KIND_CLEAR, clears(2, [(1.0, 1.0, 1.0, 1.0)]))]
    return Frame(t.arrays(), textures, [[Target("target", depth="depth", ops=ops)]])


# Filter::as_int (internal_types.rs) / blend.glsl:13-24
(FILTER_CONTRAST, FILTER_GRAYSCALE, FILTER_HUE_ROTATE, FILTER_INVERT, FILTER_SATURATE, FILTER_SEPIA,
 FILTER_BRIGHTNESS, FILTER_COLOR_MATRIX, FILTER_SRGB_TO_LINEAR, FILTER_LINEAR_TO_SRGB, FILTER_FLOOD,
 FILTER_COMPONENT_TRANSFER) = range(12)


def blend_frame(width=640, height=400, seed=1, fractional=False, opaque_source=False, rotate=None):
    """Brush(Blend) batch (batch.rs:1715-1890): one picture per CSS filter op —
    contrast, grayscale, hue-rotate, invert, saturate, sepia, brightness, colour
    matrix, sRGB<->linear, flood and a component transfer (table / discrete /
    linear / gamma) — each reading its off-screen surface through sColor0."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    aw, ah = 320, 200
    inst = []
    xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0), axis_aligned=False) if rotate is not None else 0
    filters = [(FILTER_CONTRAST, 1.6), (FILTER_GRAYSCALE, 0.7), (FILTER_HUE_ROTATE, 110.0), (FILTER_INVERT, 0.85),
               (FILTER_SATURATE, 2.2), (FILTER_SEPIA, 0.6), (FILTER_BRIGHTNESS, 1.4), (FILTER_COLOR_MATRIX, None),
               (FILTER_SRGB_TO_LINEAR, None), (FILTER_LINEAR_TO_SRGB, None), (FILTER_FLOOD, None),
               (FILTER_COMPONENT_TRANSFER, None), (FILTER_CONTRAST, 0.4), (FILTER_BRIGHTNESS, 0.5)]
    for i, (op, amount) in enumerate(filters):
        col, row = i % 5, i // 5
        x0, y0 = 8 + col * 126 + (float(rng.uniform(0, 1)) if fractional else 0.0), 8 + row * 130 + (float(rng.uniform(0, 1)) if fractional else 0.0)
        r = (x0, y0, x0 + 118.0, y0 + 122.0)
        src = _picture_source(t, rng, aw, ah, 118, 122, i % 2 == 0)
        mode = op
        if op in (FILTER_CONTRAST, FILTER_GRAYSCALE, FILTER_INVERT, FILTER_SATURATE, FILTER_SEPIA, FILTER_BRIGHTNESS):
            user = int(amount * 65536.0)
        elif op == FILTER_HUE_ROTATE:
            user = int(0.01745329251 * amount * 65536.0)
        elif op == FILTER_COLOR_MATRIX:
            m = rng.uniform(-0.3, 0.9, (4, 4)).astype(np.float32)
            user = t.push_gpu_cache([tuple(float(v) for v in m[k]) for k in range(4)] +
                                    [tuple(float(v) for v in rng.uniform(-0.1, 0.2, 4))])
        elif op == FILTER_FLOOD:
            user = t.push_gpu_cache([(0.2, 0.6, 0.4, 0.7)])
        elif op == FILTER_COMPONENT_TRANSFER:
            # r: table (256 values = 64 blocks), g: discrete, b: linear, a: gamma
            table = np.clip(np.linspace(0, 1, 256) ** 0.5 + rng.uniform(-0.02, 0.02, 256), -0.1, 1.1).astype(np.float32)
            disc = (np.floor(np.linspace(0, 0.999, 256) * 5) / 4).astype(np.float32)
            blocks = [tuple(float(v) for v in table[4 * k: 4 * k + 4]) for k in range(64)]
            blocks += [tuple(float(v) for v in disc[4 * k: 4 * k + 4]) for k in range(64)]
            blocks += [(0.8, 0.1, 0.0, 0.0), (0.9, 1.7, 0.05, 0.0)]
            user = t.push_gpu_cache(blocks)
            mode = op | (1 << 28) | (2 << 24) | (3 << 20) | (4 << 16)
        else:
            user = 0
        spec = t.push_gpu_cache([(0.0, 0.0, 0.0, 0.0)] * 3)
        hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), i + 1, spec, xf, pic, (src, mode, user, 0))
        inst.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "surface": TextureDesc(abi.FMT_RGBA8, aw, ah, data=tile_texture(aw, ah, seed + 51, opaque=opaque_source),
                                       filter=abi.LINEAR)}
    blend = abi.BLEND_NONE if opaque_source else abi.BLEND_PREMULTIPLIED_ALPHA
    ops = [Clear(color=(0.8, 0.85, 0.9, 1.0)),
           Batch(abi.KIND_BRUSH_BLEND, np.stack(inst), blend=blend,
                 features=0 if opaque_source else abi.FEAT_ALPHA_PASS, color=("surface", "", ""))]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


FILTER_REFTESTS = {
    # wrench/reftests/filters/<name>.yaml == <name>-ref.yaml (filters/reftest.list:11-41): a rect under a CSS filter must
    # equal a plain rect of the colour the reference's authors computed.  (page background, [(rect, source colour
    # 0-255 + alpha, filter, amount, expected colour 0-255 + alpha)], allowed (max diff, pixels))
    "filter-grayscale": ((255, 255, 255), [((10, 10, 210, 210), (0, 255, 0, 1.0), FILTER_GRAYSCALE, 1.0, (182, 182, 182, 1.0))], (0, 0)),
    "filter-brightness": ((0, 0, 0), [((10, 10, 110, 110), (255, 255, 255, 0.25), FILTER_BRIGHTNESS, 2.0, (64, 64, 64, 1.0))], (0, 0)),
    "filter-brightness-2": ((255, 255, 255), [((10, 10, 110, 110), (255, 0, 0, 1.0), FILTER_BRIGHTNESS, 0.0, (0, 0, 0, 1.0))], (0, 0)),
    "filter-invert": ((255, 255, 255), [((10, 10, 110, 110), (255, 255, 255, 0.25), FILTER_INVERT, 1.0, (0, 0, 0, 0.25))], (0, 0)),
    "filter-saturate-red-2": ((0, 0, 0), [((10, 10, 110, 110), (255, 0, 0, 1.0), FILTER_SATURATE, 0.5, (155, 27, 27, 1.0))], (0, 0)),
    "filter-contrast-gray-alpha-1": ((255, 255, 255), [((10, 10, 110, 110), (128, 128, 128, 0.25), FILTER_CONTRAST, 0.0,
                                                        (223, 223, 223, 1.0))], (0, 0)),
    "filter-hue-rotate-1": ((0, 0, 0), [((10, 10, 60, 60), (255, 0, 0, 1.0), FILTER_HUE_ROTATE, 90.0, (0, 91, 0, 1.0)),
                                        ((10, 60, 60, 110), (0, 255, 0, 1.0), FILTER_HUE_ROTATE, 90.0, (0, 218, 255, 1.0)),
                                        ((60, 10, 110, 60), (0, 0, 255, 1.0), FILTER_HUE_ROTATE, 90.0, (255, 0, 37, 1.0)),
                                        ((60, 60, 110, 110), (128, 128, 128, 1.0), FILTER_HUE_ROTATE, 90.0, (128, 128, 128, 1.0))],
                            (1, 14)),   # fuzzy(1,14)
}


def filter_reftest_frames(name, size=(220, 220)):
    """(test frame, reference frame) of one of FILTER_REFTESTS: the filtered rects as Brush(Blend) instances reading
    uniform picture surfaces (premultiplied 8-bit, as the picture pass leaves them), the reference rects as alpha
    Brush(Solid) instances, both premultiplied-over the page colour."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    bg, cases, _ = FILTER_REFTESTS[name]
    w, h = size
    out = []
    for ref in (False, True):
        t = FrameTables()
        pic = t.add_render_task((0.0, 0.0, float(w), float(h)), 1.0, (0.0, 0.0))
        inst = []
        textures = {"target": TextureDesc(abi.FMT_RGBA8, w, h)}
        sw, sh = 64 * len(cases), 64
        surf = np.zeros((sh, sw, 4), dtype=np.uint8)
        for i, (r, src, op, amount, exp) in enumerate(cases):
            rect = tuple(float(v) for v in r)
            if ref:
                a = float(exp[3])
                c = tuple(float(v) / 255.0 * a for v in exp[:3]) + (a,)
                addr = t.push_gpu_cache([c])
                hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), i + 1, addr, 0, pic, (65535, 0, 0, 0))
                inst.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
                continue
            a = float(src[3])
            px = [int(np.float32(v / 255.0 * a) * np.float32(255.0) + np.float32(0.5)) for v in src[:3]] + [int(a * 255.0 + 0.5)]
            surf[:, 64 * i: 64 * i + 64] = (px[2], px[1], px[0], px[3])   # BGRA
            res = t.push_gpu_cache([(64.0 * i + 8, 8.0, 64.0 * i + 56, 56.0), (0.0, 0.0, 0.0, 0.0),
                                    (0.0, 0.0, 0.0, 1.0), (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0), (1.0, 1.0, 0.0, 1.0)])
            user = int(0.01745329251 * amount * 65536.0) if op == FILTER_HUE_ROTATE else int(amount * 65536.0)
            spec = t.push_gpu_cache([(0.0, 0.0, 0.0, 0.0)] * 3)
            hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), i + 1, spec, 0, pic, (res, op, user, 0))
            inst.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
        clear = Clear(color=tuple(v / 255.0 for v in bg) + (1.0,))
        if ref:
            ops = [clear, Batch(abi.KIND_BRUSH_SOLID, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS)]
        else:
            textures["surface"] = TextureDesc(abi.FMT_RGBA8, sw, sh, data=surf.reshape(sh, sw * 4), filter=abi.LINEAR)
            ops = [clear, Batch(abi.KIND_BRUSH_BLEND, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                features=abi.FEAT_ALPHA_PASS, color=("surface", "", ""))]
        out.append(Frame(t.arrays(), textures, [[Target("target", ops=ops)]]))
    return out[0], out[1]


PICTURE_REFTESTS = {
    # Known answers the reference's authors wrote down for picture compositing (a yaml that must equal a plain rect of
    # the stated colour): (page background, rect, kind, source colour 0-255 + alpha, parameter, backdrop colour or None,
    # expected colour 0-255, allowed (max diff, pixels)).
    # filters/opacity.yaml == opacity-ref.yaml, fuzzy-if(platform(swgl),1,10000): "opacity pre-multiplied color"
    "opacity": ((255, 255, 255), (20, 20, 120, 120), "opacity", (255, 255, 0, 0.2), 0.9, None, (255, 255, 209), (1, 10000)),
    # filters/opacity-overlap.yaml == opacity-overlap-ref.yaml, fuzzy-if(platform(swgl),1,10000): (0,0,128) at opacity 0.75
    # over an opaque (128,0,0) rect
    "opacity-overlap": ((255, 255, 255), (20, 20, 120, 120), "opacity", (0, 0, 128, 1.0), 0.75, (128, 0, 0), (32, 0, 96), (1, 10000)),
    # blend/multiply.yaml == multiply-ref.yaml: green x green = green
    "multiply": ((255, 255, 255), (25, 25, 75, 75), "mix", (0, 255, 0, 1.0), 1, (0, 255, 0), (0, 255, 0), (0, 0)),
    # blend/difference.yaml == difference-ref.yaml: green - green = black
    "difference": ((255, 255, 255), (0, 0, 100, 100), "mix", (0, 255, 0, 1.0), 10, (0, 255, 0), (0, 0, 0), (0, 0)),
    # blend/darken.yaml, lighten.yaml (fuzzy-if(platform(swgl),1,10000)): per-channel min / max
    "darken": ((255, 255, 255), (0, 0, 100, 100), "mix", (30, 20, 10, 1.0), 4, (10, 20, 30), (10, 20, 10), (1, 10000)),
    "lighten": ((255, 255, 255), (0, 0, 100, 100), "mix", (30, 20, 10, 1.0), 5, (10, 20, 30), (30, 20, 30), (1, 10000)),
    # the same four the way SWGL itself draws them: KHR_blend_equation_advanced on the picture's draw (blend.h advanced
    # equations; parameter = wrcu_blend key)
    "adv-multiply": ((255, 255, 255), (25, 25, 75, 75), "adv", (0, 255, 0, 1.0), abi.BLEND_ADV_MULTIPLY, (0, 255, 0), (0, 255, 0), (0, 0)),
    "adv-difference": ((255, 255, 255), (0, 0, 100, 100), "adv", (0, 255, 0, 1.0), abi.BLEND_ADV_DIFFERENCE, (0, 255, 0), (0, 0, 0), (0, 0)),
    "adv-darken": ((255, 255, 255), (0, 0, 100, 100), "adv", (30, 20, 10, 1.0), abi.BLEND_ADV_DARKEN, (10, 20, 30), (10, 20, 10), (1, 10000)),
    "adv-lighten": ((255, 255, 255), (0, 0, 100, 100), "adv", (30, 20, 10, 1.0), abi.BLEND_ADV_LIGHTEN, (10, 20, 30), (30, 20, 30), (1, 10000)),
}


def picture_reftest_frame(name, size=(140, 140)):
    """One of PICTURE_REFTESTS: a uniform picture surface (premultiplied 8-bit, as the picture pass leaves it) drawn by
    Brush(Opacity) or Brush(MixBlend) — backdrop readback in sColor0, the picture's surface in sColor1 — over the page
    (for mix-blend: over the backdrop rect drawn first), premultiplied blending."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    bg, r, kind, src, param, backdrop, _, _ = PICTURE_REFTESTS[name]
    w, h = size
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(w), float(h)), 1.0, (0.0, 0.0))
    rect = tuple(float(v) for v in r)

    def uniform(col, alpha):
        px = [int(np.float32(v / 255.0 * alpha) * np.float32(255.0) + np.float32(0.5)) for v in col] + [int(alpha * 255.0 + 0.5)]
        img = np.zeros((64, 64, 4), dtype=np.uint8)
        img[:, :] = (px[2], px[1], px[0], px[3])   # BGRA
        return img.reshape(64, 256)

    def source():
        return t.push_gpu_cache([(8.0, 8.0, 56.0, 56.0), (0.0, 0.0, 0.0, 0.0),
                                 (0.0, 0.0, 0.0, 1.0), (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0), (1.0, 1.0, 0.0, 1.0)])
    textures = {"target": TextureDesc(abi.FMT_RGBA8, w, h),
                "surface": TextureDesc(abi.FMT_RGBA8, 64, 64, data=uniform(src[:3], float(src[3])), filter=abi.LINEAR)}
    ops = [Clear(color=tuple(v / 255.0 for v in bg) + (1.0,))]
    spec = t.push_gpu_cache([(0.0, 0.0, 0.0, 0.0)] * 3)
    if kind == "opacity":
        if backdrop is not None:   # an opaque rect under the picture
            baddr = t.push_gpu_cache([tuple(float(v) / 255.0 for v in backdrop) + (1.0,)])
            bh = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), 1, baddr, 0, pic, (65535, 0, 0, 0))
            ops.append(Batch(abi.KIND_BRUSH_SOLID, brush_instance(bh, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)[None, :],
                             blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS))
        hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), 2, spec, 0, pic, (source(), int(param * 65536.0), 0, 0))
        ops.append(Batch(abi.KIND_BRUSH_OPACITY, brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)[None, :],
                         blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS, color=("surface", "", "")))
    elif kind == "adv":
        # the backdrop rect, then the picture's content drawn with the advanced blend equation
        baddr = t.push_gpu_cache([tuple(float(v) / 255.0 for v in backdrop) + (1.0,)])
        bh = t.add_prim_header((0.0, 0.0, 100.0, 100.0), (-1e9, -1e9, 1e9, 1e9), 1, baddr, 0, pic, (65535, 0, 0, 0))
        ops.append(Batch(abi.KIND_BRUSH_SOLID, brush_instance(bh, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)[None, :],
                         blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS))
        a = float(src[3])
        saddr = t.push_gpu_cache([tuple(float(v) / 255.0 * a for v in src[:3]) + (a,)])
        sh = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), 2, saddr, 0, pic, (65535, 0, 0, 0))
        ops.append(Batch(abi.KIND_BRUSH_SOLID, brush_instance(sh, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)[None, :],
                         blend=int(param), features=abi.FEAT_ALPHA_PASS))
    else:
        # the backdrop content (an opaque rect of the blend container), then the mix-blend picture over it
        baddr = t.push_gpu_cache([tuple(float(v) / 255.0 for v in backdrop) + (1.0,)])
        bh = t.add_prim_header((0.0, 0.0, 100.0, 100.0), (-1e9, -1e9, 1e9, 1e9), 1, baddr, 0, pic, (65535, 0, 0, 0))
        ops.append(Batch(abi.KIND_BRUSH_SOLID, brush_instance(bh, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)[None, :],
                         blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS))
        textures["backdrop"] = TextureDesc(abi.FMT_RGBA8, 64, 64, data=uniform(backdrop, 1.0), filter=abi.LINEAR)
        hdr = t.add_prim_header(rect, (-1e9, -1e9, 1e9, 1e9), 2, spec, 0, pic, (int(param), source(), source(), 0))
        ops.append(Batch(abi.KIND_BRUSH_MIX_BLEND, brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)[None, :],
                         blend=abi.BLEND_PREMULTIPLIED_ALPHA, features=abi.FEAT_ALPHA_PASS, color=("backdrop", "surface", "")))
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def mix_blend_frame(width=640, height=400, seed=1, fractional=False, rotate=None):
    """Brush(MixBlend) batch (batch.rs:1931-2001): one picture per non-separable /
    separable mix-blend-mode handled in the shader (multiply, overlay, darken,
    lighten, colour-dodge, colour-burn, hard-light, soft-light, difference, hue,
    saturation, colour, luminosity): sColor0 = backdrop readback, sColor1 = the
    picture's own surface; user data = [mode, backdrop uv, source uv, 0]."""
    from webrender_b200.gpu_types import brush_instance, CLIP_TASK_EMPTY
    rng = np.random.RandomState(seed)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(width), float(height)), 1.0, (0.0, 0.0))
    aw, ah = 320, 200
    inst = []
    xf = t.add_transform(rotation_matrix(rotate, width / 2.0, height / 2.0), axis_aligned=False) if rotate is not None else 0
    modes = [1, 3, 4, 5, 6, 7, 8, 9, 10, 12, 13, 14, 15, 9, 6]
    for i, mode in enumerate(modes):
        col, row = i % 5, i // 5
        jx = float(rng.uniform(0, 1)) if fractional else 0.0
        jy = float(rng.uniform(0, 1)) if fractional else 0.0
        x0, y0 = 8 + col * 126 + jx, 8 + row * 130 + jy
        r = (x0, y0, x0 + 118.0, y0 + 122.0)
        back = _picture_source(t, rng, aw, ah, 118, 122, True)
        src = _picture_source(t, rng, aw, ah, 118, 122, i % 3 != 2)
        spec = t.push_gpu_cache([(0.0, 0.0, 0.0, 0.0)] * 3)
        hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), i + 1, spec, xf, pic, (mode, back, src, 0))
        inst.append(brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, width, height),
                "backdrop": TextureDesc(abi.FMT_RGBA8, aw, ah, data=tile_texture(aw, ah, seed + 61, opaque=seed % 2 == 0),
                                        filter=abi.LINEAR),
                "surface": TextureDesc(abi.FMT_RGBA8, aw, ah, data=tile_texture(aw, ah, seed + 62, opaque=False),
                                       filter=abi.LINEAR)}
    ops = [Clear(color=(0.8, 0.85, 0.9, 1.0)),
           Batch(abi.KIND_BRUSH_MIX_BLEND, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                 features=abi.FEAT_ALPHA_PASS, color=("backdrop", "surface", ""))]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])


def config_a_frame():
    """Config A: wrench/reftests/aa/rounded-rects.yaml — three solid rects under
    rounded-rect clips (uniform radius 8; per-corner circular 16/32/48/64;
    per-corner elliptical), white background, drawn the Indirect way (see
    rounded_rects_frame) at the size of its reference image (1036x604)."""
    spec = [((50, 50, 250, 250), (1.0, 0.0, 0.0, 1.0), 8.0),
            ((270, 50, 470, 250), (0.0, 1.0, 0.0, 1.0), ((16.0, 16.0), (32.0, 32.0), (48.0, 48.0), (64.0, 64.0))),
            ((490, 50, 990, 550), (0.0, 0.0, 1.0, 1.0), ((32.0, 16.0), (40.0, 24.0), (48.0, 64.0), (52.0, 80.0)))]
    return rounded_rects_frame(width=1036, height=604, spec=spec, surface=(1024, 512))


def blur_frame(width=384, height=256, seed=1, color=False, sigmas=(1.0, 2.5, 6.0, 0.0)):
    """cs_blur the way draw_blurs issues it (renderer/mod.rs:3675-3692; render
    tasks from RenderTask::new_blur, render_task.rs): for each source region a
    vertical pass into an intermediate target and a horizontal pass from it into
    the final target — ALPHA_TARGET (R8 box-shadow masks) or COLOR_TARGET (RGBA8
    filter blurs).  Regions sit at different offsets so the clamped sampling at
    the region edges is exercised."""
    from webrender_b200.gpu_types import blur_instance
    rng = np.random.RandomState(seed)
    t = FrameTables()
    fmt = abi.FMT_RGBA8 if color else abi.FMT_R8
    sw, sh = 256, 192
    src = tile_texture(sw, sh, seed + 5, opaque=False) if color else shadow_mask_texture(256, seed + 5)[:sh, :sw].copy()
    vert, hori = [], []
    x_cursor = 0
    for i, sigma in enumerate(sigmas):
        w, h = int(rng.randint(40, 90)), int(rng.randint(30, 120))
        sx, sy = int(rng.randint(0, sw - w)), int(rng.randint(0, sh - h))
        src_task = t.add_render_task((float(sx), float(sy), float(sx + w), float(sy + h)), 1.0, (0.0, 0.0))
        mid_task = t.add_render_task((float(x_cursor), 4.0, float(x_cursor + w), float(4 + h)), 1.0, (0.0, 0.0))
        dst_task = t.add_render_task((float(x_cursor + 2), 7.0, float(x_cursor + 2 + w), float(7 + h)), 1.0, (0.0, 0.0))
        region = (float(w), float(h)) if i % 2 == 0 else (float(w - 6), float(h - 4))
        vert.append(blur_instance(mid_task, src_task, 1, sigma, region))
        hori.append(blur_instance(dst_task, mid_task, 0, sigma, region))
        x_cursor += w + 6
    feat = abi.FEAT_COLOR_TARGET if color else abi.FEAT_ALPHA_TARGET
    textures = {"source": TextureDesc(fmt, sw, sh, data=src, filter=abi.LINEAR),
                "mid": TextureDesc(fmt, width, height, filter=abi.LINEAR),
                "target": TextureDesc(fmt, width, height, filter=abi.LINEAR)}
    p0 = [Clear(color=(0.0, 0.0, 0.0, 0.0)),
          Batch(abi.KIND_BLUR, np.stack(vert), features=feat, color=("source", "", ""))]
    p1 = [Clear(color=(0.0, 0.0, 0.0, 0.0)),
          Batch(abi.KIND_BLUR, np.stack(hori), features=feat, color=("mid", "", ""))]
    return Frame(t.arrays(), textures, [[Target("mid", ops=p0)], [Target("target", ops=p1)]])


def scale_frame(width=384, height=256, seed=1, r8=False, filter=abi.LINEAR):
    """cs_scale (handle_scaling, renderer/mod.rs:2472-2530): ScalingInstance
    copies of source rects at 1:1, 2:1 down (the blur pipeline's downscale
    steps), arbitrary scales and a flipped source rect; unnormalised uvs."""
    rng = np.random.RandomState(seed)
    fmt = abi.FMT_R8 if r8 else abi.FMT_RGBA8
    sw, sh = 320, 200
    src = shadow_mask_texture(320, seed + 3)[:sh, :sw].copy() if r8 else tile_texture(sw, sh, seed + 3, opaque=False)
    inst = np.zeros((5, 9), dtype=np.float32)
    x_cursor = 4
    for i in range(5):
        w, h = int(rng.randint(30, 70)), int(rng.randint(24, 110))
        tx, ty = x_cursor, int(rng.randint(2, 40))
        x_cursor += w + 5
        if i == 0:
            sw_, sh_ = w, h
        elif i == 1:
            sw_, sh_ = 2 * w, 2 * h
        else:
            sw_, sh_ = int(rng.randint(20, 140)), int(rng.randint(16, 90))
        sx, sy = int(rng.randint(0, sw - sw_)), int(rng.randint(0, sh - sh_))
        s = (float(sx), float(sy), float(sx + sw_), float(sy + sh_))
        if i == 3:
            s = (s[2], s[1], s[0], s[3])   # inverted u
        inst[i, 0:4] = (tx, ty, tx + w, ty + h)
        inst[i, 4:8] = s
        inst[i, 8] = 1.0
    textures = {"source": TextureDesc(fmt, sw, sh, data=src, filter=filter),
                "target": TextureDesc(fmt, width, height)}
    ops = [Clear(color=(0.0, 0.0, 0.0, 0.0)),
           Batch(abi.KIND_SCALE, inst, features=abi.FEAT_TEXTURE_2D, color=("source", "", ""))]
    return Frame(FrameTables().arrays(), textures, [[Target("target", ops=ops)]])


def _no_corner_overlap(radii, w, h):
    """ensure_no_corner_overlap (webrender/src/border.rs:168-215) in f32."""
    f = np.float32
    (tl, tr, bl, br) = [(f(a), f(b)) for a, b in radii]
    ratio = f(1.0)
    for size, s1, s2 in ((f(w), tl[0] + tr[0], bl[0] + br[0]), (f(h), tl[1] + bl[1], tr[1] + br[1])):
        if size > 0:
            for ssum in (s1, s2):
                if size < ssum:
                    ratio = min(ratio, f(size / ssum))
    if ratio < 1.0:
        tl, tr, bl, br = [(f(a * ratio), f(b * ratio)) for a, b in (tl, tr, bl, br)]
    return tuple((float(a), float(b)) for a, b in (tl, tr, bl, br))


def reftest_clip_frame(which="clip-mode"):
    """wrench/reftests/clip/clip-mode.yaml and clip-ellipse.yaml: 100x100 rects under
    rounded-rect clips (uniform radius 32 / elliptical radii incl. over-large ones
    that the frame builder scales down), alternately Clip and ClipOut, drawn the
    Indirect way at the size of their reference images."""
    red, green = (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0)
    spec = []
    if which == "clip-mode":
        spec = [((20, 20, 120, 120), red, 32.0, 0), ((130, 20, 230, 120), green, 32.0, 1)]
        size = (250, 140)
    else:
        for row, (rx, ry) in enumerate([(32, 16), (16, 32), (128, 32), (32, 128)]):
            y0 = 20 + 110 * row
            rad = _no_corner_overlap(((rx, ry),) * 4, 100, 100)
            spec.append(((20, y0, 120, y0 + 100), red, rad, 0))
            spec.append(((130, y0, 230, y0 + 100), green, rad, 1))
        size = (250, 470)
    return rounded_rects_frame(width=size[0], height=size[1], spec=spec, surface=(512, 512))


def reftest_box_shadow_frame(which="inset-no-blur-radius"):
    if which == "suite-no-blur":
        return reftest_box_shadow_suite_no_blur_frame()
    return _reftest_box_shadow_frame(which)


def _reftest_box_shadow_frame(which="inset-no-blur-radius"):
    """wrench/reftests/boxshadow/inset-no-blur-radius.yaml: an INSET box shadow with blur radius 0 takes the frame
    builder's no-blur path (box_shadow.rs:341-401): a Rectangle primitive = the box (10,10)-(90,90) in the shadow
    colour under two rounded clips — Clip to the box (radius 10) and ClipOut of the shadow rect = the box moved by the
    offset (10,10), same radius (spread 0).  A clipped rect of this size is drawn the Indirect way (quad.rs:722-792):
    off-screen task, one ps_quad_mask per clip multiplied in, textured composite.  Reference image 106x112."""
    if which == "box-shadow-spread":
        # boxshadow/box-shadow-spread.yaml: nine inset shadows, spread 10, no blur, no offset, border radii 20..4: the
        # shadow rect is the box shrunk by the spread, its radius max(r - 10, 0) (adjust_radius_for_box_shadow,
        # box_shadow.rs:577-583).  Reference image 917x125.
        blue = (0.0, 0.0, 1.0, 1.0)
        spec = []
        for k, r in enumerate([20, 25, 10, 9, 8, 7, 6, 5, 4]):
            x = 20 + 100 * k
            spec.append(((x, 20, x + 80, 100), blue, float(r), 0,
                         [((x + 10.0, 30.0, x + 70.0, 90.0), float(max(r - 10, 0)), 1)]))
        return rounded_rects_frame(width=917, height=125, spec=spec, surface=(512, 512))
    if which == "boxshadow-spread-only":
        # boxshadow/boxshadow-spread-only.yaml: OUTSET, spread 20, no blur, radius 200 on a 400x400 box: the primitive
        # is the shadow rect (box inflated by the spread, radius 220) clipped OUT of the box (box_shadow.rs:351-367).
        # Reference image 562x497.  (The reference splits a quad this large into tiles; the per-pixel coverage is the
        # same whichever tile computes it.)
        spec = [((20, 20, 460, 460), (0.0, 0.0, 0.0, 1.0), 220.0, 0, [((40.0, 40.0, 440.0, 440.0), 200.0, 1)])]
        return rounded_rects_frame(width=562, height=497, spec=spec, surface=(512, 512))
    assert which == "inset-no-blur-radius"
    red = (1.0, 0.0, 0.0, 1.0)
    spec = [((10, 10, 90, 90), red, 10.0, 0, [((20.0, 20.0, 100.0, 100.0), 10.0, 1)])]
    return rounded_rects_frame(width=106, height=112, spec=spec, surface=(256, 256))


def reftest_border_overlapping_frame():
    """wrench/reftests/border/overlapping.yaml (== overlapping.png, fuzzy-if(platform(swgl),1,20)): a blue 200x200 rect
    under a complex clip whose top-left and bottom-right radii are 180 — the two corner ellipses overlap, and every
    pixel must still take exactly one corner's distance (ps_quad_mask.glsl:55-60 per-corner radii, the slow path).
    Drawn the Indirect way like config A; reference image 233x240."""
    spec = [((0, 0, 200, 200), (0.0, 0.0, 1.0, 1.0), ((180.0, 180.0), (0.0, 0.0), (0.0, 0.0), (180.0, 180.0)), 0)]
    return rounded_rects_frame(width=233, height=240, spec=spec, surface=(256, 256))


def reftest_border_no_bogus_line_frame():
    """wrench/reftests/border/border-no-bogus-line.yaml (== border-no-bogus-line-ref.png, fuzzy-if(platform(swgl),1,8)):
    a solid black border, width 3, radius 40.5, on the box (10,10)-(100,90).  The radii do not fit the 80-pixel height:
    ensure_no_corner_overlap (border.rs:168-215, called by add_normal_border) scales them by 80/81 — exactly 40.0 in
    fp32 — so the corners are 40x40, the left and right edges have no length (no "bogus line" between the corners)
    and the top and bottom edges are 10 long.  Draw list as the frame builder makes it (border.rs:654-898, 904-1042,
    1245-1297): each corner a cs_border_solid task of 40x40 in the texture cache (widths 3, radius 40, AA, the adjacent
    corners' clips collapsed onto the task's own corners since their radii do not reach it), each edge an 8x3 task;
    then one Brush(Image) instance per segment — SEGMENT_RELATIVE | SEGMENT_TEXEL_RECT corners, SEGMENT_RELATIVE |
    SEGMENT_REPEAT_X edges — with premultiplied blending over the white page.  Reference image 116x108."""
    from webrender_b200 import gpu_types as G
    W, H = 116, 108
    black = (0.0, 0.0, 0.0, 1.0)
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    r, bw, bh = 40.0, 90.0, 80.0
    # (segment, task origin in the cache, segment rect relative to the border rect, adjacent-corner clip points)
    corners = [(G.SEGMENT_TOP_LEFT, (0, 0), (0.0, 0.0, r, r), (r, 0.0, 0.0, r)),
               (G.SEGMENT_TOP_RIGHT, (40, 0), (bw - r, 0.0, bw, r), (0.0, 0.0, r, r)),
               (G.SEGMENT_BOTTOM_RIGHT, (0, 40), (bw - r, bh - r, bw, bh), (0.0, r, r, 0.0)),
               (G.SEGMENT_BOTTOM_LEFT, (40, 40), (0.0, bh - r, r, bh), (r, r, 0.0, 0.0))]
    edges = [(G.SEGMENT_TOP, (80, 0), (r, 0.0, bw - r, 3.0)), (G.SEGMENT_BOTTOM, (80, 8), (r, bh - 3.0, bw - r, bh))]
    inst, segs = [], []
    for seg, org, srect, adj in corners:
        inst.append(G.border_instance(task_origin=(float(org[0]), float(org[1])), local_rect=(0.0, 0.0, r, r), color0=black,
                                      color1=black, segment=seg, style0=G.BORDER_STYLE_SOLID, style1=G.BORDER_STYLE_SOLID,
                                      do_aa=True, widths=(3.0, 3.0), radius=(r, r),
                                      clip_params=(adj[0], adj[1], 0.0, 0.0, adj[2], adj[3], 0.0, 0.0)))
        segs.append((srect, (0.0, 0.0, 1.0, 1.0), 2 | 512, (float(org[0]), float(org[1]), org[0] + r, org[1] + r)))
    for seg, org, srect in edges:
        inst.append(G.border_instance(task_origin=(float(org[0]), float(org[1])), local_rect=(0.0, 0.0, 8.0, 3.0), color0=black,
                                      color1=black, segment=seg, style0=G.BORDER_STYLE_SOLID, style1=G.BORDER_STYLE_SOLID,
                                      do_aa=True, widths=(8.0, 3.0), radius=(0.0, 0.0)))
        segs.append((srect, (0.0, 0.0, 8.0, 3.0), 2 | 4, (float(org[0]), float(org[1]), org[0] + 8.0, org[1] + 3.0)))
    # the border primitive: brush data (colour, background, stretch size = the border's size) + two blocks per segment
    blocks = [(1.0, 1.0, 1.0, 1.0), (0.0, 0.0, 0.0, 0.0), (bw, bh, 0.0, 0.0)]
    for srect, texel, _, _ in segs:
        blocks += [srect, texel]
    addr = t.push_gpu_cache(blocks)
    hdr = t.add_prim_header((10.0, 10.0, 10.0 + bw, 10.0 + bh), (-1e9, -1e9, 1e9, 1e9), 1, addr, 0, pic,
                            (4 | (1 << 16), 0, 65535, 0))
    draws = []
    for i, (_, _, flags, uv) in enumerate(segs):
        res = t.push_gpu_cache([uv, (0.0, 0.0, 0.0, 0.0)])
        draws.append(G.brush_instance(hdr, G.CLIP_TASK_EMPTY, i, 0, flags, res))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H),
                "cache": TextureDesc(abi.FMT_RGBA8, 128, 128, filter=abi.LINEAR)}
    p0 = [Target("cache", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0)),
                               Batch(abi.KIND_BORDER_SOLID, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA)])]
    p1 = [Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                                Batch(abi.KIND_BRUSH_IMAGE, np.stack(draws), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                      features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D, color=("cache", "", ""))])]
    return Frame(t.arrays(), textures, [p0, p1])


def solid_border_frame(size, borders, cache=(512, 512)):
    """Solid one-colour CSS borders as the frame builder draws them (border.rs:168-215 ensure_no_corner_overlap,
    654-898 create_border_segments, 1044-1241 corner / edge segments and their cache keys in app units, 1245-1297
    build_border_instances): per border four corner tasks (cs_border_solid, the adjacent corners' clips kept only
    where their radii reach into the task) and up to four 8-pixel edge tasks in the texture cache, then one Brush(Image)
    instance per segment (SEGMENT_RELATIVE | SEGMENT_TEXEL_RECT corners, SEGMENT_RELATIVE | SEGMENT_REPEAT_X/Y edges),
    premultiplied over the white page.  borders = [(rect, width, (tl, tr, br, bl) radii as (rx, ry), rgba)]."""
    from webrender_b200 import gpu_types as G
    f32 = np.float32
    W, H = size
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    pack = _ShelfPacker(cache[0], cache[1])
    inst, draws = [], []
    au = lambda v: float(f32(round(float(v) * 60.0) / 60.0))  # noqa: E731  (LayoutSizeAu round trip)
    for bi, (rect, width, radii, rgba) in enumerate(borders):
        bw, bh = f32(rect[2] - rect[0]), f32(rect[3] - rect[1])
        r = [[f32(v[0]), f32(v[1])] for v in radii]  # tl, tr, br, bl
        ratio = f32(1.0)
        for a_, b_, ext, k in ((0, 1, bw, 0), (3, 2, bw, 0), (0, 3, bh, 1), (1, 2, bh, 1)):
            sm = f32(r[a_][k] + r[b_][k])
            if ext > 0 and ext < sm:
                ratio = min(ratio, f32(ext / sm))
        if ratio < 1.0:
            r = [[f32(v[0] * ratio), f32(v[1] * ratio)] for v in r]
        r = [(au(v[0]), au(v[1])) for v in r]
        w = float(width)
        bw, bh = float(bw), float(bh)
        sz = [(max(v[0], w), max(v[1], w)) for v in r]  # local sizes tl, tr, br, bl
        tl, tr, br, bl = sz
        col = tuple(float(f32(c * rgba[3])) for c in rgba[:3]) + (float(rgba[3]),)
        segs = []  # (segment rect rel. to the border, texel rect, brush flags, task rect in the cache)

        def corner(seg, img, h_out, h_rad, h_keep, h_dflt, v_out, v_rad, v_keep, v_dflt, radius):
            cw, ch = img[2] - img[0], img[3] - img[1]
            tw, th = int(np.ceil(cw)), int(np.ceil(ch))
            at = pack.place(tw, th)
            ho, hr = (h_out, h_rad) if h_keep else (h_dflt, (0.0, 0.0))
            vo, vr = (v_out, v_rad) if v_keep else (v_dflt, (0.0, 0.0))
            cp = (round(ho[0] - img[0]), round(ho[1] - img[1]), float(np.ceil(hr[0])), float(np.ceil(hr[1])),
                  round(vo[0] - img[0]), round(vo[1] - img[1]), float(np.ceil(vr[0])), float(np.ceil(vr[1])))
            inst.append(G.border_instance(task_origin=(float(at[0]), float(at[1])), local_rect=(0.0, 0.0, float(tw), float(th)),
                                          color0=col, color1=col, segment=seg, style0=G.BORDER_STYLE_SOLID,
                                          style1=G.BORDER_STYLE_SOLID, do_aa=True, widths=(float(np.ceil(w)), float(np.ceil(w))),
                                          radius=(float(np.ceil(radius[0])), float(np.ceil(radius[1]))),
                                          clip_params=tuple(float(v) for v in cp)))
            segs.append((img, (0.0, 0.0, 1.0, 1.0), 2 | 512, (float(at[0]), float(at[1]), float(at[0] + tw), float(at[1] + th))))

        def edge(seg, img, vertical):
            if img[2] - img[0] <= 0.0 or img[3] - img[1] <= 0.0:
                return
            size = (w, 8.0) if vertical else (8.0, w)
            tw, th = int(np.ceil(size[0])), int(np.ceil(size[1]))
            at = pack.place(tw, th)
            inst.append(G.border_instance(task_origin=(float(at[0]), float(at[1])), local_rect=(0.0, 0.0, float(tw), float(th)),
                                          color0=col, color1=col, segment=seg, style0=G.BORDER_STYLE_SOLID,
                                          style1=G.BORDER_STYLE_SOLID, do_aa=True, widths=(float(tw), float(th)), radius=(0.0, 0.0)))
            segs.append((img, (0.0, 0.0, size[0], size[1]), 2 | (8 if vertical else 4),
                         (float(at[0]), float(at[1]), float(at[0] + tw), float(at[1] + th))))
        edge(G.SEGMENT_LEFT, (0.0, tl[1], w, bh - bl[1]), True)
        edge(G.SEGMENT_TOP, (tl[0], 0.0, bw - tr[0], w), False)
        edge(G.SEGMENT_RIGHT, (bw - w, tr[1], bw, bh - br[1]), True)
        edge(G.SEGMENT_BOTTOM, (bl[0], bh - w, bw - br[0], bh), False)
        i_tl, i_tr = (0.0, 0.0, tl[0], tl[1]), (bw - tr[0], 0.0, bw, tr[1])
        i_br, i_bl = (bw - br[0], bh - br[1], bw, bh), (0.0, bh - bl[1], bl[0], bh)
        corner(G.SEGMENT_TOP_LEFT, i_tl, (bw, 0.0), r[1], bw - r[1][0] < i_tl[2], (i_tl[2], i_tl[1]),
               (0.0, bh), r[3], bh - r[3][1] < i_tl[3], (i_tl[0], i_tl[3]), r[0])
        corner(G.SEGMENT_TOP_RIGHT, i_tr, (0.0, 0.0), r[0], 0.0 + r[0][0] > i_tr[0], (i_tr[0], i_tr[1]),
               (bw, bh), r[2], bh - r[2][1] < i_tr[3], (i_tr[2], i_tr[3]), r[1])
        corner(G.SEGMENT_BOTTOM_RIGHT, i_br, (0.0, bh), r[3], 0.0 + r[3][0] > i_br[0], (i_br[0], i_br[3]),
               (bw, 0.0), r[1], 0.0 + r[1][1] > i_br[1], (i_br[2], i_br[1]), r[2])
        corner(G.SEGMENT_BOTTOM_LEFT, i_bl, (bw, bh), r[2], bw - r[2][0] < i_bl[2], (i_bl[2], i_bl[3]),
               (0.0, 0.0), r[0], 0.0 + r[0][1] > i_bl[1], (i_bl[0], i_bl[1]), r[3])
        blocks = [(1.0, 1.0, 1.0, 1.0), (0.0, 0.0, 0.0, 0.0), (bw, bh, 0.0, 0.0)]
        for srect, texel, _, _ in segs:
            blocks += [tuple(float(v) for v in srect), texel]
        addr = t.push_gpu_cache(blocks)
        hdr = t.add_prim_header(tuple(float(v) for v in rect), (-1e9, -1e9, 1e9, 1e9), bi + 1, addr, 0, pic,
                                (4 | (1 << 16), 0, 65535, 0))
        for i, (_, _, flags, uv) in enumerate(segs):
            res = t.push_gpu_cache([uv, (0.0, 0.0, 0.0, 0.0)])
            draws.append(G.brush_instance(hdr, G.CLIP_TASK_EMPTY, i, 0, flags, res))
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H),
                "cache": TextureDesc(abi.FMT_RGBA8, cache[0], cache[1], filter=abi.LINEAR)}
    p0 = [Target("cache", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0)),
                               Batch(abi.KIND_BORDER_SOLID, np.stack(inst), blend=abi.BLEND_PREMULTIPLIED_ALPHA)])]
    p1 = [Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                                Batch(abi.KIND_BRUSH_IMAGE, np.stack(draws), blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                      features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D, color=("cache", "", ""))])]
    return Frame(t.arrays(), textures, [p0, p1])


BORDER_REFTESTS = {
    # wrench/reftests/border/<name>.yaml against its reference image: (image size, borders, allowed (max diff, pixels))
    # border-radii.yaml == border-radii.png, fuzzy(1,10): per-corner radii 16 / 8 on a width-10 border
    "border-radii": ((113, 119), [((10, 10, 100, 100), 10.0, ((16, 16), (8, 8), (16, 16), (8, 8)), (0.0, 0.0, 1.0, 1.0))], (1, 10)),
    # border-clamp-corner-radius.yaml == border-clamp-corner-radius.png: radii of 180 on 200-pixel boxes are scaled to fit
    "border-clamp-corner-radius": ((430, 230), [((0, 0, 200, 200), 10.0, ((180, 180),) * 4, (0.0, 0.0, 1.0, 1.0)),
                                                ((200, 0, 400, 200), 10.0, ((180, 180), (0, 0), (180, 180), (0, 0)),
                                                 (0.0, 0.0, 1.0, 1.0))], (0, 0)),
}


def reftest_clip_inverted_ellipse_frame():
    """wrench/reftests/clip/inverted-ellipse.yaml (== inverted-ellipse.png): a 225x150 red rect under a complex clip
    whose corner radii (112.5, 75) make it an ellipse "where the ratio of the corner size is inverted from the ratio of
    the primitive size".  Indirect path like config A; reference image 319x236."""
    spec = [((50, 50, 275, 200), (1.0, 0.0, 0.0, 1.0), ((112.5, 75.0),) * 4, 0)]
    return rounded_rects_frame(width=319, height=236, spec=spec, surface=(256, 256))


def reftest_border_frame(name):
    size, borders, _ = BORDER_REFTESTS[name]
    return solid_border_frame(size, borders)


def reftest_split_near_plane_frame():
    """wrench/reftests/split/near-plane.yaml (== near-plane.png, fuzzy(1,20); fuzzy-if(platform(swgl),128,39)): a
    600x600 rect of (255,0,0,0.5) in a stacking context rotated by rotate-x(-60) about its centre, inside a
    preserve-3d context with perspective 200 — "a single polygon intersecting the near plane".  Draw list
    (picture.rs Picture3DContext::In, batch.rs:2040-2080): the child picture is rasterised in its local space into a
    600x600 surface (one premultiplied Brush(Solid) = 128,0,0,128), the plane splitter hands back ONE polygon — the
    picture rect cut where it comes too close to the eye (w -> 0 at y = 300 + 200/sin(60) = 530.9; cut here at
    y = 500, which projects far below the 600-pixel viewport, so where exactly the cut lies cannot be seen) — and
    ps_split_composite draws it over the white page with premultiplied blending."""
    from webrender_b200.gpu_types import brush_instance, split_composite_instance, CLIP_TASK_EMPTY
    W = H = 600
    t = FrameTables()
    surf_task = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    # the wrench rotation sign: the bottom half comes towards the eye (it fills the width of the reference image)
    xf = t.add_transform(perspective_matrix(W, H, d=200.0, ry=0.0, rx=60.0), axis_aligned=False)
    color = (0.5, 0.0, 0.0, 0.5)
    addr = t.push_gpu_cache([color])
    hdr0 = t.add_prim_header((0.0, 0.0, float(W), float(H)), (-1e9, -1e9, 1e9, 1e9), 1, addr, 0, surf_task, (65535, 0, 0, 0))
    solid = brush_instance(hdr0, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)
    yc = 500.0
    poly_addr = t.push_gpu_cache([(0.0, 0.0, float(W), 0.0), (float(W), yc, 0.0, yc)])
    res = t.push_gpu_cache([(0.0, 0.0, float(W), float(H)), (0.0, 0.0, 0.0, 0.0),
                            (0.0, 0.0, 0.0, 1.0), (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0), (1.0, 1.0, 0.0, 1.0)])
    hdr = t.add_prim_header((0.0, 0.0, float(W), float(H)), (-1e9, -1e9, 1e9, 1e9), 1, 0, xf, pic, (res, 1, 0, CLIP_TASK_EMPTY))
    poly = split_composite_instance(hdr, poly_addr, 1, pic)
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H),
                "surface": TextureDesc(abi.FMT_RGBA8, W, H, filter=abi.LINEAR)}
    p0 = [Target("surface", ops=[Clear(color=(0.0, 0.0, 0.0, 0.0)),
                                 Batch(abi.KIND_BRUSH_SOLID, solid[None, :], blend=abi.BLEND_PREMULTIPLIED_ALPHA)])]
    p1 = [Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                                Batch(abi.KIND_SPLIT_COMPOSITE, poly[None, :], blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                      color=("surface", "", ""))])]
    return Frame(t.arrays(), textures, [p0, p1])


def reftest_box_shadow_suite_no_blur_frame():
    """wrench/reftests/boxshadow/box-shadow-suite-no-blur.yaml (== box-shadow-suite-no-blur.png): four rows of five box
    shadows without blur — outset, outset with border-radius 32, inset, inset with radius 32 — each with offsets (20,0),
    (0,-40), spread 30, and spread 30 + offset (50,-10); the first of a row (no offset, no spread) is rejected as
    invisible.  The frame builder's no-blur path (box_shadow.rs:331-401): outset = the shadow rect (box moved by the
    offset, inflated by the spread, radius r + spread when r > 0) under ClipOut of the box; inset = the box under
    ClipOut of the shadow rect (box moved, shrunk by the spread, radius max(r - spread, 0)).  Reference image 894x789."""
    red, green = (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0)
    spec = []
    cols = [(0, 0, 0), (20, 0, 0), (0, -40, 0), (0, 0, 30), (50, -10, 30)]
    for y, inset, r, col in ((50, False, 0, red), (250, False, 32, green), (450, True, 0, red), (650, True, 32, red)):
        for i, (ox, oy, sp) in enumerate(cols):
            if ox == 0 and oy == 0 and sp == 0:
                continue
            x = 50 + 150 * i
            box = (x, y, x + 100, y + 100)
            if not inset:
                sh = (box[0] + ox - sp, box[1] + oy - sp, box[2] + ox + sp, box[3] + oy + sp)
                spec.append((sh, col, float(r + sp if r > 0 else 0), 0, [(tuple(float(v) for v in box), float(r), 1)]))
            else:
                sh = (box[0] + ox + sp, box[1] + oy + sp, box[2] + ox - sp, box[3] + oy - sp)
                extra = [(tuple(float(v) for v in sh), float(max(r - sp, 0) if r > 0 else 0), 1)] if sh[2] > sh[0] and sh[3] > sh[1] else []
                spec.append((box, col, float(r), 0, extra))
    return rounded_rects_frame(width=894, height=789, spec=spec, surface=(1024, 1024))


def reftest_filter_blur_frame():
    """wrench/reftests/filters/filter-small-blur-radius.yaml: a 512x512 red rect at (100,100) in a stacking context with
    filter blur(2,2), on the 700x700 page of its reference image.  Draw list (picture.rs:5873-5938, render_task.rs
    new_blur): the picture surface = the rect inflated by ceil(2) * BLUR_SAMPLE_SCALE = 6 px (524x524 task, content
    origin (94,94)) drawn with an opaque Quad; std deviation 2 <= MAX_BLUR_STD_DEVIATION so no downscale: one vertical
    and one horizontal cs_blur COLOR_TARGET pass (blur region = the picture size); the result composited 1:1 by
    Brush(Image) with premultiplied blending."""
    from webrender_b200.gpu_types import blur_instance, brush_instance, CLIP_TASK_EMPTY
    t = FrameTables()
    W = H = 700
    inflate, std = 6.0, 2.0
    x0, y0, x1, y1 = 100.0 - inflate, 100.0 - inflate, 612.0 + inflate, 612.0 + inflate
    pw, ph = int(x1 - x0), int(y1 - y0)
    tile_task = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    pic_task = t.add_render_task((0.0, 0.0, float(pw), float(ph)), 1.0, (x0, y0))
    mid_task = t.add_render_task((0.0, 0.0, float(pw), float(ph)), 1.0, (0.0, 0.0))
    out_task = t.add_render_task((0.0, 0.0, float(pw), float(ph)), 1.0, (0.0, 0.0))
    rect = (100.0, 100.0, 612.0, 612.0)
    prim_f = t.add_quad_prim(rect, rect, (1.0, 0.0, 0.0, 1.0))
    prim_i = t.add_quad_header(0, 1)
    qi = quad_instance(prim_i, prim_f, QF_APPLY_DEVICE_CLIP, 0, PART_ALL, INVALID_SEGMENT_INDEX, pic_task)
    vert = blur_instance(mid_task, pic_task, 1, std, (float(pw), float(ph)))
    hori = blur_instance(out_task, mid_task, 0, std, (float(pw), float(ph)))
    addr = t.push_gpu_cache([(1.0, 1.0, 1.0, 1.0), (0.0, 0.0, 0.0, 0.0), (-1.0, -1.0, 0.0, 0.0)])
    res = t.push_gpu_cache([(0.0, 0.0, float(pw), float(ph)), (0.0, 0.0, 0.0, 0.0)])
    hdr = t.add_prim_header((x0, y0, x1, y1), (-1e9, -1e9, 1e9, 1e9), 1, addr, 0, tile_task, (4 | (1 << 16), 0, 65535, 0))
    comp = brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, res)
    textures = {"pic": TextureDesc(abi.FMT_RGBA8, pw, ph), "mid": TextureDesc(abi.FMT_RGBA8, pw, ph),
                "blurred": TextureDesc(abi.FMT_RGBA8, pw, ph), "target": TextureDesc(abi.FMT_RGBA8, W, H)}
    zero = (0.0, 0.0, 0.0, 0.0)
    return Frame(t.arrays(), textures, [
        [Target("pic", ops=[Clear(color=zero), Batch(abi.KIND_QUAD_TEXTURED, qi[None, :], blend=abi.BLEND_NONE)])],
        [Target("mid", ops=[Clear(color=zero), Batch(abi.KIND_BLUR, vert[None, :], features=abi.FEAT_COLOR_TARGET, color=("pic", "", ""))])],
        [Target("blurred", ops=[Clear(color=zero), Batch(abi.KIND_BLUR, hori[None, :], features=abi.FEAT_COLOR_TARGET, color=("mid", "", ""))])],
        [Target("target", ops=[Clear(color=(1.0, 1.0, 1.0, 1.0)),
                               Batch(abi.KIND_BRUSH_IMAGE, comp[None, :], blend=abi.BLEND_PREMULTIPLIED_ALPHA,
                                     features=abi.FEAT_ALPHA_PASS | abi.FEAT_TEXTURE_2D, color=("blurred", "", ""))])]])


def reftest_gradient_frame(which="linear"):
    """wrench/reftests/gradient/linear.yaml (four hard-stop bands), linear-reverse.yaml
    and linear-hard-stop.yaml as ONE Brush(LinearGradient) each on a 300x300 white
    page — the uncached brush path an `is_software` frame builder keeps."""
    from webrender_b200.gpu_types import brush_instance, build_gradient_table, CLIP_TASK_EMPTY
    W = H = 300
    red, green, blue, black = (1.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.0, 1.0), (0.0, 0.0, 1.0, 1.0), (0.0, 0.0, 0.0, 1.0)
    clear = (0.0, 0.0, 0.0, 0.0)
    r = (50.0, 50.0, 250.0, 250.0)
    blend = abi.BLEND_NONE
    if which == "linear":
        start, end = (0.0, 100.0), (200.0, 100.0)
        stops = [(0.0, red), (0.25, red), (0.25, green), (0.5, green), (0.5, blue), (0.75, blue), (0.75, black), (1.0, black)]
    elif which == "linear-reverse":
        start, end = (200.0, 100.0), (0.0, 100.0)
        stops = [(0.0, black), (0.25, black), (0.25, blue), (0.5, blue), (0.5, green), (0.75, green), (0.75, red), (1.0, red)]
    elif which in ("premultiplied-aligned", "premultiplied-angle"):
        # red -> transparent black -> green: stop colours are premultiplied when the table is
        # built, the brush goes to the alpha pass (premultiplied over the white page)
        start, end = ((0.0, 100.0), (200.0, 100.0)) if which.endswith("aligned") else ((0.0, 0.0), (200.0, 200.0))
        stops = [(0.0, red), (0.5, clear), (1.0, green)]
        blend = abi.BLEND_PREMULTIPLIED_ALPHA
    elif which == "linear-stops":
        r = (0.0, 0.0, 200.0, 200.0)
        start, end = (0.0, 100.0), (200.0, 100.0)
        stops = [(0.0, red), (0.5, green), (1.0, blue)]
    else:
        # yaml: end (0,100), stops [0 blue, 0.5 red, 0.5 green].  The display-list builder
        # normalises stops to [0, 1] and moves the end point accordingly
        # (GradientBuilder::normalize, webrender_api/src/gradient_builder.rs)
        start, end = (0.0, 0.0), (0.0, 50.0)
        stops = [(0.0, blue), (1.0, red), (1.0, green)]
    t = FrameTables()
    pic = t.add_render_task((0.0, 0.0, float(W), float(H)), 1.0, (0.0, 0.0))
    lut = t.push_gpu_buffer_f(list(build_gradient_table(stops)))
    addr = t.push_gpu_cache([(start[0], start[1], end[0], end[1]), (0.0, 200.0, 200.0, 0.0)])
    hdr = t.add_prim_header(r, (-1e9, -1e9, 1e9, 1e9), 1, addr, 0, pic, (lut, 0, 0, 0))
    inst = np.stack([brush_instance(hdr, CLIP_TASK_EMPTY, 0xFFFF, 0, 0, 0)])
    textures = {"target": TextureDesc(abi.FMT_RGBA8, W, H)}
    ops = [Clear(color=(1.0, 1.0, 1.0, 1.0)),
           Batch(abi.KIND_BRUSH_LINEAR_GRADIENT, inst, blend=blend,
                 features=abi.FEAT_ALPHA_PASS if blend != abi.BLEND_NONE else 0)]
    return Frame(t.arrays(), textures, [[Target("target", ops=ops)]])
