"""The raster stage in every work-item shape, the binner at its segment boundaries and the depth cull over
the whole float range, against the CPU oracle (-m gpu, except the sweep arithmetic test).

Three parts of the device code take a different path depending on the size or the values of a flush:

- Work items (raster_body in dtr_kernels.cu, raster_opaque_kernel in dtr_deferred.cuh).  A busy 64x32 tile
  is two 32x32 region items, except the last nSmall busy tiles, which are four 32x16, eight 32x8 or sixteen
  32x4 items.  The cut depends on the busy tile count nBusy, on S = smallTilesMin (half the raster stage's
  resident warps: it comes from the occupancy query and differs per stage and with ids on or off) and on
  fewPrims (list entries <= 64 per busy tile).  The sweep renders batches of N frames whose tiles are all
  busy, N growing geometrically, so that every S of 1 to 6 resident CTAs per SM meets every regime.
- Bin segments: a flush whose largest frame has more than BIN_SEG = 8192 primitives is binned per
  (tile, segment), with one segment count shared by every frame of the flush.
- The region and sub-block depth cull (setup's depth bound zU, depth_key, the region minimum) must stay
  conservative for every float a depth plane or a vertex can hold.

Every check compares colour and depth bit for bit, the SetPixels counter and, with ids on, the id planes.
"""
import functools
import os
import re

import numpy as np
import pytest

from dtrenderer_b200 import api, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dtrenderer_b200", "csrc")

TILE_W, TILE_H = 64, 32
MAX_CTAS_PER_SM = 6            # the sweep covers S = 2 * sms * k for k = 1 .. 6 resident raster CTAs per SM
SIZES = ((600, 340), (609, 323))  # last tile column 24 px / 33 px wide, last tile row 20 px / 3 px high
K = 3                          # distinct scenes cycled over the frames of a batch
FULL_SHAPES = {(32, 4), (32, 8), (32, 16), (32, 32)}
DENSE_SHAPES = {(32, 16), (32, 32)}  # many list entries per tile: small tiles are always 32x16 items
# raster paths: (content, opaque-stage setting, what last_pass_stage() must report)
PATHS = {"single": ("blend", api.OPAQUE_ONE_KERNEL, api.OPAQUE_SINGLE_KERNEL),
         "one_kernel": ("opaque", api.OPAQUE_ONE_KERNEL, api.OPAQUE_ONE_KERNEL),
         "two_kernels": ("opaque", api.OPAQUE_TWO_KERNELS, api.OPAQUE_TWO_KERNELS)}


# ---- the item arithmetic of the raster kernels, restated ---------------------------------------------
def _source_constant(name):
    for f in ("dtr_records.h", "dtr_deferred.cuh", "dtr_kernels.cu"):
        with open(os.path.join(CSRC, f)) as fh:
            m = re.search(r"constexpr\s+int\s+" + name + r"\s*=\s*(\d+)\s*;", fh.read())
        if m:
            return int(m.group(1))
    raise AssertionError(f"{name} not found in {CSRC}")


def tiles_per_frame(w, h):
    return -(-w // TILE_W) * -(-h // TILE_H)


def sweep(tpf, sms):
    """Batch sizes N: N * tpf starts below sms, grows by at most 2x per step and ends above 2 * 12 * sms."""
    top = 2 * 2 * MAX_CTAS_PER_SM * sms
    ns = [max(1, (sms - 1) // tpf)]
    while ns[-1] * tpf <= top:
        ns.append(min(2 * ns[-1], top // tpf + 1))
    return ns


def item_shapes(n_busy, s, few, small_percent=5):
    """The (width, height) of the region items raster_body / raster_opaque_kernel cut n_busy busy tiles into."""
    n_small = min(n_busy, max(n_busy * small_percent // 100, s))
    n_big = n_busy - n_small
    shift = 2 if not few else (4 if 2 * n_busy < s else (3 if n_busy < s else 2))
    return ({(32, 32)} if n_big else set()) | ({(32, 32 >> (shift - 1))} if n_small else set())


def regime(n_busy, s):
    return "thin" if 2 * n_busy < s else ("eighth" if n_busy < s else ("big" if n_busy > s else "edge"))


@pytest.mark.parametrize("sms", [148, 132, 160])
def test_sweep_arithmetic_reaches_every_item_shape(sms):
    """CPU: for every frame size and density the sweep uses, its batch sizes meet every regime (2*nBusy < S,
    S/2 <= nBusy < S, nBusy > S) and every item shape for every S of 1 to MAX_CTAS_PER_SM resident CTAs per
    SM.  The per-SM CTA counts of the raster kernels' __launch_bounds__ are read from the sources, and raising
    one beyond what the sweep covers fails here.  They are the residency the kernels are built for, not a cap:
    the occupancy query decides S at run time, and could report more CTAs per SM than these if a kernel's
    resources shrank, which this test cannot see."""
    caps = {n: _source_constant(n) for n in ("RASTER_CTAS_PER_SM", "VIS_CTAS_PER_SM", "VIS_IDS_CTAS_PER_SM")}
    assert all(1 <= c <= MAX_CTAS_PER_SM for c in caps.values()), caps
    small_percent = _source_constant("RASTER_SMALL_PERCENT")
    warps = _source_constant("RASTER_THREADS") // 32
    for w, h in SIZES:
        tpf = tiles_per_frame(w, h)
        ns = sweep(tpf, sms)
        assert ns[0] * tpf < sms and ns[-1] * tpf > 2 * 2 * MAX_CTAS_PER_SM * sms
        assert all(b <= 2 * a for a, b in zip(ns, ns[1:]))
        # smallTilesMin = resident CTAs * warps per CTA / 2, resident = sms * (1 .. cap)
        for s in range(warps * sms // 2, warps * sms * MAX_CTAS_PER_SM // 2 + 1):
            assert {"thin", "eighth", "big"} <= {regime(n * tpf, s) for n in ns}, (w, h, s)
            for few, want in ((True, FULL_SHAPES), (False, DENSE_SHAPES)):
                got = set().union(*(item_shapes(n * tpf, s, few, small_percent) for n in ns))
                assert got == want, (w, h, s, few, got)
    # the batch of the depth-domain test reaches 32x32 regions for every such S
    n = depth_batch(sms)
    assert item_shapes(n * tiles_per_frame(*DEPTH_SIZE), 2 * sms * MAX_CTAS_PER_SM, False) >= {(32, 32)}


# ---- shared helpers ----------------------------------------------------------------------------------
def _port(w, h):
    from id_reference import IdOracle
    o = IdOracle(w, h)
    o.reset_counters()
    return o


def _renderer(w, h, frames, ids, stage=api.OPAQUE_ONE_KERNEL):
    r = api.Renderer(w, h, frames, 0)
    r.set_opaque_stage(stage)
    if ids:
        r.set_id_output(True)
    return r


def _oracle_frame(w, h, ops, planes=None):
    """Render ops in the port oracle: (colour, depth, ids, SetPixels)."""
    o = _port(w, h)
    if planes is not None:
        o.upload(*planes)
    scenes.replay(ops, o)
    return o.color().copy(), o.zbuffer().copy(), o.ids().copy(), o.counters()[0]


def _check_frames(r, want, ids):
    """want[f] = (colour, depth, ids, SetPixels) of frame f; the device counter must be their sum."""
    from test_gpu_parity import _assert_same
    for f, (co, zo, _, _) in enumerate(want):
        col, z = r.end_frame(f)
        try:
            _assert_same(col, z, co, zo)
        except AssertionError as e:
            raise AssertionError(f"frame {f} of {len(want)}: {e}") from None
    if ids:
        got = r.read_ids(0, len(want))
        for f, (_, _, io, _) in enumerate(want):
            assert np.array_equal(got[f], io), f"frame {f} of {len(want)}: ids differ on {(got[f] != io).sum()} px"
    assert r.stats()["setPixels"] == sum(w[3] for w in want)


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _quad(x0, y0, x1, y1, z, col=(0.3, 0.3, 0.3, 1.0)):
    p = np.array([[x0, y0, z, x1, y0, z, x1, y1, z], [x0, y0, z, x1, y1, z, x0, y1, z]], np.float32)
    return ("triangles", dict(p=p, color=np.tile(np.asarray(col, np.float32), (2, 1)),
                              transform=scenes.DEFAULT_TRIANGLE_TRANSFORM))


# ---- A. batch-size sweep across the item shapes -------------------------------------------------------
def _opaque_ops(rng, w, h, calls):
    """Opaque triangles only (integer-vertex batches, transformed triangles, textured triangles, meshes)."""
    tex = scenes.random_texture(int(rng.integers(2, 40)), int(rng.integers(2, 40)), int(rng.integers(1 << 16)), opaque=True)
    mesh = scenes.uv_sphere(14, 7)
    ops = []
    for i in range(calls):
        kind = int(rng.integers(0, 4))
        col = (*rng.random(3).tolist(), 1.0)
        if kind == 0:
            n = int(rng.integers(1, 30))
            c = rng.integers(-10, [w + 10, h + 10], (n, 1, 2))
            p = np.concatenate([c + rng.integers(-30, 31, (n, 3, 2)), rng.uniform(0, 255, (n, 3, 1))], 2).astype(np.float32)
            cols = rng.random((n, 4)).astype(np.float32)
            cols[:, 3] = 1.0
            ops.append(("triangles", dict(p=p.reshape(n, 9), color=cols, transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
        elif kind == 1:
            p = np.concatenate([rng.uniform(-40, [w + 40, h + 40], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
            tr = scenes.transform7(float(rng.uniform(-3, 3)), tuple(rng.random(3)), (float(rng.uniform(0.4, 2)), float(rng.uniform(0.4, 2)), 1.0))
            ops.append(("triangle", dict(p=p.reshape(-1), color=col, transform=tr)))
        elif kind == 2:
            p = np.concatenate([rng.integers(-20, [w + 20, h + 20], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
            ops.append(("textured_triangle", dict(p=p.reshape(-1), uv=(rng.random(6) * 0.999).astype(np.float32), tex=tex,
                                                  color=col, transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
        elif i % 4 == 0:
            view = scenes.view_transforms(4096)[int(rng.integers(0, 4096))]
            ops.append(("mesh", dict(mesh=mesh, tex=tex, light_mode=int(rng.integers(0, 3)), light_vector=(1, -1, 1),
                                     light_color=(1, 1, 1, 1), pos=(0.1, 0.0, 0.0), transform=view)))
    return ops


@functools.lru_cache(maxsize=None)
def _sweep_scene(size, density, content, k, seed=0):
    """Scene k of a (size, density, content, seed) family and its oracle frame.  Every scene starts with a
    clear and a full-frame quad, so that every tile of every frame is busy."""
    w, h = size
    rng = np.random.default_rng([w, h, density == "dense", content == "opaque", k] + ([seed] if seed else []))
    ops = [("clear", dict(rgb=tuple(rng.random(3).tolist()))), _quad(-2, -2, w + 2, h + 2, float(rng.uniform(5, 40)))]
    if density == "dense":
        # ~8k small integer-vertex triangles: more than 64 list entries per tile
        p, col = scenes.small_triangles(w, h, 8000, seed=int(rng.integers(1 << 30)))
        if content == "blend":
            col[rng.random(len(col)) < 0.25, 3] = 0.5
        ops.append(("triangles", dict(p=p, color=col, transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    elif content == "blend":
        from test_gpu_ids import _fuzz_ops
        ops += [op for op in _fuzz_ops(100 + 10 * k + (w & 7) + 1000 * seed, size)[1:70] if op[0] != "flush"]
    else:
        ops += _opaque_ops(rng, w, h, 40)
    return ops, _oracle_frame(w, h, ops)


@pytest.mark.parametrize("ids", [False, True], ids=["ids_off", "ids_on"])
@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("density", ["sparse", "dense"])
@pytest.mark.parametrize("size", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
@pytest.mark.gpu
def test_batch_sweep_equals_oracle(built, size, density, path, ids):
    """Batches of N frames in one flush, N swept from one frame (32x4 / 32x8 items, or 32x16 when dense) to
    more busy tiles than 2 * 12 * SMs (32x32 regions, the 512-view benchmark shape).  Frames cycle K scenes;
    each device frame equals its scene's oracle frame, and the counter the sum of theirs."""
    check_sweep(size, density, path, ids)


def check_sweep(size, density, path, ids, seed=0):
    """The batch sweep of one (size, density, raster path, ids) combination (also run by tools/fuzz_soak.py)."""
    content, stage, want_stage = PATHS[path]
    w, h = size
    tpf = tiles_per_frame(w, h)
    refs = [_sweep_scene(size, density, content, k, seed) for k in range(K)]
    for n in sweep(tpf, _sms()):
        r = _renderer(w, h, n, ids, stage)
        for f in range(n):
            r.begin_frame(f)
            scenes.replay(refs[f % K][0], r)
        r.flush()
        assert r.last_pass_stage() == want_stage, (n, r.last_pass_stage())
        entries, n_busy = r.stats()["listEntries"], n * tpf
        assert (entries <= 64 * n_busy) == (density == "sparse"), (n, entries, n_busy)
        try:
            _check_frames(r, [refs[f % K][1] for f in range(n)], ids)
        except AssertionError as e:
            raise AssertionError(f"batch of {n} frames ({n_busy} busy tiles): {e}") from None
        r.close()


# ---- B. bin segments ----------------------------------------------------------------------------------
SEG_SIZE = (300, 170)
SEG_COUNTS = (0, 1, 8191, 8192, 8193, 16385)   # triangles per frame: segs = 3, most segments empty
SEG_EDGES = (2048, 4096, 6144, 8191, 8192, 8193, 12288, 16384)
ROTATED = scenes.transform7(0.05, (0.5, 0.5, 0.5), (1.01, 0.99, 1.0))  # transformed (inexact) triangles


@functools.lru_cache(maxsize=None)
def _segment_frames(opaque):
    """One op list and oracle frame per SEG_COUNTS entry.  Triangle batches alternate between exact
    (integer-vertex) and rotated; a chunk edge sits on every segment boundary.  Unless opaque: frame 3 has a
    rectangle and a bitmap at primitive positions 8191 and 8192, and frame 4 is partly translucent."""
    w, h = SEG_SIZE
    rng = np.random.default_rng(8192 + opaque)
    tex = scenes.random_texture(13, 9, 5, opaque=False)
    frames = []
    for i, n in enumerate(SEG_COUNTS):
        ops = [("clear", dict(rgb=tuple(rng.random(3).tolist())))]
        p, col = scenes.small_triangles(w, h, n, seed=300 + i, max_edge=20)
        if not opaque and i == 4:
            col[rng.random(n) < 0.5, 3] = np.float32(0.6)
        edges = [0] + [e for e in SEG_EDGES if e < n] + [n]
        for j, (a, b) in enumerate(zip(edges[:-1], edges[1:])):
            if not opaque and i == 3 and a == 8191:
                ops.append(("rectangle", dict(mn=(20.0, 30.0), mx=(170.0, 120.0), color=(0.9, 0.2, 0.1, 0.7), transform=scenes.DEFAULT_TRANSFORM)))
                ops.append(("bitmap", dict(tex=tex, pos=(90.0, 60.0), transform=scenes.transform7(0.4, (0.5, 0.5, 0), (3, 3, 1)), color=(1, 1, 1, 0.8))))
            ops.append(("triangles", dict(p=p[a:b], color=col[a:b], transform=ROTATED if j % 2 else scenes.DEFAULT_TRIANGLE_TRANSFORM)))
        frames.append((ops, _oracle_frame(w, h, ops)))
    return frames


@pytest.mark.gpu
@pytest.mark.parametrize("ids", [False, True], ids=["ids_off", "ids_on"])
def test_segment_boundaries_in_one_flush(built, ids):
    """Frames of 0, 1, 8191, 8192, 8193 and 16385 triangles in one flush (three segments, most of them
    empty), with blits at positions 8191 and 8192 and translucent content across a boundary; then the same
    counts all opaque through both deferred forms.  Ids above 8192 check the per-item triangle base."""
    w, h = SEG_SIZE
    runs = [(False, api.OPAQUE_ONE_KERNEL, api.OPAQUE_SINGLE_KERNEL), (True, api.OPAQUE_ONE_KERNEL, api.OPAQUE_ONE_KERNEL),
            (True, api.OPAQUE_TWO_KERNELS, api.OPAQUE_TWO_KERNELS)]
    for opaque, stage, want_stage in runs:
        frames = _segment_frames(opaque)
        r = _renderer(w, h, len(frames), ids, stage)
        for f, (ops, _) in enumerate(frames):
            r.begin_frame(f)
            scenes.replay(ops, r)
        r.flush()
        assert r.last_pass_stage() == want_stage
        _check_frames(r, [ref for _, ref in frames], ids)
        if ids:
            assert r.read_ids(len(frames) - 1, 1).max() > 2 * 8192  # triangles of the third segment are visible
        r.close()


@pytest.mark.gpu
def test_segment_count_changes_between_flushes(built):
    """The same frames recorded over two flushes, split where the segment count changes (1, then 2): the
    16385-triangle frame continues in the second flush (ids number on across it)."""
    w, h = SEG_SIZE
    frames = _segment_frames(False)
    last = len(frames) - 1
    ops5 = frames[last][0]
    cut = 1 + sum(1 for e in SEG_EDGES if e <= 8191)     # clear + the batches that end at or before 8191
    r = _renderer(w, h, len(frames), True)
    for f in (0, 1, 2):
        r.begin_frame(f)
        scenes.replay(frames[f][0], r)
    r.begin_frame(last)
    scenes.replay(ops5[:cut], r)
    r.flush()                                             # largest frame: 8191 primitives -> one segment
    for f in (3, 4):
        r.begin_frame(f)
        scenes.replay(frames[f][0], r)
    r.set_target(last)
    scenes.replay(ops5[cut:], r)
    r.flush()                                             # 8194 -> two segments
    _check_frames(r, [ref for _, ref in frames], True)


# ---- C. depth domain of the cull ----------------------------------------------------------------------
DEPTH_SIZE = (320, 192)   # 5 x 6 tiles, 10 x 6 regions of 32x32
F32 = np.float32
SPECIAL_BITS = np.array([0x00000000, 0x80000000, 0x00000001, 0x80000001, 0x7F7FFFFF, 0xFF7FFFFF,
                         0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000, 0x7FC12345], np.uint32)
SPECIAL = SPECIAL_BITS.view(np.float32)
Z_TIE = F32(100.0)
R_INF = (224, 128)         # a 32x32 region clear of the frame's last row and column (triangles never draw those)
VERTEX_Z = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1e38, -1e38, 3.4028235e38, -3.4028235e38,
                     np.inf, -np.inf, np.nan], np.float32)


def depth_batch(sms):
    """Frames in the batch of the depth-domain test: more busy tiles than 2 * 12 * SMs."""
    return 2 * 2 * MAX_CTAS_PER_SM * sms // tiles_per_frame(*DEPTH_SIZE) + 1


def _fragments(p, w, h):
    """float32 model of the oracle / kernel for an integer-vertex triangle: (x, y, z) of its covered pixels,
    z = (z1 + bB*dz2) + bC*dz3 with bB = e2 * (1/area), bC = e3 * (1/area), in that operation order."""
    (x1, y1, z1), (x2, y2, z2), (x3, y3, z3) = np.asarray(p, np.float32).reshape(3, 3)
    minx, miny = int(max(0, min(x1, x2, x3))), int(max(0, min(y1, y2, y3)))
    maxx, maxy = int(min(max(x1, x2, x3), w - 1)), int(min(max(y1, y2, y3), h - 1))
    X, Y = np.meshgrid(np.arange(minx, maxx, dtype=F32), np.arange(miny, maxy, dtype=F32))

    def ef(ax, ay, bx, by, cx, cy):
        return ((bx - ax) * (cy - ay)) - ((by - ay) * (cx - ax))
    e1, e2, e3 = ef(x2, y2, x3, y3, X, Y), ef(x3, y3, x1, y1, X, Y), ef(x1, y1, x2, y2, X, Y)
    sx, sy = F32(minx), F32(miny)
    area = (ef(x2, y2, x3, y3, sx, sy) + ef(x3, y3, x1, y1, sx, sy)) + ef(x1, y1, x2, y2, sx, sy)
    cov = (e1 >= 0) & (e2 >= 0) & (e3 >= 0)
    if area == 0 or not cov.any():
        return np.empty(0, int), np.empty(0, int), np.empty(0, F32)
    inv = F32(1) / area
    z = (z1 + (e2 * inv) * (z2 - z1)) + (e3 * inv) * (z3 - z1)
    return X[cov].astype(int), Y[cov].astype(int), z[cov].astype(F32)


@functools.lru_cache(maxsize=None)
def _overshoot_triangle():
    """A small integer-vertex triangle one of whose fragments rounds ABOVE its largest vertex depth: drawn
    over a depth that holds that vertex depth, the fragment must pass.  The search also asks that setup's
    unpadded bound zV = max(z1, z1 + dz2, z1 + dz3) be no larger than that vertex depth (z1 far below,
    z2 == z3: z1 + dz2 rounds down), so that only the bound's rounding margin keeps the cull from dropping
    the fragment."""
    rng = np.random.default_rng(11)
    for _ in range(20000):
        z = rng.choice([-1, 1], 3) * rng.random(3) * 2.0 ** rng.integers(-20, 20, 3)
        p = np.concatenate([rng.integers(0, 32, (3, 2)), z[:, None]], 1).astype(F32)
        p[2, 2] = p[1, 2]
        zs = p[:, 2]
        with np.errstate(all="ignore"):
            x, y, zf = _fragments(p, 64, 64)
            zv = max(zs[0], zs[0] + (zs[1] - zs[0]), zs[0] + (zs[2] - zs[0]))
        above = zf > zs.max()
        if above.any() and zv <= zs.max():
            return p, int(x[above][0]), int(y[above][0]), F32(zf[above][0])
    raise AssertionError("no overshooting fragment found")


def _overshoot_floor():
    """The overshoot triangle's largest vertex depth: the depth under it before it is drawn."""
    return _overshoot_triangle()[0][:, 2].max()


def overshoot_pixel():
    """(x, y, z) of the overshooting fragment in a DEPTH_SIZE frame (the triangle sits in the last region)."""
    _, px, py, zf = _overshoot_triangle()
    return px + DEPTH_SIZE[0] - 32, py + DEPTH_SIZE[1] - 32, zf


def _depth_plane(rng, w, h):
    """Finite depths around the triangles' range, with the special values as whole 32x32 regions, whole 8x4
    sub-blocks and single pixels, and regions at Z_TIE and one ulp either side of it.  R_INF holds FLT_MAX."""
    z = rng.uniform(-300, 300, (h, w)).astype(F32)
    regions = [(ry, rx) for ry in range(h // 32) for rx in range(w // 32) if (rx * 32, ry * 32) != R_INF]
    order = rng.permutation(len(regions) - 1)                        # the last region is the overshoot's
    fills = list(SPECIAL) + [Z_TIE, np.nextafter(Z_TIE, F32(np.inf)), np.nextafter(Z_TIE, F32(-np.inf))]
    for v, i in zip(fills, order):
        ry, rx = regions[i]
        z.view(np.uint32)[ry * 32:ry * 32 + 32, rx * 32:rx * 32 + 32] = F32(v).view(np.uint32)
    for v in SPECIAL:
        for _ in range(6):
            sy, sx = int(rng.integers(0, h // 4)), int(rng.integers(0, w // 8))
            z.view(np.uint32)[sy * 4:sy * 4 + 4, sx * 8:sx * 8 + 8] = F32(v).view(np.uint32)
        ys, xs = rng.integers(0, h, 12), rng.integers(0, w, 12)
        z.view(np.uint32)[ys, xs] = F32(v).view(np.uint32)
    z[h - 32:, w - 32:] = _overshoot_floor()                         # the first look already sees the floor
    z[R_INF[1]:R_INF[1] + 32, R_INF[0]:R_INF[0] + 32] = np.finfo(F32).max
    return z


def _depth_ops(rng, w, h, opaque):
    """Triangles whose bounding boxes each stay inside one 64x32 tile but span both of its regions (so that
    ~50 of them pass every region, more than 8 groups of 6, and a tile list stays under 64 entries), with
    vertex depths drawn from finite values, the tie depth and its neighbours, signed zeros, denormals,
    +-1e38 (the bound zU overflows to inf), +-FLT_MAX, +-inf and NaN, and gradients from -1e38 to 1e38;
    every other batch is rotated (inexact).  The last region gets a floor at the overshoot triangle's
    largest vertex depth, eight hidden triangles (the cull takes the region and sub-block minima only
    between groups of GROUP = 6 hits, so these make it look at the floor, in 32x4 items as well as in
    32x32 regions) and the triangle itself.  R_INF
    gets a floor at FLT_MAX, eight hidden triangles and a triangle with vertex depths (1, inf, inf): its
    inner fragments are inf and pass, although the region minimum FLT_MAX is the key just below inf."""
    tiles = [(tx, ty) for ty in range(h // 32) for tx in range(w // 64)]
    n = 50 * len(tiles)
    t = np.array([tiles[i % len(tiles)] for i in range(n)])
    x = t[:, :1] * 64 + rng.integers(2, 62, (n, 3))
    x[:, 0], x[:, 1] = t[:, 0] * 64 + rng.integers(2, 24, n), t[:, 0] * 64 + rng.integers(40, 62, n)
    y = t[:, 1:] * 32 + rng.integers(2, 30, (n, 3))
    kind = rng.integers(0, 6, n)
    z = rng.uniform(-300, 300, (n, 3)).astype(F32)
    z[kind == 1] = Z_TIE
    z[kind == 2] = rng.choice([np.nextafter(Z_TIE, F32(np.inf)), np.nextafter(Z_TIE, F32(-np.inf))], ((kind == 2).sum(), 1))
    z[kind == 3] = rng.choice(VERTEX_Z, ((kind == 3).sum(), 3))
    z[kind == 4] = rng.choice(np.array([-1e38, 0.0, 1e38], F32), ((kind == 4).sum(), 3))
    z[kind == 5] = rng.choice(SPECIAL, ((kind == 5).sum(), 3))
    p = np.stack([x, y, z], 2).astype(F32).reshape(n, 9)
    reserved = ((x.max(1) >= w - 32) & (y.max(1) >= h - 32)) | \
        ((x.max(1) >= R_INF[0]) & (x.min(1) < R_INF[0] + 32) & (y.max(1) >= R_INF[1]) & (y.min(1) < R_INF[1] + 32))
    p = p[~reserved]                                                 # keep the reserved regions free
    col = rng.random((len(p), 4)).astype(F32)
    col[:, 3] = 1.0 if opaque else np.where(rng.random(len(p)) < 0.3, F32(0.5), F32(1.0))
    ops = []
    for j, a in enumerate(range(0, len(p), 97)):
        ops.append(("triangles", dict(p=p[a:a + 97], color=col[a:a + 97], transform=ROTATED if j % 2 else scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    x0, y0 = R_INF
    ops.append(_quad(x0, y0, x0 + 32, y0 + 32, np.finfo(F32).max))
    # hidden triangles whose bounding boxes span the region's full height: thin items see them too
    hid = np.array([[x0 + 2 + 3 * i, y0, 0, x0 + 28, y0 + 16, 0, x0 + 2 + i, y0 + 31, 0] for i in range(8)], F32)
    ops.append(("triangles", dict(p=hid, color=np.tile(np.array([0.1, 0.9, 0.1, 1.0], F32), (8, 1)), transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    inf_tri = np.array([[x0 + 3, y0 + 3, 1.0, x0 + 29, y0 + 6, np.inf, x0 + 12, y0 + 29, np.inf]], F32)
    ops.append(("triangles", dict(p=inf_tri, color=np.array([[0.2, 0.3, 0.9, 1.0]], F32), transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    q, _, _, _ = _overshoot_triangle()
    q = q + np.array([w - 32, h - 32, 0], F32)
    ops.append(_quad(w - 32, h - 32, w, h, float(_overshoot_floor())))
    ops.append(("triangles", dict(p=hid + np.array([w - 32 - x0, h - 32 - y0, -1000.0] * 3, F32),
                                  color=np.tile(np.array([0.1, 0.9, 0.1, 1.0], F32), (8, 1)), transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    ops.append(("triangles", dict(p=q.reshape(1, 9), color=np.array([[0.9, 0.8, 0.1, 1.0]], F32), transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    return ops


@functools.lru_cache(maxsize=None)
def _depth_scene(k, uploaded):
    w, h = DEPTH_SIZE
    rng = np.random.default_rng([7, k, uploaded])
    if uploaded:
        planes = (rng.integers(0, 1 << 24, (h, w)).astype(np.uint32), _depth_plane(rng, w, h))
        ops = _depth_ops(rng, w, h, opaque=False)
    else:
        planes, ops = None, [("clear", dict(rgb=tuple(rng.random(3).tolist())))] + _depth_ops(rng, w, h, opaque=True)
    ref = _oracle_frame(w, h, ops, planes)
    # the overshooting fragment passed the depth of its own largest vertex
    gx, gy, zf = overshoot_pixel()
    assert ref[1][gy, gx] == zf and zf > _overshoot_floor(), (ref[1][gy, gx], zf)
    assert np.isposinf(ref[1][R_INF[1] + 12, R_INF[0] + 14])        # an inf fragment passed FLT_MAX
    return ops, planes, ref


@pytest.mark.gpu
@pytest.mark.parametrize("batch", ["one_frame", "batch"])
@pytest.mark.parametrize("target", ["uploaded", "cleared_one_kernel", "cleared_two_kernels"])
def test_depth_cull_over_the_float_range(built, target, batch):
    """Uploaded depth planes full of +-0, denormals, +-FLT_MAX, +-inf and NaNs (single-kernel stage), and
    cleared frames (deferred stage), under exact and rotated triangles with extreme and non-finite vertex
    depths: one frame (thin items) and a batch large enough for 32x32 regions, ids on."""
    w, h = DEPTH_SIZE
    uploaded = target == "uploaded"
    stage = api.OPAQUE_TWO_KERNELS if target.endswith("two_kernels") else api.OPAQUE_ONE_KERNEL
    n = 1 if batch == "one_frame" else depth_batch(_sms())
    refs = [_depth_scene(k, uploaded) for k in range(min(K, n))]
    r = _renderer(w, h, n, True, stage)
    for f in range(n):
        ops, planes, _ = refs[f % len(refs)]
        if planes is not None:
            r.begin_frame(f, color=planes[0], z=planes[1])
        else:
            r.begin_frame(f)
        scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == (api.OPAQUE_SINGLE_KERNEL if uploaded else stage)
    if n == 1:
        assert r.stats()["listEntries"] <= 64 * tiles_per_frame(w, h)  # few primitives: the thinnest items
    # the two placed cases first, so that a failure names the cull decision that went wrong
    gx, gy, zf = overshoot_pixel()
    for f in range(n):
        z = r.end_frame(f)[1]
        assert z[gy, gx] == zf, f"frame {f}: the fragment above its largest vertex depth was culled ({z[gy, gx]!r})"
        assert np.isposinf(z[R_INF[1] + 12, R_INF[0] + 14]), f"frame {f}: the inf fragment over FLT_MAX was culled"
    _check_frames(r, [refs[f % len(refs)][2] for f in range(n)], True)
