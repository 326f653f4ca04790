"""Triangles far beyond the frame and at the limits of the exact-edge rule in every raster stage, against the CPU
oracle (the classification model and its constructions run without a GPU; the rest is -m gpu).

setup_kernel sorts every triangle into one of two classes, and the raster stage trusts that choice:

- EXACT (PF_EXACT): integer vertices, every edge-function value the raster kernels can meet below 2^24 (the
  per-edge bound |e0| + w|dx| + h|dy| over the clipped bbox grown by one 8x4 sub-block), no start value of -0,
  and |E1 + E2 + E3| below 2^24.  These get int32 edges, direct per-pixel evaluation, a depth bound for the
  region cull and, in the general raster kernel's fragment queue, E1 recovered as (sum - E2) - E3.
- INEXACT: everything else replays the reference's sequential fp32 accumulation.

E1 + E2 + E3 is twice the signed area: one edge function at the opposite vertex, which can lie far outside the
clipped window the per-edge bound covers.  A triangle whose window passes that bound but whose sum is 2^24 or
more would recover a wrong E1 (the float sum rounds), and with it a wrong barycentric bA in the Gouraud / flat
light sum.  Part B renders exactly such triangles; the other parts push every coordinate of every primitive kind
to the ends of the float range (1e9, 1e30, +-FLT_MAX, +-inf, NaN), where the clip collapses the bbox to the frame.

Every GPU check compares colour and depth bit for bit with the oracle, the SetPixels counter and, with ids on,
the id planes.  The stages run as in test_gpu_launch_shapes.py: the default one-kernel stage, the two-kernel
stage and the single kernel for all-opaque passes, and passes that blend (the general kernel in every mode).
"""
import functools
import os
import re

import numpy as np
import pytest

from dtrenderer_b200 import api, scenes
from test_gpu_launch_shapes import CSRC, _check_frames, _oracle_frame, _renderer, _source_constant

F32 = np.float32
FLT_MAX = float(np.finfo(F32).max)
SUB_W, SUB_H = _source_constant("SUB_W"), _source_constant("SUB_H")
ANCHOR = F32(0.33)                        # DEFAULT_TRIANGLE_TRANSFORM and the mesh's triangle transform
# raster paths: (translucent content?, opaque-stage setting, what last_pass_stage() must report)
PATHS = {"blend": (True, api.OPAQUE_ONE_KERNEL, api.OPAQUE_SINGLE_KERNEL),
         "single": (False, api.OPAQUE_SINGLE_KERNEL, api.OPAQUE_SINGLE_KERNEL),
         "one_kernel": (False, api.OPAQUE_ONE_KERNEL, api.OPAQUE_ONE_KERNEL),
         "two_kernels": (False, api.OPAQUE_TWO_KERNELS, api.OPAQUE_TWO_KERNELS)}


def _edge_limits():
    """The two 2^24 thresholds of setup_kernel's exactness rule: the per-edge bound and |E1 + E2 + E3|."""
    with open(os.path.join(CSRC, "dtr_kernels.cu")) as fh:
        src = fh.read()
    bound = re.search(r"\(bound\s*<\s*([0-9.]+)\)", src)
    total = re.search(r"abs\(eSum\)\s*<\s*([0-9]+)", src)
    assert bound and total, "the exactness rule of setup_kernel was not found"
    return float(bound.group(1)), int(total.group(1))


BOUND_LIMIT, SUM_LIMIT = _edge_limits()


# ---- A. the setup classification, restated -----------------------------------------------------------
def _rmin(a, b):
    return np.where(a < b, a, b)          # DQN_MIN: the comparison direction decides NaN and -0


def _rmax(a, b):
    return np.where(a < b, b, a)


def _edge(ax, ay, bx, by, cx, cy):
    return ((bx - ax) * (cy - ay)) - ((by - ay) * (cx - ax))


def setup_model(p, w, h, anchor=ANCHOR):
    """float32 model of setup_kernel for triangles p (n, 9) under an unrotated, unscaled transform (xAxis (1, 0),
    yAxis (-0, 1)) with the given anchor: winding swap, anchor round trip, bbox clip and truncation, e0 / dx / dy
    at the bbox origin, the per-edge bound, the -0 rule and the sum rule.  Clipped bboxes must lie in the int
    range (the test scenes keep them there)."""
    p = np.asarray(p, F32).reshape(-1, 3, 3)
    x, y, z = [p[:, :, i].copy() for i in range(3)]
    one, zero, nzero, a = F32(1), F32(0), F32(-0.0), F32(anchor)
    with np.errstate(all="ignore"):
        area2 = (((x[:, 1] - x[:, 0]) * (y[:, 1] + y[:, 0])) + ((x[:, 2] - x[:, 1]) * (y[:, 2] + y[:, 1]))) + \
            ((x[:, 0] - x[:, 2]) * (y[:, 0] + y[:, 2]))
        sw = area2 > 0
        for v in (x, y, z):
            v[sw, 1], v[sw, 2] = v[sw, 2].copy(), v[sw, 1].copy()
        ox = (x[:, 0] + ((x[:, 1] - x[:, 0]) * a)) + ((x[:, 2] - x[:, 0]) * a)
        oy = (y[:, 0] + ((y[:, 1] - y[:, 0]) * a)) + ((y[:, 2] - y[:, 0]) * a)
        qx, qy = x - ox[:, None], y - oy[:, None]
        x = (ox[:, None] + (one * qx)) + (nzero * qy)
        y = (oy[:, None] + (zero * qx)) + (one * qy)
        bminx, bmaxx = _rmin(_rmin(x[:, 0], x[:, 1]), x[:, 2]), _rmax(_rmax(x[:, 0], x[:, 1]), x[:, 2])
        bminy, bmaxy = _rmin(_rmin(y[:, 0], y[:, 1]), y[:, 2]), _rmax(_rmax(y[:, 0], y[:, 1]), y[:, 2])
        bmaxx, bmaxy = _rmin(bmaxx, F32(w - 1)), _rmin(bmaxy, F32(h - 1))
        bminx, bminy = _rmax(zero, bminx), _rmax(zero, bminy)
        clip = np.stack([bminx, bminy, bmaxx, bmaxy], 1)
        assert (np.abs(clip) < 2.0 ** 31).all(), "clipped bbox outside the int range"
        minx, miny, maxx, maxy = [np.trunc(v).astype(np.int64) for v in (bminx, bminy, bmaxx, bmaxy)]
        sx, sy = minx.astype(F32), miny.astype(F32)
        e0 = np.stack([_edge(x[:, 1], y[:, 1], x[:, 2], y[:, 2], sx, sy), _edge(x[:, 2], y[:, 2], x[:, 0], y[:, 0], sx, sy),
                       _edge(x[:, 0], y[:, 0], x[:, 1], y[:, 1], sx, sy)], 1)
        dx = np.stack([y[:, 1] - y[:, 2], y[:, 2] - y[:, 0], y[:, 0] - y[:, 1]], 1)
        dy = np.stack([x[:, 2] - x[:, 1], x[:, 0] - x[:, 2], x[:, 1] - x[:, 0]], 1)
        area = (e0[:, 0] + e0[:, 1]) + e0[:, 2]
        small = ((x == np.trunc(x)) & (np.abs(x) < 2.0 ** 24) & (y == np.trunc(y)) & (np.abs(y) < 2.0 ** 24)).all(1)
        wd, hd = (maxx - minx + SUB_W).astype(np.float64), (maxy - miny + SUB_H).astype(np.float64)
        bound = np.abs(e0.astype(np.float64)) + wd[:, None] * np.abs(dx.astype(np.float64)) + hd[:, None] * np.abs(dy.astype(np.float64))
        negzero = (e0.view(np.uint32) == 0x80000000).any(1)
        exact_old = small & (bound < BOUND_LIMIT).all(1) & ~negzero
        esum = np.where(exact_old, np.nan_to_num(e0.astype(np.float64)).astype(np.int64).sum(1), 0)
        exact = exact_old & (np.abs(esum) < SUM_LIMIT)
    return dict(x=x, y=y, z=z, minx=minx, miny=miny, maxx=maxx, maxy=maxy, e0=e0, dx=dx, dy=dy, area=area,
                inv=one / area, skip=(area == 0) | (maxx <= minx) | (maxy <= miny), bound=bound.max(1),
                negzero=negzero, exact_old=exact_old, esum=esum, exact=exact)


def _one(s, i):
    return {k: v[i] for k, v in s.items()}


def sequential_edges(t):
    """The oracle's edge values over the window of one modelled triangle: rows accumulate dy from e0 and every
    row accumulates dx, in fp32, in the reference's order.  (ny, nx, 3)."""
    nx, ny = int(t["maxx"] - t["minx"]), int(t["maxy"] - t["miny"])
    out = np.empty((ny, nx, 3), F32)
    for k in range(3):
        rows = np.add.accumulate(np.r_[t["e0"][k], np.full(ny - 1, t["dy"][k], F32)].astype(F32))
        m = np.empty((ny, nx), F32)
        m[:, 0], m[:, 1:] = rows, t["dx"][k]
        out[:, :, k] = np.add.accumulate(m, axis=1)
    return out


def direct_edges(t):
    """Exact integer edge values over the window (what the int32 path of an exact triangle evaluates)."""
    nx, ny = int(t["maxx"] - t["minx"]), int(t["maxy"] - t["miny"])
    X, Y = np.meshgrid(np.arange(nx), np.arange(ny))
    return np.stack([int(t["e0"][k]) + X * int(t["dx"][k]) + Y * int(t["dy"][k]) for k in range(3)], 2)


def recovered_e1(t, e2, e3):
    """E1 as the queued fragments of the general kernel recover it: (float(E1 + E2 + E3) - E2) - E3."""
    return (F32(int(t["esum"])) - e2) - e3


def _fragment_z(t, e, zs):
    z1, z2, z3 = [F32(v) for v in zs]
    with np.errstate(all="ignore"):
        return (z1 + (e[..., 1] * t["inv"]) * (z2 - z1)) + (e[..., 2] * t["inv"]) * (z3 - z1)


# ---- triangles built for each class ------------------------------------------------------------------
def _search_bound(target, w, h, want_exact):
    """An integer-vertex triangle whose largest per-edge bound is exactly `target` = a * b: a horizontal edge of
    length b at y0 = -(a - hd) above the frame (its bound is b * (|y0| + hd), hd = h - 1 + SUB_H), the apex just
    below the frame, so that the clipped window is the whole frame and twice the area stays below 2^24."""
    a, b = (4095, 4097) if want_exact else (4096, 4096)
    assert a * b == target
    hd = h - 1 + SUB_H
    y0 = -(a - hd)
    for dx in range(0, 400, 7):
        x0 = w // 2 - b // 2 - dx
        p = np.array([x0, y0, 1.0, x0 + b, y0, 5.0, w // 2 + dx // 3, h + 2, 30.0], F32)
        t = _one(setup_model(p, w, h), 0)
        if t["bound"] == target and t["exact"] == want_exact and not t["skip"] and (t["x"] == np.trunc(t["x"])).all():
            return p
    raise AssertionError(f"no triangle with bound {target}")


def _search_rounding(w, h, seed):
    """An integer-vertex sliver through the frame, its long edge 2^24 / (w + h) to 2^25 / (w + h) px long and its
    apex a few px off that edge: the largest bound lies in [2^24, 2^25) while |E1 + E2 + E3| stays below 2^24, so
    only the per-edge bound makes it inexact.  Its sequential accumulation rounds on the pixels of the window
    far from the long edge and carries the error into covered pixels: the depth of at least one covered pixel
    differs from what a direct evaluation gives."""
    rng = np.random.default_rng(seed)
    for _ in range(50):
        n = 4096
        length = rng.uniform(2.0 ** 24 / (w + h), 2.0 ** 25 / (w + h), n)
        ang = rng.uniform(0, np.pi, n)
        cx, cy = rng.uniform(0, w, n), rng.uniform(0, h, n)
        half = np.stack([length / 2 * np.cos(ang), length / 2 * np.sin(ang)], 1)
        p = np.zeros((n, 9), F32)
        p[:, 0:2] = (np.stack([cx, cy], 1) - half).round()
        p[:, 3:5] = (np.stack([cx, cy], 1) + half).round()
        p[:, 6:8] = np.stack([cx, cy], 1).round() + rng.integers(-60, 61, (n, 2))
        p[:, 2::3] = rng.uniform(-200, 200, (n, 3))
        s = setup_model(p, w, h)
        total = np.abs(np.nan_to_num(s["e0"].astype(np.float64)).sum(1))
        ints = ((s["x"] == np.trunc(s["x"])) & (s["y"] == np.trunc(s["y"]))).all(1)
        ok = ~s["skip"] & (s["bound"] >= BOUND_LIMIT) & (s["bound"] < 2 * BOUND_LIMIT) & ~s["negzero"] & (total < SUM_LIMIT) & ints
        for i in np.flatnonzero(ok):
            t = _one(s, i)
            es, ed = sequential_edges(t), direct_edges(t).astype(F32)
            cov = (es >= 0).all(2)
            if cov.sum() > 20 and ((_fragment_z(t, es, t["z"]) != _fragment_z(t, ed, t["z"])) & cov).any():
                return p[i]
    raise AssertionError("no rounding triangle found")


def _search_negzero(w, h, seed):
    """A triangle with vertex p1 on the frame's corner pixel (0, 0), p2 left of the frame and below it, p3 right of
    it and above the frame, and vertex depths of -0, -1 and 1: e0 of edge p1 -> p2 is (p2x - 0) * (+0) - (p2y - 0)
    * (+0) = -0, the corner pixel is covered, and its depth is -0 from the sequential accumulation but +0 from an
    int32 evaluation (only the sign of the zero depth differs)."""
    rng = np.random.default_rng(seed)
    for _ in range(20000):
        p = np.array([0, 0, -0.0, -rng.integers(1, 40), rng.integers(1, 40), -1.0,
                      rng.integers(1, 60), -rng.integers(1, 60), -0.0], F32)
        p[[2, 5, 8]] = rng.choice(np.array([-0.0, -0.0, -1.0, 1.0], F32), 3)
        if rng.random() < 0.5:
            p[3:6], p[6:9] = p[6:9].copy(), p[3:6].copy()
        t = _one(setup_model(p, w, h), 0)
        if t["skip"] or not t["negzero"]:
            continue
        es = sequential_edges(t)
        ed = direct_edges(t).astype(F32)
        cov = (es >= 0).all(2)
        zq, zd = _fragment_z(t, es, t["z"]), _fragment_z(t, ed, t["z"])
        if (cov & (zq.view(np.uint32) != zd.view(np.uint32))).any() and (zq[cov] == 0).any():
            return p
    raise AssertionError("no -0 triangle found")


@functools.lru_cache(maxsize=None)
def bound_triangles(w, h):
    """{name: p}: the constructions of part C, each checked against its class by test_constructed_classes."""
    return {"bound_2^24-1": _search_bound(BOUND_LIMIT - 1, w, h, True),
            "bound_2^24": _search_bound(BOUND_LIMIT, w, h, False),
            "rounds": _search_rounding(w, h, 3),
            "negzero": _search_negzero(w, h, 4)}


# mesh vertices land on chosen pixels: with pos 0, rotation 0, anchor 0, scale 1 a model vertex (x, y, 0, 1)
# projects to ((W/4) x + W/2, (H/4) y + H/2) exactly in power-of-two frames, and the snap (int)(v + 0.5)
# truncates toward zero: a pixel P < 0 comes from P - 1.
MESH_TRANSFORM = scenes.transform7(0.0, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))
MESH_SIZES = (64, 128, 256)


def mesh_model_coords(pix, w, h):
    pix = np.asarray(pix, np.float64).reshape(-1, 2)
    pre = np.where(pix < 0, pix - 1, pix)
    return ((pre - [w / 2, h / 2]) / [w / 4, h / 4]).astype(F32)


def one_face_mesh(pix, w, h, normals, uv):
    v = mesh_model_coords(pix, w, h)
    vert = np.concatenate([v, np.zeros((3, 1), F32), np.ones((3, 1), F32)], 1)
    texuv = np.concatenate([np.asarray(uv, F32).reshape(3, 2), np.zeros((3, 1), F32)], 1)
    return {"vertexes": vert, "texUV": texuv, "normals": np.asarray(normals, F32).reshape(3, 3),
            "faces": np.array([[0, 1, 2, 0, 1, 2, 0, 1, 2]], np.int32)}


@functools.lru_cache(maxsize=None)
def huge_exact_triangles(size, count=2, seed=0):
    """Snapped screen triangles around a size x size frame that the parent rule called exact while
    |E1 + E2 + E3| >= 2^24, that cover pixels of the frame and whose recovered E1 is wrong on covered pixels."""
    rng = np.random.default_rng([size, seed])
    found = []
    while len(found) < count:
        p = np.zeros((4096, 9), F32)
        p[:, [0, 1, 3, 4, 6, 7]] = rng.integers(-4500, 4500 + size, (4096, 6))
        s = setup_model(p, size, size)
        for i in np.flatnonzero(s["exact_old"] & ~s["exact"] & ~s["skip"]):
            t = _one(s, i)
            e = direct_edges(t)
            cov = (e >= 0).all(2)
            if cov.sum() < size * size // 4:
                continue
            e1 = recovered_e1(t, e[..., 1].astype(F32), e[..., 2].astype(F32))
            if (cov & (e1 != e[..., 0].astype(F32))).sum() > cov.sum() // 8:
                found.append(p[i])
                break
    return np.array(found)


# ---- CPU tests ----------------------------------------------------------------------------------------
def test_limits_read_from_the_sources():
    assert (SUB_W, SUB_H) == (8, 4)
    assert BOUND_LIMIT == 2.0 ** 24 and SUM_LIMIT == 2 ** 24


@pytest.mark.parametrize("w,h", [(64, 64), (257, 131)])
def test_constructed_classes(w, h):
    """Each construction lands in the class it was built for, by the model of setup_kernel."""
    tris = bound_triangles(w, h)
    s = setup_model(np.array(list(tris.values())), w, h)
    c = {k: _one(s, i) for i, k in enumerate(tris)}
    assert c["bound_2^24-1"]["bound"] == BOUND_LIMIT - 1 and c["bound_2^24-1"]["exact"]
    assert c["bound_2^24"]["bound"] == BOUND_LIMIT and not c["bound_2^24"]["exact"] and not c["bound_2^24"]["negzero"]
    assert BOUND_LIMIT <= c["rounds"]["bound"] < 2 * BOUND_LIMIT and not c["rounds"]["exact"]
    assert abs(float(np.sum(c["rounds"]["e0"].astype(np.float64)))) < SUM_LIMIT   # the per-edge bound alone decides
    assert c["negzero"]["negzero"] and not c["negzero"]["exact"]
    # without the -0 rule it would be exact
    t = c["negzero"]
    assert t["bound"] < BOUND_LIMIT and abs(int(np.nansum(t["e0"]))) < SUM_LIMIT


@pytest.mark.parametrize("size", MESH_SIZES)
def test_huge_triangles_are_exact_by_the_old_rule_only(size):
    """The part B triangles: every per-edge bound below 2^24 and no -0, but |E1 + E2 + E3| >= 2^24: inexact."""
    s = setup_model(huge_exact_triangles(size), size, size)
    assert s["exact_old"].all() and not s["exact"].any()
    assert (np.abs(s["esum"]) >= SUM_LIMIT).all() and (s["bound"] < BOUND_LIMIT).all()
    # and an ordinary exact triangle stays exact
    t = setup_model(np.array([3, 4, 0, 40, 9, 0, 12, 50, 0], F32), size, size)
    assert t["exact"].all() and t["exact_old"].all()


@pytest.mark.parametrize("size", MESH_SIZES)
def test_mesh_vertices_land_on_chosen_pixels(built, size):
    """A one-face mesh placed with mesh_model_coords covers, in the oracle, exactly the pixels of the 2D triangle
    at the chosen pixels (vertices left of and above the frame included)."""
    from oracle import dtro
    rng = np.random.default_rng(size)
    for _ in range(6):
        pix = rng.integers(-size // 2, size + size // 2, (3, 2))
        m = one_face_mesh(pix, size, size, np.tile([0, 0, 1], 3), np.zeros(6))
        a, b = dtro.Oracle(size, size), dtro.Oracle(size, size)
        a.mesh(m, scenes.WHITE_TEXTURE, scenes.SHADE_FULLBRIGHT, (0, 0, 1), (1, 1, 1, 1), (0, 0, 0), MESH_TRANSFORM)
        p = np.concatenate([pix, np.zeros((3, 1))], 1).astype(F32).reshape(9)
        b.triangle(p, (1, 1, 1, 1), scenes.DEFAULT_TRIANGLE_TRANSFORM)
        assert a.counters()[0] == b.counters()[0]
        assert np.array_equal(a.color(), b.color()), pix


# ---- B. E1 of huge exact triangles in lit meshes ------------------------------------------------------
LIGHT_VECTOR = (0.3, -0.4, 1.0)
MESH_KINDS = ((scenes.SHADE_FLAT, False), (scenes.SHADE_FLAT, True), (scenes.SHADE_GOURAUD, False), (scenes.SHADE_GOURAUD, True))
MESH_TEX = scenes.random_texture(13, 11, 31, opaque=True)
FRAMES_PER_KIND = 2                       # light colours per (mesh kind, triangle) and batch
# light colours tried per (mesh kind, triangle).  Gouraud triangles always find FRAMES_PER_KIND sensitive ones;
# in flat mode the three light products are equal and a wrong E1 rarely moves a byte, so fewer are tried there
CANDIDATES = {scenes.SHADE_GOURAUD: 2000, scenes.SHADE_FLAT: 400}
INV_255 = F32(1) / F32(255)


def _norm(v):
    v = np.asarray(v, F32)
    inv = F32(1) / np.sqrt(((v[..., 0] * v[..., 0]) + (v[..., 1] * v[..., 1])) + (v[..., 2] * v[..., 2]))
    return v * inv[..., None]


def _dot(a, b):
    r = np.zeros(np.broadcast(a[..., 0], b[..., 0]).shape, F32)
    for i in range(3):
        r = r + (a[..., i] * b[..., i])
    return r


def _mesh_inputs(size, k):
    """Mesh pixels, normals and uv of huge triangle k of a size x size frame."""
    p = huge_exact_triangles(size)[k].reshape(3, 3)
    rng = np.random.default_rng([size, k, 5])
    normals = np.c_[rng.uniform(-0.6, 0.6, (3, 2)), rng.uniform(0.5, 1.0, 3)].astype(F32)
    uv = rng.uniform(0, 0.999, 6).astype(F32)
    return p[:, :2].astype(np.int64), normals, uv


def shade_bytes(t, e1, e2, e3, mode, normals, uv, tex, colours, dst):
    """Output words of queued fragments (colour model of SlowTriangle's inner loop) for light colours (m, 4):
    (m, npix) uint32.  dst: the destination word under each pixel."""
    cols = np.asarray(colours, F32)
    L = _norm(np.asarray(LIGHT_VECTOR, F32))
    if mode == scenes.SHADE_FLAT:
        pts = np.stack([t["x"], t["y"], t["z"]], 1)
        a, b = pts[1] - pts[0], pts[2] - pts[0]
        n = np.array([(a[1] * b[2]) - (a[2] * b[1]), (a[2] * b[0]) - (a[0] * b[2]), (a[0] * b[1]) - (a[1] * b[0])], F32)
        n = _norm(n)
        inten = _dot(n, L)
        inten = inten if F32(0) < inten else F32(0)
        cols = cols.copy()
        cols[:, :3] = cols[:, :3] * inten
        m = np.ones(3, F32)
    else:
        I = _dot(_norm(normals), L)
        m = np.where(F32(0) < I, I, F32(0)).astype(F32)
    c = (cols[:, :3] * cols[:, :3]) * cols[:, 3:4]                          # (m, 3) premultiplied linear
    light = c[:, None, :] * m[None, :, None]                               # (m, vertex, channel)
    inv = t["inv"]
    bA, bB, bC = e1 * inv, e2 * inv, e3 * inv
    f = np.empty((len(cols), 3, len(e1)), F32)
    for ch in range(3):
        l = ((light[:, 0, ch, None] * bA) + (light[:, 1, ch, None] * bB)) + (light[:, 2, ch, None] * bC)
        f[:, ch] = c[:, ch, None] * l
    fa = np.broadcast_to(cols[:, 3:4], (len(cols), len(e1))).astype(F32)
    if tex is not None:
        u1, v1, u2, v2, u3, v3 = [F32(v) for v in uv]
        u = (u1 + ((u2 - u1) * bB)) + ((u3 - u1) * bC)
        v = (v1 + ((v2 - v1) * bB)) + ((v3 - v1) * bC)
        th, tw = tex.shape[:2]
        tx = np.trunc(np.clip(u, 0, 1) * F32(tw)).astype(np.int64)
        ty = np.trunc(np.clip(v, 0, 1) * F32(th)).astype(np.int64)
        texel = tex.reshape(-1, 4)[ty * tw + tx].astype(np.uint32)
        for ch, byte in ((0, 0), (1, 1), (2, 2)):
            tc = texel[:, byte].astype(F32) * INV_255
            f[:, ch] = f[:, ch] * (tc * tc)
        fa = fa * (texel[:, 3].astype(F32) * INV_255)
    inv_a = F32(1) - fa
    out = np.zeros((len(cols), len(e1)), np.uint32)
    for ch, shift in ((0, 16), (1, 8), (2, 0)):
        dl = ((dst >> shift) & 0xFF).astype(F32) * F32(1) / F32(255)
        d = f[:, ch] + (inv_a * (dl * dl))
        with np.errstate(invalid="ignore"):
            d = np.where(d == 0, F32(0), np.sqrt(d)) * F32(255)
        d = np.where(d > 255, F32(255), d)
        out |= d.astype(np.uint32) << shift
    return out


CLEAR_RGB = (0.25, 0.5, 0.75)


def _clear_word():
    r, g, b = [int(F32(c) * F32(255)) for c in CLEAR_RGB]
    return (r << 16) | (g << 8) | b


@functools.lru_cache(maxsize=None)
def sensitive_colours(size, k, mode, textured, translucent):
    """Light colours for which the recovery of E1 as (sum - E2) - E3 changes at least one output byte of huge
    triangle k, by the model: the colours of part B's frames."""
    pix, normals, uv = _mesh_inputs(size, k)
    p = np.concatenate([pix, np.zeros((3, 1))], 1).astype(F32)
    t = _one(setup_model(p.reshape(1, 9), size, size), 0)
    # the mesh's projected depth is the same at every vertex; only x, y matter to the flat normal's direction
    t["z"] = np.zeros(3, F32)
    e = direct_edges(t)
    cov = (e >= 0).all(2)
    e1, e2, e3 = [e[..., i][cov].astype(F32) for i in range(3)]
    bad = recovered_e1(t, e2, e3) != e1
    e1, e2, e3, r1 = e1[bad], e2[bad], e3[bad], recovered_e1(t, e2[bad], e3[bad])
    dst = np.full(len(e1), _clear_word(), np.uint32)
    rng = np.random.default_rng([size, k, mode, textured, translucent])
    keep, rest = [], []
    for start in range(0, CANDIDATES[mode], 200):
        cols = rng.uniform(0.05, 1.0, (200, 4)).astype(F32)
        cols[:, 3] = rng.uniform(0.3, 0.95, 200) if translucent else 1.0
        tex = MESH_TEX if textured else None
        good = shade_bytes(t, e1, e2, e3, mode, normals, uv, tex, cols, dst)
        wrong = shade_bytes(t, r1, e2, e3, mode, normals, uv, tex, cols, dst)
        hit = (good != wrong).any(1)
        keep += [tuple(float(v) for v in c) for c in cols[hit]]
        rest += [tuple(float(v) for v in c) for c in cols[~hit][:FRAMES_PER_KIND]]
        if len(keep) >= FRAMES_PER_KIND:
            break
    keep = keep[:FRAMES_PER_KIND]
    return tuple(keep), tuple(rest[:FRAMES_PER_KIND - len(keep)])


def _mesh_op(size, k, mode, textured, colour):
    pix, normals, uv = _mesh_inputs(size, k)
    return ("mesh", dict(mesh=one_face_mesh(pix, size, size, normals, uv), tex=MESH_TEX if textured else scenes.WHITE_TEXTURE,
                         light_mode=mode, light_vector=LIGHT_VECTOR, light_color=colour, pos=(0, 0, 0), transform=MESH_TRANSFORM))


@functools.lru_cache(maxsize=None)
def mesh_frames(size, translucent):
    """One frame per (triangle, mesh kind, sensitive light colour): a clear and the one-face mesh."""
    frames = []
    for k in range(len(huge_exact_triangles(size))):
        for mode, textured in MESH_KINDS:
            cols = sum(sensitive_colours(size, k, mode, textured, translucent), ())
            for c in cols:
                ops = [("clear", dict(rgb=CLEAR_RGB)), _mesh_op(size, k, mode, textured, c)]
                frames.append((ops, _oracle_frame(size, size, ops)))
    return frames


@pytest.mark.parametrize("translucent", [False, True], ids=["opaque", "translucent"])
@pytest.mark.parametrize("size", MESH_SIZES)
def test_shading_model_matches_the_oracle(built, size, translucent):
    """The colour model that picks part B's light colours reproduces the oracle's bytes with the true E1, and
    enough sensitive colours exist for every mesh kind: part B cannot lose its sensitivity unnoticed."""
    n_tris = len(huge_exact_triangles(size))
    frames = mesh_frames(size, translucent)
    assert len(frames) == n_tris * len(MESH_KINDS) * FRAMES_PER_KIND
    f = 0
    for k in range(n_tris):
        pix, normals, uv = _mesh_inputs(size, k)
        p = np.concatenate([pix, np.zeros((3, 1))], 1).astype(F32)
        t = _one(setup_model(p.reshape(1, 9), size, size), 0)
        t["z"] = np.zeros(3, F32)
        e = direct_edges(t)
        cov = (e >= 0).all(2)
        ys, xs = np.nonzero(cov)
        e1, e2, e3 = [e[..., i][cov].astype(F32) for i in range(3)]
        for mode, textured in MESH_KINDS:
            sensitive, other = sensitive_colours(size, k, mode, textured, translucent)
            if mode == scenes.SHADE_GOURAUD:
                assert len(sensitive) >= 1, (size, k, textured, translucent)
            for c in sensitive + other:
                col = frames[f][1][0]
                want = col[ys + int(t["miny"]), xs + int(t["minx"])]
                dst = np.full(len(e1), _clear_word(), np.uint32)
                got = shade_bytes(t, e1, e2, e3, mode, normals, uv, MESH_TEX if textured else None, np.array([c], F32), dst)[0]
                assert np.array_equal(got, want), (size, k, mode, textured, c, (got != want).sum())
                wrong = shade_bytes(t, recovered_e1(t, e2, e3), e2, e3, mode, normals, uv, MESH_TEX if textured else None,
                                    np.array([c], F32), dst)[0]
                assert (wrong != want).any() == (c in sensitive)
                f += 1


@pytest.mark.gpu
@pytest.mark.parametrize("ids", [False, True], ids=["ids_off", "ids_on"])
@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("size", MESH_SIZES)
def test_huge_exact_mesh_triangles(built, size, path, ids):
    """Lit one-face meshes (flat and Gouraud, untextured and textured) whose triangle covers the frame from
    thousands of pixels out, with |E1 + E2 + E3| >= 2^24, one light colour per frame of a batch: each colour was
    picked because a wrong E1 changes at least one byte of its frame."""
    translucent, stage, want_stage = PATHS[path]
    frames = mesh_frames(size, translucent)
    r = _renderer(size, size, len(frames), ids, stage)
    for f, (ops, _) in enumerate(frames):
        r.begin_frame(f)
        scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == want_stage
    _check_frames(r, [ref for _, ref in frames], ids)
    r.close()


# ---- C. the bound at its edge -------------------------------------------------------------------------
BOUND_SIZES = ((64, 64), (257, 131))
TEX_OPAQUE = scenes.random_texture(9, 7, 41, opaque=True)
TEX_TRANSLUCENT = scenes.random_texture(10, 6, 42, opaque=False)


def _padded(tex):
    """The texture as a view of a larger array: the oracle's read at v = 1 (row h) and at u = 1 in the last row
    meets what the device's spare texels hold, opaque white after an opaque texture and zeros after any other."""
    h, w = tex.shape[:2]
    buf = np.full((h + 2, w, 4), 255 if (tex[..., 3] == 255).all() else 0, np.uint8)
    buf[:h] = tex
    return buf[:h]


PAD_OPAQUE, PAD_TRANSLUCENT = _padded(TEX_OPAQUE), _padded(TEX_TRANSLUCENT)


@functools.lru_cache(maxsize=None)
def bound_frames(size, translucent):
    """One frame per construction and texture kind (none / textured): a clear, then the triangle."""
    w, h = size
    rng = np.random.default_rng([w, h, translucent])
    frames = []
    for name, p in bound_triangles(w, h).items():
        for textured in (False, True):
            a = F32(0.6) if translucent else F32(1)
            col = (*rng.uniform(0.2, 1.0, 3).tolist(), float(a))
            if textured:
                op = ("textured_triangle", dict(p=p, uv=rng.uniform(-0.2, 1.2, 6).astype(F32), tex=PAD_TRANSLUCENT if translucent else PAD_OPAQUE,
                                                color=col, transform=scenes.DEFAULT_TRIANGLE_TRANSFORM))
            else:
                op = ("triangle", dict(p=p, color=col, transform=scenes.DEFAULT_TRIANGLE_TRANSFORM))
            ops = [("clear", dict(rgb=tuple(rng.random(3).tolist()))), op]
            frames.append((ops, _oracle_frame(w, h, ops)))
    return frames


@pytest.mark.gpu
@pytest.mark.parametrize("ids", [False, True], ids=["ids_off", "ids_on"])
@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("size", BOUND_SIZES, ids=[f"{w}x{h}" for w, h in BOUND_SIZES])
def test_bound_at_its_edge(built, size, path, ids):
    """Integer triangles whose largest per-edge bound is 2^24 - 1 (exact) and 2^24 (inexact), one past 2^24
    whose sequential accumulation rounds on covered pixels, and one with an e0 of -0 and vertex depths of -0
    (the covered corner pixel's depth is -0, an int32 evaluation would give +0)."""
    w, h = size
    translucent, stage, want_stage = PATHS[path]
    frames = bound_frames(size, translucent)
    r = _renderer(w, h, len(frames), ids, stage)
    for f, (ops, _) in enumerate(frames):
        r.begin_frame(f)
        scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == want_stage
    _check_frames(r, [ref for _, ref in frames], ids)
    r.close()


# ---- D. far coordinates ----------------------------------------------------------------------------------
FAR_SIZES = ((64, 64), (257, 131), (1920, 1080))
FAR = [2.0 ** 12, 2.0 ** 24 - 1, 2.0 ** 24, 2.0 ** 24 + 1, 2.0 ** 25, 1e9, 1e30, FLT_MAX, np.inf]
FAR_TRANSFORMS = (scenes.DEFAULT_TRIANGLE_TRANSFORM, scenes.transform7(0.7, (0.33, 0.33, 0.33), (1.0, 1.0, 1.0)),
                  scenes.transform7(0.0, (0.33, 0.33, 0.33), (-1.0, 1.0, 1.0)), scenes.transform7(2.5, (-3.0, 4.0, 0.0), (1.3, -0.7, 1.0)),
                  scenes.transform7(0.0, (0.33, 0.33, 0.33), (1.0, -1.0, 1.0)))


def _clipped_min_in_range(p, transform, w, h):
    """The oracle truncates the clipped bbox with a C cast, which x86 and the device only agree on inside the int
    range: a triangle whose clipped minimum lies beyond 2^31 (every vertex far right or below) is left out."""
    x = setup_model_transformed(p, transform)
    bmin = [_rmax(F32(0), _rmin(_rmin(v[0], v[1]), v[2])) for v in x]
    return all(float(b) < 2.0 ** 31 for b in bmin)


def setup_model_transformed(p, transform):
    """Screen x and y of a 2D triangle after the winding swap and the transform (the oracle's order)."""
    p = np.asarray(p, F32).reshape(3, 3)
    x, y = p[:, 0].copy(), p[:, 1].copy()
    with np.errstate(all="ignore"):
        area2 = (((x[1] - x[0]) * (y[1] + y[0])) + ((x[2] - x[1]) * (y[2] + y[1]))) + ((x[0] - x[2]) * (y[0] + y[2]))
        if area2 > 0:
            x[[1, 2]], y[[1, 2]] = x[[2, 1]], y[[2, 1]]
        rot, ax, ay, _, sx, sy, _ = [F32(v) for v in transform]
        c, s = F32(np.cos(np.float32(rot))), F32(np.sin(np.float32(rot)))
        xa, ya = (c * sx, s * sx), (-s * sy, c * sy)
        ox = (x[0] + ((x[1] - x[0]) * ax)) + ((x[2] - x[0]) * ax)
        oy = (y[0] + ((y[1] - y[0]) * ay)) + ((y[2] - y[0]) * ay)
        qx, qy = x - ox, y - oy
        return (ox + (xa[0] * qx)) + (ya[0] * qy), (oy + (xa[1] * qx)) + (ya[1] * qy)


def _far_triangles(w, h, rng):
    """2D triangles with vertices at FAR (both signs, integer and not) and NaN: slivers clipped along each frame
    edge, triangles covering the whole frame, and non-finite ones."""
    tris = []
    cx, cy = w / 2, h / 2
    for v in FAR:
        frac = 0.0 if v >= 2.0 ** 23 else 0.37
        big = v + frac
        # slivers along the four edges (one vertex inside, two far out along the edge)
        tris += [(1.5 + frac, 2.0, -big, 0.0, big, 3.0), (w - 3.0, 1.0 + frac, w - 1.0, -big, w + 2.0, big),
                 (-big, h - 2.0, big, h - 1.0 + frac, cx, h - 4.0), (0.0, -big, 3.0 + frac, big, 1.0, cy)]
        # covering the frame
        tris += [(-big, -big, big, -big, cx, big), (cx + frac, -big, big, big, -big, big)]
    # NaN and +-inf: the clip collapses the bbox to the frame
    nan, inf = np.nan, np.inf
    tris += [(nan, 1.0, 20.0, 5.0, 3.0, 30.0), (1.0, nan, 20.0, 5.0, 3.0, 30.0), (nan, nan, nan, nan, nan, nan),
             (-inf, -inf, inf, -inf, cx, inf), (inf, 2.0, -inf, 9.0, 3.0, 40.0), (-FLT_MAX, -FLT_MAX, FLT_MAX, 0.0, 0.0, FLT_MAX),
             (2.0, 3.0, 2.0 ** 24 + 1, 5.0, 7.0, 2.0 ** 24 + 3)]
    out = []
    for t in tris:
        z = rng.uniform(-50, 50, 3)
        out.append(np.array([t[0], t[1], z[0], t[2], t[3], z[1], t[4], t[5], z[2]], F32))
    return out


@functools.lru_cache(maxsize=None)
def far_frames(size, translucent):
    """Frames of far triangles, plain and textured (uv in [-2, 3]: the clamp, the u = 1 column and the v = 1
    padding row), under every transform of FAR_TRANSFORMS."""
    w, h = size
    rng = np.random.default_rng([w, h, translucent, 9])
    tris = _far_triangles(w, h, rng)
    frames = []
    for ti, tr in enumerate(FAR_TRANSFORMS):
        ops = [("clear", dict(rgb=tuple(rng.random(3).tolist())))]
        n = 0
        for i, p in enumerate(tris):
            if not _clipped_min_in_range(p, tr, w, h):
                continue
            a = float(rng.choice([0.5, 1.0])) if translucent else 1.0
            col = (*rng.uniform(0.1, 1.0, 3).tolist(), a)
            if (i + ti) % 3 == 0:
                uv = rng.choice(np.array([-2.0, -0.5, 0.0, 0.3, 0.999, 1.0, 1.7, 3.0], F32), 6)
                ops.append(("textured_triangle", dict(p=p, uv=uv, tex=PAD_TRANSLUCENT if translucent else PAD_OPAQUE, color=col, transform=tr)))
            else:
                ops.append(("triangle", dict(p=p, color=col, transform=tr)))
            n += 1
        assert n > len(tris) // 2
        frames.append((ops, _oracle_frame(w, h, ops)))
    return frames


@pytest.mark.gpu
@pytest.mark.parametrize("ids", [False, True], ids=["ids_off", "ids_on"])
@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("size", FAR_SIZES, ids=[f"{w}x{h}" for w, h in FAR_SIZES])
def test_far_triangles(built, size, path, ids):
    """2D triangles with vertices from 2^12 to 2^25, 1e9, 1e30, +-FLT_MAX, +-inf and NaN, one frame per transform
    (rotated, mirrored, anchored outside [0, 1])."""
    if size == (1920, 1080) and ids:
        pytest.skip("the 1080p frames run with ids off only: the id planes add nothing the smaller frames lack")
    w, h = size
    translucent, stage, want_stage = PATHS[path]
    frames = far_frames(size, translucent)
    r = _renderer(w, h, len(frames), ids, stage)
    for f, (ops, _) in enumerate(frames):
        r.begin_frame(f)
        scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == want_stage
    _check_frames(r, [ref for _, ref in frames], ids)
    r.close()


def test_oracle_draws_no_pixel_for_non_finite_triangles(built):
    """Pins the oracle's behaviour that part D holds the device to: NaN and +-inf vertices are defined inputs, the
    clip collapses the bbox to the frame, no pixel is drawn and the triangle is counted."""
    from oracle import dtro
    o = dtro.Oracle(64, 64)
    for t in ((np.nan, 1, 20, 5, 3, 30), (np.nan,) * 6, (-np.inf, -np.inf, np.inf, -np.inf, 32, np.inf)):
        o.triangle(np.array([t[0], t[1], 1, t[2], t[3], 1, t[4], t[5], 1], F32), (1, 1, 1, 1))
    assert o.counters() == (0, 3)


# ---- E. the other primitive kinds far out -------------------------------------------------------------
FONT = scenes.synthetic_font(51, cell=(8, 10))
BITMAP = scenes.random_texture(11, 7, 52, opaque=False)
OTHER_SIZES = ((64, 64), (257, 131))
LINE_FAR = (0, 1, 37, 1000, 65535, 65536, 10 ** 6)


def _lines(w, h, rng):
    """Lines in all eight octants from points in and around the frame to points up to +-10^6 away."""
    ops = []
    for d in LINE_FAR[1:]:
        for sx, sy in ((1, 0), (1, 1), (0, 1), (-1, 1), (-1, 0), (-1, -1), (0, -1), (1, -1)):
            for steep in (False, True):
                a = (int(rng.integers(-3, w + 3)), int(rng.integers(-3, h + 3)))
                k = int(rng.integers(0, max(1, d // 3) + 1))
                dx, dy = (sx * d + sy * k, sy * d + sx * k) if not steep else (sx * k + sy * d, sy * k + sx * d)
                ops.append(("line", dict(a=a, b=(a[0] + dx, a[1] + dy), color=(*rng.random(3).tolist(), float(rng.choice([0.5, 1.0]))))))
    ops.append(("line", dict(a=(-10 ** 6, -10 ** 6 + 3), b=(10 ** 6, 10 ** 6), color=(1, 1, 1, 1))))
    ops.append(("line", dict(a=(w // 2, -10 ** 6), b=(w // 2 + 1, 10 ** 6), color=(1, 0.5, 0, 0.7))))
    return ops


def _quads(w, h, rng, kind):
    """Rectangles (corners up to +-1e30 and +-inf, sizes at the 65536 loop cap of loop_count) or bitmaps (positions up
    to +-1e30), axis-aligned and rotated."""
    far = [70.0, 65535.0, 65536.0, 65537.0, 1e6, 1e30, np.inf]
    ops = []
    rot = scenes.transform7(0.6, (0.5, 0.5, 0.5), (1.0, 1.0, 1.0))
    for v in far:
        for mn, mx in (((-v, -v), (v, v)), ((3.0, 2.0), (3.0 + v, 9.0)), ((-v, h - 5.0), (w - 2.0, h + v)), ((w - 8.0, -v), (w + v, 5.0)),
                       ((w + v, 3.0), (w + 2 * v, 9.0)), ((-2 * v, -2 * v), (-v, -v))):
            col = (*rng.random(3).tolist(), float(rng.choice([0.5, 1.0])))
            for tr in (scenes.DEFAULT_TRANSFORM, rot):
                if kind == "rectangle":
                    ops.append(("rectangle", dict(mn=mn, mx=mx, color=col, transform=tr)))
                elif np.isfinite(v):
                    # a bitmap's extent is its texture's: the far corner goes in as the position.  Non-finite
                    # corners are left out: the reference samples its texture at NaN coordinates for them
                    ops.append(("bitmap", dict(tex=BITMAP, pos=mn, transform=tr, color=col)))
                    ops.append(("bitmap", dict(tex=BITMAP, pos=(mx[0] - 5.0, mn[1]), transform=tr, color=col)))
    return ops


def _texts(w, h, rng):
    """Strings far off-screen on every side and straddling each edge."""
    ops = []
    for pos in ((-1e9, 10.0), (1e9, 10.0), (10.0, -1e9), (10.0, 1e9), (-30.0, h / 2), (w - 12.0, h / 2), (w / 3, -4.0), (w / 3, h + 3.0),
                (-1e6, -1e6), (float(w), float(h))):
        ops.append(("text", dict(font=FONT, pos=pos, text="Far text 0123", color=(*rng.random(3).tolist(), float(rng.choice([0.6, 1.0]))))))
    return ops


@functools.lru_cache(maxsize=None)
def other_frames(size):
    w, h = size
    rng = np.random.default_rng([w, h, 77])
    frames = []
    for part in (_lines(w, h, rng), _quads(w, h, rng, "rectangle"), _quads(w, h, rng, "bitmap"), _texts(w, h, rng)):
        ops = [("clear", dict(rgb=tuple(rng.random(3).tolist())))] + part
        frames.append((ops, _oracle_frame(w, h, ops)))
    return frames


@pytest.mark.gpu
@pytest.mark.parametrize("ids", [False, True], ids=["ids_off", "ids_on"])
@pytest.mark.parametrize("size", OTHER_SIZES, ids=[f"{w}x{h}" for w, h in OTHER_SIZES])
def test_far_lines_rectangles_bitmaps_text(built, size, ids):
    """Lines to +-10^6 in all eight octants, rectangles and bitmaps with corners to +-1e30 and +-inf and sizes
    at the loop cap, text far off-screen and across each edge: one frame per kind, one flush."""
    w, h = size
    frames = other_frames(size)
    r = _renderer(w, h, len(frames), ids)
    for f, (ops, _) in enumerate(frames):
        r.begin_frame(f)
        scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == api.OPAQUE_SINGLE_KERNEL
    _check_frames(r, [ref for _, ref in frames], ids)
    r.close()
