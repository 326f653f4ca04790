"""Colours outside [0, 1] in every raster stage, against the CPU oracle (-m gpu).

The C ABI takes any float as a colour or an alpha, and the reference defines what each one gives:

- DTRRender_Clear packs (int32)(c * 255) per channel with shifts, so negative, large and non-finite channels
  spill into the neighbouring channels and into the top byte (tests/test_host_math_cpu.py pins the words).
  The deferred opaque stage tells a pending pixel by bit 31 of its colour word (VIS_PENDING, dtr_records.h),
  and the pixels no triangle covers keep the clear colour: a pass over a frame cleared to a word with that
  bit must take the single raster kernel instead.
- SetPixel stores sqrtf of the blend (0 stays 0), times 255, clamped at 255 and truncated: every blend >= 1
  gives 255, +inf included, and NaN (a negative blend, inf * 0) gives 0.  A blend reaches +inf through an
  infinite channel, a finite one whose square overflows, or alpha = -inf over a non-zero destination byte; a
  negative denormal blend (a tiny channel under a negative alpha) gives 0.

Every check compares colour and depth bit for bit and the SetPixels counter (with ids on, the id planes too).
No colour here selects a texel or a record: geometry and uv stay in range.
"""
import functools

import numpy as np
import pytest

from dtrenderer_b200 import api, scenes
from test_gpu_launch_shapes import _check_frames, _oracle_frame, _renderer
from test_host_math_cpu import CLEAR_WORDS

pytestmark = pytest.mark.gpu

F32 = np.float32
SIZES = ((257, 131), (333, 217))
SIZE_IDS = [f"{w}x{h}" for w, h in SIZES]
STAGES = {"single": api.OPAQUE_SINGLE_KERNEL, "two_kernels": api.OPAQUE_TWO_KERNELS, "one_kernel": api.OPAQUE_ONE_KERNEL}
PENDING = 0x80000000       # VIS_PENDING
Z_RESET = F32(-3.4028234663852886e38)


def _rgb_id(rgb):
    return "_".join(f"{c:g}" for c in rgb)


# ---- A. clear colours x raster stages -------------------------------------------------------------
# The words of CLEAR_WORDS (bit 31 set: tag 0, tag 256, tags far past the record buffer; bit 31 clear with a
# non-zero top byte; NaN and inf packed to 0) and in-range controls.
CLEARS = list(CLEAR_WORDS) + [(0.0, 0.0, np.nan), (0.0, 0.0, -np.inf), (0.2, 0.6, 0.9), (1.0, 1.0, 1.0), (0.0, 0.0, 0.0)]


def _cleared_word(rgb):
    """The word the oracle's clear leaves in every pixel."""
    from oracle import dtro
    o = dtro.Oracle(1, 1, "port")
    o.clear(rgb)
    return int(o.color()[0, 0])


@functools.lru_cache(maxsize=None)
def _opaque_content(size, k=0):
    """An all-opaque pass that the host defers over a cleared frame: two integer-vertex batches (the queued exact
    path; primitive 0 of the pass is an untextured one of them), a rotated (inexact) triangle, an exact textured
    triangle with an opaque texture and a small mesh in each light mode.  The triangles are small and scattered,
    so most busy regions keep pixels that no triangle covers and that show the clear colour."""
    w, h = size
    rng = np.random.default_rng([w, h, k])
    tex = scenes.random_texture(9, 7, 3 + k, opaque=True)
    mesh = scenes.uv_sphere(10, 5)
    n = 80
    c = rng.integers(10, [w - 10, h - 10], (n, 1, 2))
    p = np.concatenate([c + rng.integers(-9, 10, (n, 3, 2)), rng.uniform(0, 255, (n, 3, 1))], 2).astype(F32).reshape(n, 9)
    p[0] = (10, 10, 50, 60, 14, 50, 30, 50, 50)
    col = rng.random((n, 4)).astype(F32)
    col[:, 3] = 1.0
    tri = np.array([0.6, 0.2, 90, 0.8, 0.25, 90, 0.7, 0.5, 90], F32) * np.array([w, h, 1] * 3, F32)
    ttri = np.round(np.array([0.1, 0.6, 120, 0.35, 0.62, 120, 0.2, 0.95, 120], F32) * np.array([w, h, 1] * 3, F32))
    ops = [("triangles", dict(p=p[:n // 2], color=col[:n // 2], transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)),
           ("triangle", dict(p=tri, color=(0.7, 0.2, 0.4, 1.0), transform=scenes.transform7(0.4, (0.33, 0.33, 0.33), (1.1, 0.9, 1.0)))),
           ("textured_triangle", dict(p=ttri, uv=np.array([0.05, 0.1, 0.95, 0.2, 0.4, 0.9], F32), tex=tex, color=(0.9, 0.8, 0.6, 1.0),
                                      transform=scenes.DEFAULT_TRIANGLE_TRANSFORM))]
    for mode in (scenes.SHADE_FULLBRIGHT, scenes.SHADE_FLAT, scenes.SHADE_GOURAUD):
        ops.append(("mesh", dict(mesh=mesh, tex=tex, light_mode=mode, light_vector=(1, -1, 1), light_color=(0.9, 0.7, 0.5, 1.0),
                                 pos=(-0.5 + 0.5 * mode, 0.3 - 0.1 * k, 0.0), transform=scenes.transform7(30.0 * (mode + k), (0, 1, 0), (0.25, 0.25, 0.25)))))
    ops.append(("triangles", dict(p=p[n // 2:], color=col[n // 2:], transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    return ops


def _clear_ops(size, rgb, k=0):
    return [("clear", dict(rgb=rgb))] + _opaque_content(size, k)


@functools.lru_cache(maxsize=None)
def _clear_frame(size, rgb, k=0):
    ref = _oracle_frame(*size, _clear_ops(size, rgb, k))
    # the pass leaves busy tiles with uncovered pixels, where the deferred stage would read the clear word
    cov, (h, w) = ref[1] != Z_RESET, ref[1].shape
    mixed = [(y, x) for y in range(0, h, 32) for x in range(0, w, 64) if cov[y:y + 32, x:x + 64].any() and not cov[y:y + 32, x:x + 64].all()]
    assert len(mixed) > 4, mixed
    return ref


@pytest.mark.parametrize("size", SIZES, ids=SIZE_IDS)
@pytest.mark.parametrize("stage", sorted(STAGES))
@pytest.mark.parametrize("rgb", CLEARS, ids=[_rgb_id(c) for c in CLEARS])
def test_clear_colour_in_every_stage(built, rgb, stage, size):
    """A clear outside [0, 1], then an all-opaque pass, under each opaque-stage setting.  The pass runs the
    selected stage unless the cleared word has bit 31 set; then it runs the single kernel."""
    w, h = size
    r = _renderer(w, h, 1, False, STAGES[stage])
    r.begin_frame(0)
    scenes.replay(_clear_ops(size, rgb), r)
    r.flush()
    ran = r.last_pass_stage()
    _check_frames(r, [_clear_frame(size, rgb)], False)
    want = api.OPAQUE_SINGLE_KERNEL if _cleared_word(rgb) & PENDING else STAGES[stage]
    assert ran == want, (hex(_cleared_word(rgb)), ran)
    r.close()


BATCH_CLEARS = [(0.3, 0.3, 0.7), (0.9, 0.1, 0.5), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0), (0.2, 0.6, 0.1)]


@pytest.mark.parametrize("ids", [False, True], ids=["ids_off", "ids_on"])
@pytest.mark.parametrize("stage", ["two_kernels", "one_kernel"])
def test_one_tag_like_clear_sends_its_batch_to_the_single_kernel(built, stage, ids):
    """Five frames in one flush, each cleared and then given its own all-opaque pass: with in-range clears the
    batch takes the selected deferred form; when the middle frame's clear has bit 31 set, the whole pass runs
    the single kernel, and every frame is still right."""
    size = SIZES[1]
    w, h = size
    for odd in (None, (-0.01, 0.0, 0.0), (0.0, 0.0, 1e10), (130.0, 0.0, 0.0)):
        clears = list(BATCH_CLEARS)
        if odd is not None:
            clears[2] = odd
        r = _renderer(w, h, len(clears), ids, STAGES[stage])
        for f, rgb in enumerate(clears):
            r.begin_frame(f)
            scenes.replay(_clear_ops(size, rgb, f), r)
        r.flush()
        assert r.last_pass_stage() == (STAGES[stage] if odd is None else api.OPAQUE_SINGLE_KERNEL), odd
        try:
            _check_frames(r, [_clear_frame(size, rgb, f) for f, rgb in enumerate(clears)], ids)
        except AssertionError as e:
            raise AssertionError(f"odd clear {odd}: {e}") from None
        r.close()


@pytest.mark.parametrize("stage", sorted(STAGES))
def test_out_of_range_mid_frame_clears(built, stage):
    """The same clears recorded after a draw call: a raw clear record, which always takes the single kernel.
    One frame per clear, in one flush; each frame is cleared in range first, drawn, cleared again, drawn on."""
    size = SIZES[0]
    w, h = size
    frames = []
    for f, rgb in enumerate(CLEARS):
        content = _opaque_content(size, f)
        ops = [("clear", dict(rgb=(0.3, 0.3, 0.7)))] + content[:2] + [("clear", dict(rgb=rgb))] + content[2:]
        frames.append((ops, _oracle_frame(w, h, ops)))
    r = _renderer(w, h, len(frames), False, STAGES[stage])
    for f, (ops, _) in enumerate(frames):
        r.begin_frame(f)
        scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == api.OPAQUE_SINGLE_KERNEL
    _check_frames(r, [ref for _, ref in frames], False)
    r.close()


# ---- B. draw colours outside [0, 1], every primitive kind -------------------------------------------
FLT_MAX = float(np.finfo(F32).max)
ABOVE_1, BELOW_1 = float(np.nextafter(F32(1), F32(2))), float(np.nextafter(F32(1), F32(0)))
# 2e19: the square overflows; 1e-20: the square is a denormal, negative once premultiplied by a negative alpha
CHANNELS = (-2.0, -0.0, 0.0, 1e-20, ABOVE_1, 3.0, 2e19, FLT_MAX, np.inf, -np.inf, np.nan)
ALPHAS = (1.0, 0.0, BELOW_1, ABOVE_1, -0.5, 1.5, np.inf, -np.inf, np.nan)
LIGHT_VECTORS = ((1.0, -1.0, 1.0), (0.0, 0.0, 0.0), (1e30, 0.0, 0.0), (np.inf, 0.0, 0.0), (np.nan, 0.0, 0.0))
CELL_W, CELL_H = 16, 8
KINDS = ("exact_triangles", "rotated_triangles", "textured_opaque", "textured_translucent", "mesh",
         "rectangle_fill", "rectangle_rotated", "bitmap", "line", "text")
OPAQUE_KINDS = ("exact_triangles", "rotated_triangles", "textured_opaque", "mesh")  # what the deferred stage takes
ROTATED = scenes.transform7(0.35, (0.33, 0.33, 0.33), (1.1, 0.9, 1.0))
TEX_OPAQUE = scenes.random_texture(7, 5, 21, opaque=True)
TEX_TRANSLUCENT = scenes.random_texture(12, 6, 22, opaque=False)
FONT = scenes.synthetic_font(23, cell=(8, 10))
MESH = scenes.uv_sphere(8, 4)
UV = np.array([0.05, 0.1, 0.95, 0.2, 0.4, 0.9], F32)


def _colours(alphas):
    """(r, g, b, a): per alpha, for every channel value a grey colour (r = g = b: the single-root path at
    alpha 1) and a non-grey one."""
    n = len(CHANNELS)
    out = []
    for a in alphas:
        for i, v in enumerate(CHANNELS):
            out += [(v, v, v, a), (v, CHANNELS[(i + 3) % n], CHANNELS[(i + 7) % n], a)]
    return np.array(out, F32)


def _background(w, h):
    """A clear and opaque one-row rectangles: within every cell each destination channel holds the bytes 0,
    127 and 255 (alpha -inf over byte 0 blends to inf * 0 = NaN, over the others to inf)."""
    ops = [("clear", dict(rgb=(0.0, 1.0, 0.5)))]
    for y in range(h):
        if y % 3:
            col = (1.0, 0.5, 0.0, 1.0) if y % 3 == 1 else (0.5, 0.0, 1.0, 1.0)
            ops.append(("rectangle", dict(mn=(0.0, float(y)), mx=(float(w), float(y + 1)), color=col, transform=scenes.DEFAULT_TRANSFORM)))
    return ops


def _cells(kind, colours, first, size):
    """One primitive of `kind` per colour, each in its own CELL_W x CELL_H cell from cell `first` on."""
    w, h = size
    cols = w // CELL_W
    assert first + len(colours) <= cols * (h // CELL_H), (kind, first, len(colours), size)
    xy = [(((first + i) % cols) * CELL_W, ((first + i) // cols) * CELL_H) for i in range(len(colours))]
    if kind in ("exact_triangles", "rotated_triangles"):
        p = np.array([[x + 1, y + 1, 10, x + 15, y + 2, 10, x + 5, y + 7, 10] for x, y in xy], F32)
        return [("triangles", dict(p=p, color=colours, transform=ROTATED if kind == "rotated_triangles" else scenes.DEFAULT_TRIANGLE_TRANSFORM))]
    ops = []
    # the mesh: a small sphere per cell, light mode and light vector cycled over the cells
    ms = min((CELL_W / 2 - 1) / (w / 2), (CELL_H / 2 - 0.5) / (h / 2)) / 0.8
    for i, ((x, y), c) in enumerate(zip(xy, colours)):
        c = tuple(float(v) for v in c)
        if kind in ("textured_opaque", "textured_translucent"):
            p = np.array([x + 1, y + 1, 10, x + 15, y + 2, 10, x + 5, y + 7, 10], F32)
            ops.append(("textured_triangle", dict(p=p, uv=UV, tex=TEX_OPAQUE if kind == "textured_opaque" else TEX_TRANSLUCENT, color=c,
                                                  transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
        elif kind == "mesh":
            pos = ((x + CELL_W / 2) / (w / 2) - 1, (y + CELL_H / 2) / (h / 2) - 1, 0.0)
            ops.append(("mesh", dict(mesh=MESH, tex=TEX_OPAQUE, light_mode=i % 3, light_vector=LIGHT_VECTORS[(i // 3) % len(LIGHT_VECTORS)],
                                     light_color=c, pos=pos, transform=scenes.transform7(20.0 * i, (0, 1, 0), (ms, ms, ms)))))
        elif kind == "rectangle_fill":
            ops.append(("rectangle", dict(mn=(x + 1.0, y + 1.0), mx=(x + 15.0, y + 7.0), color=c, transform=scenes.DEFAULT_TRANSFORM)))
        elif kind == "rectangle_rotated":
            ops.append(("rectangle", dict(mn=(x + 2.0, y + 2.0), mx=(x + 14.0, y + 6.0), color=c,
                                          transform=scenes.transform7(0.5, (0.5, 0.5, 0.5), (0.8, 0.8, 1.0)))))
        elif kind == "bitmap":
            ops.append(("bitmap", dict(tex=TEX_TRANSLUCENT, pos=(x + 2.0, y + 1.0), transform=scenes.DEFAULT_TRANSFORM, color=c)))
        elif kind == "line":
            ops.append(("line", dict(a=(x + 1, y + 1), b=(x + 14, y + 6), color=c)))
        elif kind == "text":
            ops.append(("text", dict(font=FONT, pos=(x + 1.0, y + 6.0), text="Ag", color=c)))
        else:
            raise AssertionError(kind)
    return ops


@functools.lru_cache(maxsize=None)
def _mixed_scene(kind, size):
    ops = _background(*size) + _cells(kind, _colours(ALPHAS), 0, size)
    return ops, _oracle_frame(*size, ops)


@pytest.mark.parametrize("size", SIZES, ids=SIZE_IDS)
@pytest.mark.parametrize("kind", KINDS)
def test_draw_colours_outside_unit_range(built, kind, size):
    """Every primitive kind in every (colour, alpha) of CHANNELS x ALPHAS, grey and not, over a destination
    of bytes 0, 127 and 255.  The pass blends, so it runs the single kernel."""
    w, h = size
    ops, ref = _mixed_scene(kind, size)
    r = _renderer(w, h, 1, False)
    r.begin_frame(0)
    scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == api.OPAQUE_SINGLE_KERNEL
    _check_frames(r, [ref], False)
    r.close()


@functools.lru_cache(maxsize=None)
def _opaque_scene(size):
    """Alpha-1 triangles with out-of-range rgb over an in-range clear: the structured colours of _colours and
    random picks of CHANNELS per channel, in each kind the deferred stage takes."""
    rng = np.random.default_rng(list(size))
    ops = [("clear", dict(rgb=(0.25, 0.5, 0.75)))]
    for k, kind in enumerate(OPAQUE_KINDS):
        cols = np.concatenate([_colours((1.0,)), np.c_[rng.choice(np.array(CHANNELS, F32), (40, 3)), np.ones(40, F32)]])
        ops += _cells(kind, cols, k * 64, size)
    return ops, _oracle_frame(*size, ops)


@pytest.mark.parametrize("size", SIZES, ids=SIZE_IDS)
@pytest.mark.parametrize("stage", sorted(STAGES))
def test_opaque_colours_outside_unit_range_in_every_stage(built, stage, size):
    """A pass made only of alpha-1 triangles with out-of-range rgb (exact, rotated, textured, meshes with
    out-of-range light colours and degenerate light vectors in all three modes) takes the selected stage."""
    w, h = size
    ops, ref = _opaque_scene(size)
    r = _renderer(w, h, 1, False, STAGES[stage])
    r.begin_frame(0)
    scenes.replay(ops, r)
    r.flush()
    assert r.last_pass_stage() == STAGES[stage]
    _check_frames(r, [ref], False)
    r.close()
