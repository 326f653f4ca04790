"""CPU checks of the product's per-draw-call HOST arithmetic (dtrenderer_b200/csrc/dtr_host_math.h)
against the unmodified reference (oracle/_ref) -- no GPU involved.  The header is compiled into a
test-only shim (tests/_shim) with the flags the product uses for host code."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import dtro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM_DIR = os.path.join(ROOT, "tests", "_shim")
_f = C.POINTER(C.c_float)
_i = C.POINTER(C.c_int)


@pytest.fixture(scope="module")
def shim():
    so = os.path.join(SHIM_DIR, "libhostmath_shim.so")
    src = os.path.join(SHIM_DIR, "host_math_shim.cpp")
    hdr = os.path.join(ROOT, "dtrenderer_b200", "csrc", "dtr_host_math.h")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                               "-I", os.path.join(ROOT, "dtrenderer_b200", "csrc"), "-o", so, src])
    lib = C.CDLL(so)
    lib.hm_pack_clear.restype = C.c_uint32
    lib.hm_pack_clear.argtypes = [_f]
    lib.hm_rect.restype = C.c_int
    lib.hm_rect.argtypes = [C.c_int, C.c_int, _f, _f, C.c_float, _f, _f, _f, _i, _i, _f]
    return lib


def _oracle(w, h):
    """The unmodified reference where its build exists, else the C restatement pinned to it."""
    kind = "reference" if dtro.available("reference") else "port"
    if not dtro.available(kind):
        pytest.skip("oracle library not built")
    return dtro.Oracle(w, h, kind)


def _fa(v):
    a = np.ascontiguousarray(v, dtype=np.float32)
    return a, a.ctypes.data_as(_f)


# Clears outside [0, 1] and the words they pack to: (int32)(c * 255) spills into the neighbouring channels
# and the top byte.  Those with bit 31 set would read as pending tags in the deferred opaque stage
# (VIS_PENDING, dtr_records.h); tests/test_gpu_colour_range.py renders them.
CLEAR_WORDS = {(0.3, 0.3, 0.7): 0x004C4CB2, (1.5, 1.2, 2.0): 0x017F33FE, (0.0, 0.0, 1e10): 0x80000000,
               (-0.01, 0.0, 0.0): 0xFFFE0000, (0.0, 0.0, -0.004): 0xFFFFFFFF, (0.0, -1.0, 0.0): 0xFFFF0100,
               (130.0, 0.0, 0.0): 0x817E0000, (np.nan, 0.0, 0.0): 0, (np.inf, 0.0, 0.0): 0,
               (0.0, 1 / 255, 1e10): 0x80000100}
CLEAR_CHANNELS = [-np.inf, -1e10, -130.0, -1.0, -0.004, -0.0, 0.0, 0.5, 1.0, float(np.nextafter(np.float32(1), np.float32(2))),
                  2.0, 128.5, 128.51, 130.0, 257.0, 33000.0, 1e5, 1e10, np.inf, np.nan]


def test_clear_colour_packing_matches_reference(shim):
    """DTRRender_Clear's truncating pack (DTRendererRender.cpp:1801-1811), in [0, 1] and over the whole float
    range: negative channels, channels > 1 and >= 128.5, 1e10, +-inf and NaN, every combination of those in
    the three channels, and the words of CLEAR_WORDS."""
    rng = np.random.default_rng(5)
    o = _oracle(4, 3)
    cases = [rng.random(3) for _ in range(1500)]
    cases += [(1.0, 1.0, 1.0), (0.0, 0.0, 0.0), (0.999999, 0.5, 0.003921569), (np.nextafter(np.float32(1), np.float32(0)),) * 3,
              (1 / 255, 2 / 255, 254 / 255), (0.5019608, 0.25, 0.75)]
    cases += list(CLEAR_WORDS)
    cases += [(r, g, b) for r in CLEAR_CHANNELS for g in CLEAR_CHANNELS for b in CLEAR_CHANNELS]
    cases += list(rng.uniform(-300, 300, (500, 3)))
    cases += list(rng.choice([-1, 1], (500, 3)) * 10.0 ** rng.uniform(-4, 12, (500, 3)))
    for rgb in cases:
        a, p = _fa(rgb)
        o.clear(tuple(float(x) for x in a))
        assert int(o.color()[0, 0]) == shim.hm_pack_clear(p), rgb
    for rgb, word in CLEAR_WORDS.items():
        a, p = _fa(rgb)
        assert shim.hm_pack_clear(p) == word, (rgb, hex(word))


def _rect(shim, w, h, mn, mx, rot, anchor, scale, color):
    (a0, p0), (a1, p1), (a2, p2), (a3, p3), (a4, p4) = _fa(mn), _fa(mx), _fa(anchor), _fa(scale), _fa(color)
    bbox = (C.c_int * 4)()
    typ = C.c_int(-1)
    pts = (C.c_float * 8)()
    vis = shim.hm_rect(w, h, p0, p1, C.c_float(rot), p2, p3, p4, bbox, C.byref(typ), pts)
    return vis, tuple(bbox), typ.value, np.array(pts, np.float32).reshape(4, 2)


def test_axis_aligned_rectangle_bounds_match_reference(shim):
    """The pixel rectangle the host hands to the device for DTRRender_Rectangle (rotation 0,
    DTRendererRender.cpp:415-449) is exactly the set of pixels the reference touches -- including
    rectangles hanging over every edge of the frame, fractional corners, scales and anchors."""
    rng = np.random.default_rng(11)
    w, h = 97, 61
    o = _oracle(w, h)
    for _ in range(400):
        mn = rng.uniform(-30, [w + 10, h + 10]).astype(np.float32)
        if rng.random() < 0.3:
            mn = np.floor(mn)
        mx = mn + rng.uniform(0.2, 60, 2).astype(np.float32)
        anchor = (0.5, 0.5) if rng.random() < 0.5 else tuple(rng.random(2))
        scale = (1.0, 1.0) if rng.random() < 0.5 else tuple(rng.uniform(0.3, 2.0, 2))
        tr = dtro.transform7(0.0, (*anchor, 0.0), (*scale, 1.0))
        o.clear((0.0, 0.0, 0.0))
        o.rectangle(mn, mx, (1.0, 1.0, 1.0, 1.0), tr)
        touched = np.argwhere(o.color() != 0)
        vis, bbox, typ, _ = _rect(shim, w, h, mn, mx, 0.0, anchor, scale, (1, 1, 1, 1))
        if touched.size == 0:
            assert not vis, (mn, mx, bbox)
            continue
        assert vis
        y0, x0 = touched.min(0)
        y1, x1 = touched.max(0) + 1
        assert bbox == (x0, y0, x1, y1), (mn, mx, anchor, scale)
        assert touched.shape[0] == (x1 - x0) * (y1 - y0)  # a solid block


def test_rotated_rectangle_bounds_contain_reference_pixels(shim):
    """Rotated rectangles (:450-470): every pixel the reference touches lies inside the bounds the
    host computes (the device then applies the four-edge test inside them)."""
    rng = np.random.default_rng(12)
    w, h = 120, 80
    o = _oracle(w, h)
    for _ in range(300):
        mn = rng.uniform(-20, [w, h]).astype(np.float32)
        mx = mn + rng.uniform(1, 70, 2).astype(np.float32)
        rot = float(rng.uniform(-3.1, 3.1))
        anchor = tuple(rng.random(2))
        scale = tuple(rng.uniform(0.4, 1.8, 2))
        tr = dtro.transform7(rot, (*anchor, 0.0), (*scale, 1.0))
        o.clear((0.0, 0.0, 0.0))
        o.rectangle(mn, mx, (1.0, 1.0, 1.0, 1.0), tr)
        touched = np.argwhere(o.color() != 0)
        vis, bbox, typ, _ = _rect(shim, w, h, mn, mx, rot, anchor, scale, (1, 1, 1, 1))
        if touched.size == 0:
            continue
        assert vis
        y0, x0 = touched.min(0)
        y1, x1 = touched.max(0) + 1
        assert bbox[0] <= x0 and bbox[1] <= y0 and bbox[2] >= x1 and bbox[3] >= y1, (mn, mx, rot, bbox, (x0, y0, x1, y1))
