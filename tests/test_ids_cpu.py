"""Triangle id planes without a GPU: the reference id planes of tests/id_reference.py (what the device's id
planes are compared with) against the oracle's colour plane, which is pinned to the reference, and the C ABI's
id entry points without a context."""
import ctypes as C

import numpy as np

from dtrenderer_b200 import scenes

Z_RESET = np.float32(-3.4028234663852886e38)
INV_255 = np.float32(1) / np.float32(255)


def _port(w, h):
    from id_reference import IdOracle
    return IdOracle(w, h)


def _out_byte(lin):
    """SetPixel's linear -> byte for an opaque fragment: sqrt, * 255, clamp, truncate (fp32)."""
    v = np.sqrt(np.float32(lin)) * np.float32(255)
    return np.uint32(min(v, np.float32(255)))


def _packed(lin_rgb):
    r, g, b = (_out_byte(c) for c in lin_rgb)
    return int((r << 16) | (g << 8) | b)


def _decode(col, colors, clear_packed):
    """Pixel colour -> 1 + triangle position (0: the clear colour); the map must be injective."""
    table = {clear_packed: 0}
    for k, c in enumerate(colors):
        assert c not in table, "two triangles (or a triangle and the clear) share a colour"
        table[c] = k + 1
    lut = np.vectorize(lambda v: table.get(int(v), -1), otypes=[np.int64])
    ids = lut(col)
    assert (ids >= 0).all(), "a pixel has a colour no triangle has"
    return ids.astype(np.uint32)


def _tri_colors(n, rng):
    """n distinct opaque colours (floats) and what an untextured full-bright fragment of each stores."""
    bytes_ = rng.choice(1 << 18, n, replace=False)
    rgb = np.stack([(bytes_ >> 12) & 63, (bytes_ >> 6) & 63, bytes_ & 63], 1).astype(np.float32) * np.float32(4) + np.float32(2)
    cols = np.ones((n, 4), np.float32)
    cols[:, :3] = rgb * INV_255
    packed = [_packed([c * c for c in cols[k, :3]]) for k in range(n)]
    return cols, packed


def _clear_packed(rgb):
    r, g, b = (int(np.float32(c) * np.float32(255)) for c in rgb)
    return (r << 16) | (g << 8) | b


def _check_ids_from_colour(o, colors, clear_rgb):
    ids = o.ids()
    assert np.array_equal(ids, _decode(o.color(), colors, _clear_packed(clear_rgb)))
    assert np.array_equal(ids == 0, o.zbuffer() == Z_RESET)


def test_reference_ids_follow_colour_of_overlapping_exact_triangles():
    w, h, n = 160, 120, 300
    rng = np.random.default_rng(1)
    cols, packed = _tri_colors(n, rng)
    c = rng.integers(0, [w, h], (n, 1, 2))
    p = np.concatenate([c + rng.integers(-25, 26, (n, 3, 2)), rng.uniform(0, 255, (n, 3, 1))], 2).astype(np.float32)
    o = _port(w, h)
    o.clear((0.0, 0.0, 0.0))
    o.triangles(p.reshape(n, 9), cols)
    _check_ids_from_colour(o, packed, (0.0, 0.0, 0.0))
    assert len(np.unique(o.ids())) > n // 3


def test_reference_ids_follow_colour_of_rotated_triangles():
    """Rotated and scaled triangles take the inexact path (sequential fp32 edge accumulation)."""
    w, h, n = 150, 110, 120
    rng = np.random.default_rng(2)
    cols, packed = _tri_colors(n, rng)
    o = _port(w, h)
    o.clear((0.0, 0.0, 0.0))
    for k in range(n):
        p = np.concatenate([rng.uniform(-10, [w + 10, h + 10], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
        o.triangle(p.reshape(-1), cols[k], scenes.transform7(float(rng.uniform(-3, 3)), tuple(rng.random(3)),
                                                             (float(rng.uniform(0.5, 2)), float(rng.uniform(0.5, 2)), 1.0)))
    _check_ids_from_colour(o, packed, (0.0, 0.0, 0.0))


def test_reference_ids_of_a_mesh_are_face_indices():
    """Full-bright mesh whose face k samples texel k only (all three texture coordinates of a face are the
    centre of its own texel): the colour names the face, and id - 1 is that face."""
    w, h = 320, 240
    mesh = scenes.uv_sphere()
    faces = np.asarray(mesh["faces"], np.int32).copy()
    nf = len(faces)
    tw = 64
    th = (nf + tw - 1) // tw
    k = np.arange(nf)
    uv = np.zeros((nf, 3), np.float32)
    uv[:, 0] = ((k % tw) + np.float32(0.5)) / np.float32(tw)
    uv[:, 1] = ((k // tw) + np.float32(0.5)) / np.float32(th)
    faces[:, 3:6] = k[:, None]
    rng = np.random.default_rng(3)
    code = rng.choice(1 << 18, tw * th, replace=False)
    tex = np.full((th, tw, 4), 255, np.uint8)
    tex[..., 0] = (((code >> 12) & 63) * 4 + 2).reshape(th, tw)
    tex[..., 1] = (((code >> 6) & 63) * 4 + 2).reshape(th, tw)
    tex[..., 2] = ((code & 63) * 4 + 2).reshape(th, tw)
    texel = tex.reshape(-1, 4)[:nf].astype(np.float32) * INV_255
    packed = [_packed([texel[f, 0] * texel[f, 0], texel[f, 1] * texel[f, 1], texel[f, 2] * texel[f, 2]]) for f in range(nf)]
    m = dict(mesh, texUV=uv, faces=faces)
    o = _port(w, h)
    o.clear((0.0, 0.0, 0.0))
    o.mesh(m, tex, scenes.SHADE_FULLBRIGHT, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), scenes.view_transforms(4096)[37])
    _check_ids_from_colour(o, packed, (0.0, 0.0, 0.0))
    assert len(np.unique(o.ids())) > 500


def test_reference_ids_mark_exactly_the_depth_written_pixels():
    """Random mixes of blits and translucent triangles: a pixel has an id exactly where its depth left the
    reset value; blits, lines, text and clears never touch the plane; reset_ids restarts it."""
    w, h = 200, 150
    for seed in range(4):
        rng = np.random.default_rng(100 + seed)
        tex = scenes.random_texture(16, 16, seed, opaque=False)
        o = _port(w, h)
        o.clear((0.3, 0.3, 0.3))
        ntri = 0
        for i in range(60):
            kind = int(rng.integers(0, 4))
            col = (*rng.random(3).tolist(), float(rng.choice([1.0, rng.random()])))
            if kind == 0:
                n = int(rng.integers(1, 10))
                c = rng.integers(0, [w, h], (n, 1, 2))
                p = np.concatenate([c + rng.integers(-30, 31, (n, 3, 2)), rng.uniform(0, 255, (n, 3, 1))], 2).astype(np.float32)
                cols = rng.random((n, 4)).astype(np.float32)
                o.triangles(p.reshape(n, 9), cols)
                ntri += n
            elif kind == 1:
                mn = rng.uniform(-20, [w, h]).astype(np.float32)
                o.rectangle(mn, mn + rng.uniform(1, 80, 2).astype(np.float32), col)
            elif kind == 2:
                o.bitmap(tex, rng.uniform(-10, [w, h]).astype(np.float32), scenes.transform7(float(rng.uniform(-3, 3))), col)
            else:
                o.line(rng.integers(0, [w, h]).astype(np.int32), rng.integers(0, [w, h]).astype(np.int32), col)
        ids = o.ids()
        assert np.array_equal(ids > 0, o.zbuffer() != Z_RESET)
        assert ids.max() <= ntri
        o.reset_ids()
        assert not o.ids().any()
        o.triangles(p.reshape(-1, 9), cols)
        assert o.ids().max() <= len(cols)


def test_split_draw_calls_leave_the_oracle_frame_unchanged():
    """The reference ids issue batches and meshes triangle by triangle: colour, depth and counters stay those of
    the oracle drawing the same calls whole."""
    from oracle import dtro
    w, h = 320, 240
    scene = scenes.cfg1_scene(w, h) + scenes.mesh_scene(w, h, textured=True, tex_size=32)[1:]
    whole, split = dtro.Oracle(w, h, "port"), _port(w, h)
    for o in (whole, split):
        o.reset_counters()
        scenes.replay(scene, o)
    assert np.array_equal(whole.color(), split.color())
    assert np.array_equal(whole.zbuffer().view(np.uint32), split.zbuffer().view(np.uint32))
    assert whole.counters() == split.counters()
    assert 0 < split.ids().max() <= whole.counters()[1]


def test_id_entry_points_fail_loudly_without_a_context(built):
    from dtrenderer_b200 import api
    lib = api.load_library()
    out = np.empty(4, np.uint32)
    p = C.c_void_p()
    assert lib.dtr_b200_set_id_output(None, 1) == -1
    assert lib.dtr_b200_set_id_output(None, 0) == -1
    assert lib.dtr_b200_read_ids(None, 0, 1, out.ctypes.data_as(C.c_void_p)) == -1
    assert lib.dtr_b200_frame_id_ptr(None, 0, C.byref(p)) == -1
