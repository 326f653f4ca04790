"""GPU parity (-m gpu): the CUDA back end, driven through the C ABI, against the CPU oracle on the
same seeded scenes, and against the reference-generated golden digests.

Bar (BASELINE.json north_star): coverage and depth-test decisions bit-exact, colour within 1/255
per 8-bit channel, depth within 1e-6 relative.  The tests hold the stronger bar the design
achieves -- depth bit-exact, colour bit-exact -- and print the north_star figures on failure.
Full-size configurations that the oracle cannot finish in seconds are covered by size-independent
properties (split-submission idempotence, band/frame partition invariance, replay determinism).
"""
import numpy as np
import pytest

from dtrenderer_b200 import scenes
from golden_scenes import DIGESTS, SCENES, digest, make_golden

pytestmark = pytest.mark.gpu

COLOR_TOL = 1          # 1/255 per channel
DEPTH_RTOL = 1e-6
Z_RESET = np.float32(-3.4028234663852886e38)


def _oracle(w, h):
    from oracle import dtro
    return dtro.Oracle(w, h, "reference" if dtro.available("reference") else "port")


def _renderer(w, h, frames=1):
    from dtrenderer_b200 import api
    return api.Renderer(w, h, frames, 0)


def _render_gpu(w, h, scene):
    r = _renderer(w, h)
    r.begin_frame(0)
    scenes.replay(scene, r)
    col, z = r.end_frame(0)
    return r, col, z


def _assert_same(col, z, co, zo):
    cov_gpu, cov_ref = z != Z_RESET, zo != Z_RESET
    assert np.array_equal(cov_gpu, cov_ref), f"coverage differs on {(cov_gpu != cov_ref).sum()} px"
    if not np.array_equal(z.view(np.uint32), zo.view(np.uint32)):
        rel = np.abs(z.astype(np.float64) - zo) / np.maximum(np.abs(zo.astype(np.float64)), 1e-30)
        raise AssertionError(f"depth differs on {(z.view(np.uint32) != zo.view(np.uint32)).sum()} px, "
                             f"max rel {rel[cov_ref].max():.3e} (north_star tolerance {DEPTH_RTOL})")
    if not np.array_equal(col, co):
        d = np.abs(col.view(np.uint8).astype(int) - co.view(np.uint8).astype(int))
        raise AssertionError(f"colour differs on {(col != co).sum()} px, max channel delta {d.max()} "
                             f"(north_star tolerance {COLOR_TOL})")


@pytest.mark.parametrize("name", sorted(SCENES))
def test_scene_matches_oracle_and_reference_digest(built, name):
    w, h, make = SCENES[name]
    scene = make()
    o = _oracle(w, h)
    o.reset_counters()
    scenes.replay(scene, o)
    r, col, z = _render_gpu(w, h, scene)
    _assert_same(col, z, o.color(), o.zbuffer())
    st = r.stats()
    assert (st["setPixels"], st["triangles"]) == o.counters()
    g = DIGESTS[name]
    assert digest(col) == g["color_sha256"] and digest(z) == g["depth_sha256"]
    assert (st["setPixels"], st["triangles"]) == (g["setPixels"], g["triangles"])


def test_random_transformed_triangles(built):
    """Rotated / scaled / translucent triangles: every one takes the sequential-accumulation path."""
    rng = np.random.default_rng(321)
    w, h = 500, 380
    o, r = _oracle(w, h), _renderer(w, h)
    r.begin_frame(0)
    for t in (o, r):
        t.clear((0.3, 0.3, 0.3))
    for _ in range(400):
        p = np.concatenate([rng.uniform(-60, [w + 60, h + 60], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
        col = np.concatenate([rng.random(3), [rng.choice([1.0, rng.random()])]]).astype(np.float32)
        tr = scenes.transform7(float(rng.uniform(-3, 3)) if rng.random() < 0.6 else 0.0, tuple(rng.random(3)),
                               (float(rng.uniform(0.3, 2)), float(rng.uniform(0.3, 2)), 1.0))
        for t in (o, r):
            t.triangle(p.reshape(-1), col, tr)
    col, z = r.end_frame(0)
    _assert_same(col, z, o.color(), o.zbuffer())


def test_depth_cull_behind_occluders(built):
    """Region-level depth cull: occluders laid down first (full-frame and partial, flat and slanted,
    one pair translucent -- it still writes depth), then thousands of integer-vertex triangles whose
    depths straddle them: behind, in front, crossing, and EXACTLY on the occluder's plane (strict `>`
    must reject those, and a later triangle one ulp nearer must still pass).  A later flush draws
    into the kept depth buffer (the cull then starts from loaded depths)."""
    rng = np.random.default_rng(99)
    w, h = 320, 200
    o, r = _oracle(w, h), _renderer(w, h)
    o.reset_counters()
    r.begin_frame(0)
    both = (o, r)
    for t in both:
        t.clear((0.1, 0.2, 0.3))

    def quad(x0, y0, x1, y1, zs, col):
        a = np.array([[x0, y0, zs[0], x1, y0, zs[1], x1, y1, zs[2]], [x0, y0, zs[0], x1, y1, zs[2], x0, y1, zs[3]]], np.float32)
        c = np.tile(np.asarray(col, np.float32), (2, 1))
        for t in both:
            t.triangles(a, c, scenes.DEFAULT_TRIANGLE_TRANSFORM)

    quad(-5, -5, w + 5, h + 5, (100, 100, 100, 100), (0.9, 0.1, 0.1, 1.0))          # flat wall at z = 100
    quad(40, 30, 200, 150, (60, 180, 220, 90), (0.1, 0.9, 0.1, 1.0))                # slanted, crosses the wall
    quad(150, 20, 300, 120, (140, 140, 140, 140), (0.2, 0.2, 0.9, 0.5))             # translucent, writes depth
    n = 4000
    c = rng.integers(-10, [w + 10, h + 10], (n, 1, 2))
    xy = c + rng.integers(-24, 25, (n, 3, 2))
    z = rng.uniform(0, 255, (n, 3)).astype(np.float32)
    kind = rng.integers(0, 6, n)
    z[kind == 0] = 100.0                                                            # exactly on the wall: never passes
    z[kind == 1] = np.nextafter(np.float32(100.0), np.float32(200.0))               # one ulp nearer: passes
    z[kind == 2] = rng.uniform(0, 99, (int((kind == 2).sum()), 1)).astype(np.float32)  # flat, behind the wall
    p = np.concatenate([xy, z[..., None]], 2).astype(np.float32).reshape(n, 9)
    cols = rng.random((n, 4)).astype(np.float32)
    cols[rng.random(n) < 0.7, 3] = 1.0
    for k in range(4):
        a, b = n * k // 4, n * (k + 1) // 4
        for t in both:
            t.triangles(p[a:b], cols[a:b], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        if k == 1:
            r.flush()                                                               # the rest starts from depths kept in HBM
    col, zb = r.end_frame(0)
    _assert_same(col, zb, o.color(), o.zbuffer())
    assert r.stats()["setPixels"] == o.counters()[0]


def test_random_blits(built):
    """Rectangles and bilinear bitmaps with random rotation/scale/anchor, partly off-screen."""
    rng = np.random.default_rng(99)
    w, h = 420, 310
    o, r = _oracle(w, h), _renderer(w, h)
    texs = [scenes.random_texture(int(rng.integers(1, 40)), int(rng.integers(1, 40)), s, opaque=bool(s & 1)) for s in range(4)]
    r.begin_frame(0)
    o.reset_counters()  # the reference's counters are process-global
    for t in (o, r):
        t.clear((0.9, 0.8, 0.1))
    for i in range(60):
        tr = scenes.transform7(float(rng.uniform(-3, 3)) if rng.random() < 0.7 else 0.0, (*rng.random(2), 0.0),
                               (float(rng.uniform(0.5, 4)), float(rng.uniform(0.5, 4)), 1.0))
        col = (*rng.random(3).tolist(), float(rng.choice([1.0, rng.random()])))
        if i % 2:
            mn = rng.uniform(-40, [w, h]).astype(np.float32)
            mx = mn + rng.uniform(1, 120, 2).astype(np.float32)
            for t in (o, r):
                t.rectangle(mn, mx, col, tr)
        else:
            pos = rng.uniform(-30, [w, h]).astype(np.float32)
            for t in (o, r):
                t.bitmap(texs[i % 4], pos, tr, col)
    col, z = r.end_frame(0)
    _assert_same(col, z, o.color(), o.zbuffer())
    assert r.stats()["setPixels"] == o.counters()[0]


def test_multi_flush_and_host_buffers(built):
    """A frame split over several flushes, and a frame started from caller-supplied colour+depth,
    give the same result as one submission (the reference draws immediately, so any split must)."""
    w, h = 333, 217
    scene = SCENES["odd_333x217"][2]()
    o = _oracle(w, h)
    scenes.replay(scene, o)
    r = _renderer(w, h)
    r.begin_frame(0)
    for i, (name, kw) in enumerate(scene):
        getattr(r, name)(**kw)
        if i % 3 == 0:
            r.flush()
    col, z = r.end_frame(0)
    _assert_same(col, z, o.color(), o.zbuffer())
    # second half on top of uploaded host buffers
    half = len(scene) // 2
    o1 = _oracle(w, h)
    scenes.replay(scene[:half], o1)
    r2 = _renderer(w, h)
    r2.begin_frame(0, color=o1.color().copy(), z=o1.zbuffer().copy())
    scenes.replay(scene[half:], r2)
    col2, z2 = r2.end_frame(0)
    _assert_same(col2, z2, o.color(), o.zbuffer())


def test_frame_batch_views_and_replay(built):
    """cfg 5 shape: a batch of viewpoints in one flush == each view rendered alone by the oracle;
    replay() reproduces the batch bit for bit."""
    w, h, n = 480, 270, 6
    mesh, tex = scenes.uv_sphere(), scenes.random_texture(64, 64, 1, True)
    ts = scenes.view_transforms(4096)[100:100 + n]
    pos = np.zeros((n, 3), np.float32)
    r = _renderer(w, h, n)
    for f in range(n):
        r.begin_frame(f)
        r.clear((0.5, 0.0, 1.0))
    r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), pos, ts, 0)
    r.flush()
    first = [r.end_frame(f) for f in range(n)]
    total = 0
    for f in range(n):
        o = _oracle(w, h)
        o.reset_counters()
        o.clear((0.5, 0.0, 1.0))
        o.mesh(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), ts[f])
        total += o.counters()[0]
        _assert_same(first[f][0], first[f][1], o.color(), o.zbuffer())
    assert r.stats()["setPixels"] == total
    r.replay()
    for f in range(n):
        col, z = r.end_frame(f)
        assert np.array_equal(col, first[f][0]) and np.array_equal(z.view(np.uint32), first[f][1].view(np.uint32))
    # pipelined replays (pre-raster stages of replay i+1 overlap the raster kernel of replay i on a
    # second stream with a second buffer set), with and without the overlap, and a flush in between
    sp0 = r.stats()["setPixels"]
    for _ in range(5):
        r.replay()
    r.set_replay_overlap(False)
    for _ in range(2):
        r.replay()
    r.set_replay_overlap(True)
    assert r.stats()["setPixels"] == sp0 + 7 * total
    for f in range(n):
        col, z = r.end_frame(f)
        assert np.array_equal(col, first[f][0]) and np.array_equal(z.view(np.uint32), first[f][1].view(np.uint32))
    r.begin_frame(0)
    r.clear((0.5, 0.0, 1.0))
    r.mesh(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), ts[0])
    r.flush()
    for _ in range(3):
        r.replay()
    col, z = r.end_frame(0)
    assert np.array_equal(col, first[0][0]) and np.array_equal(z.view(np.uint32), first[0][1].view(np.uint32))


def test_band_split_equals_full_frame(built):
    """Sort-first band split (cfg 4 shape): rendering the bands separately and stacking them is
    identical to the full frame."""
    w, h = 1024, 768
    scene = scenes.fill_scene(w, h, 30000, seed=5) + scenes.cfg1_scene(w, h)[1:]
    _, full_c, full_z = _render_gpu(w, h, scene)
    out_c, out_z = np.empty_like(full_c), np.empty_like(full_z)
    bounds = [0, 192, 416, 768]
    total = 0
    for y0, y1 in zip(bounds[:-1], bounds[1:]):
        r = _renderer(w, h)
        r.set_band(y0, y1)
        r.begin_frame(0)
        scenes.replay(scene, r)
        c, z = r.end_frame(0)
        out_c[y0:y1], out_z[y0:y1] = c[y0:y1], z[y0:y1]
        total += r.stats()["setPixels"]
    assert np.array_equal(out_c, full_c) and np.array_equal(out_z.view(np.uint32), full_z.view(np.uint32))
    o = _oracle(w, h)
    o.reset_counters()
    scenes.replay(scene, o)
    _assert_same(full_c, full_z, o.color(), o.zbuffer())
    assert total == o.counters()[0]


def test_4k_textured_mesh_full_size_properties(built):
    """cfg 3 at its full 3840x2160 size.  The oracle needs ~1 s for this frame, so it is compared
    directly, and the frame is also rendered as two band halves to check partition invariance."""
    w, h = 3840, 2160
    scene = scenes.mesh_scene(w, h, textured=True, tex_size=1024, overlays=16)
    r, col, z = _render_gpu(w, h, scene)
    o = _oracle(w, h)
    o.reset_counters()
    scenes.replay(scene, o)
    _assert_same(col, z, o.color(), o.zbuffer())
    assert r.stats()["setPixels"] == o.counters()[0]


def test_4k_fill_full_size_properties(built):
    """cfg 4 at full size (1M small triangles, 4K): too slow for the oracle in a test, so check
    (a) order independence is NOT assumed: a 50k-triangle prefix matches the oracle exactly,
    (b) the full run equals the same triangles submitted in 7 chunks (idempotent splitting),
    (c) depth is the per-pixel maximum over covering fragments -> every written depth is >= the
        prefix frame's depth wherever the prefix covered the pixel (z-buffer monotonicity)."""
    w, h, n = 3840, 2160, 1_000_000
    p, color = scenes.small_triangles(w, h, n, seed=7)
    r = _renderer(w, h)
    r.begin_frame(0)
    r.clear((0, 0, 0))
    r.triangles(p, color, scenes.DEFAULT_TRIANGLE_TRANSFORM)
    full_c, full_z = r.end_frame(0)
    r2 = _renderer(w, h)
    r2.begin_frame(0)
    r2.clear((0, 0, 0))
    for k in range(7):
        a, b = n * k // 7, n * (k + 1) // 7
        r2.triangles(p[a:b], color[a:b], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        if k in (1, 4):
            r2.flush()
    c2, z2 = r2.end_frame(0)
    assert np.array_equal(full_c, c2) and np.array_equal(full_z.view(np.uint32), z2.view(np.uint32))
    assert r.stats()["setPixels"] == r2.stats()["setPixels"]
    m = 50_000
    o = _oracle(w, h)
    o.clear((0, 0, 0))
    o.triangles(p[:m], color[:m], scenes.DEFAULT_TRIANGLE_TRANSFORM)
    r3 = _renderer(w, h)
    r3.begin_frame(0)
    r3.clear((0, 0, 0))
    r3.triangles(p[:m], color[:m], scenes.DEFAULT_TRIANGLE_TRANSFORM)
    c3, z3 = r3.end_frame(0)
    _assert_same(c3, z3, o.color(), o.zbuffer())
    cov = z3 != Z_RESET
    assert np.all(full_z[cov] >= z3[cov])


def test_null_arguments_are_silent_noops(built):
    """The reference returns silently on NULL inputs (DTRendererRender.cpp:128,420,1402,1601,1796)."""
    import ctypes as C
    from dtrenderer_b200 import api
    r = _renderer(64, 48)
    lib = r.lib
    assert lib.dtr_b200_clear(r.ctx, None) == 0
    assert lib.dtr_b200_triangle(r.ctx, None, None, None, None, None) == 0
    assert lib.dtr_b200_rectangle(r.ctx, None, None, None, None) == 0
    assert lib.dtr_b200_triangles(r.ctx, 0, None, None, None) == 0
    assert lib.dtr_b200_mesh(r.ctx, 0, None, None, None) == 0
    assert lib.dtr_b200_bitmap(r.ctx, 5, (C.c_float * 2)(0, 0), None, None) == api.load_library().dtr_b200_bitmap(
        r.ctx, 5, (C.c_float * 2)(0, 0), None, None) == -1  # bad texture id is an argument error
    col, z = r.end_frame(0)
    assert np.all(z == Z_RESET)


def test_device_arithmetic_selftest(built):
    """The blend's branch-free sqrt equals IEEE sqrtf on every float in [2^-60, 4), and the output byte
    (out_byte) equals the reference's `(v == 0 ? 0 : sqrtf(v)) * 255`, clamped at 255 and truncated with NaN
    stored as 0, on all 2^32 float bit patterns: +-inf, NaNs, negative and denormal inputs included."""
    r = _renderer(64, 48)
    assert r.selftest() == 0


def test_async_readback_double_buffered(built):
    """read_frames_async + wait_reads returns the same planes as the blocking read, and a flush that
    renders into a frame whose readback is still in flight waits for the copy (the host buffer keeps
    the OLD content of that frame)."""
    import torch
    w, h, n = 320, 200, 4
    mesh, tex = scenes.uv_sphere(), scenes.random_texture(32, 32, 3, True)
    ts = scenes.view_transforms(4096)[7:7 + n]
    pos = np.zeros((n, 3), np.float32)
    r = _renderer(w, h, 2 * n)

    def record(first, clear):
        for f in range(first, first + n):
            r.begin_frame(f)
            r.clear(clear)
        r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), pos, ts, first)

    host = torch.empty((2, n, h, w), dtype=torch.int32, pin_memory=True)
    hz = torch.empty((2, n, h, w), dtype=torch.float32, pin_memory=True)
    record(0, (0.5, 0.0, 1.0))
    r.read_frames_async_ptr(0, n, host[0].data_ptr(), hz[0].data_ptr())
    record(n, (0.1, 0.9, 0.2))          # other half: may overlap the copy
    r.read_frames_async_ptr(n, n, host[1].data_ptr(), hz[1].data_ptr())
    record(0, (0.0, 0.0, 0.0))          # same frames as the first read: must wait for it on the device
    r.flush()
    r.wait_reads()
    for half, clear in ((0, (0.5, 0.0, 1.0)), (1, (0.1, 0.9, 0.2))):
        for f in range(n):
            o = _oracle(w, h)
            o.clear(clear)
            o.mesh(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), ts[f])
            _assert_same(host[half, f].numpy().view(np.uint32), hz[half, f].numpy(), o.color(), o.zbuffer())
    # and the re-rendered first half is what a blocking read sees now
    col, z = r.end_frame(0)
    o = _oracle(w, h)
    o.clear((0.0, 0.0, 0.0))
    o.mesh(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), ts[0])
    _assert_same(col, z, o.color(), o.zbuffer())


@pytest.mark.parametrize("size", [(320, 200), (333, 217), (5, 3)])
def test_bgr24_presentation_readback(built, size):
    """On-device 24-bit DIB encode (SURVEY §8f rank 4): every row is the B,G,R bytes of the oracle's
    0x00RRGGBB pixels, padded to 4 bytes with zeros; three reads in a row alternate the staging
    buffers while the frames are re-rendered in between."""
    import torch
    w, h = size
    n = 3
    r = _renderer(w, h, n)
    pitch = r.bgr24_pitch()
    assert pitch == (3 * w + 3) // 4 * 4
    mesh, tex = scenes.uv_sphere(12, 6), scenes.random_texture(16, 16, 5, True)
    ts = scenes.view_transforms(4096)[100:100 + n]
    host = torch.full((3, n, h, pitch), 0xAB, dtype=torch.uint8, pin_memory=True)
    clears = [(0.5, 0.0, 1.0), (0.1, 0.9, 0.2), (1.0, 1.0, 1.0)]
    for k, clear in enumerate(clears):
        for f in range(n):
            r.begin_frame(f)
            r.clear(clear)
        r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), np.zeros((n, 3), np.float32), ts, 0)
        r.read_frames_bgr24_async_ptr(0, n, host[k].data_ptr())
    r.wait_reads()
    for k, clear in enumerate(clears):
        for f in range(n):
            o = _oracle(w, h)
            o.clear(clear)
            o.mesh(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), ts[f])
            want = np.zeros((h, pitch), np.uint8)
            want[:, :3 * w] = o.color().view(np.uint8).reshape(h, w, 4)[:, :, :3].reshape(h, 3 * w)
            assert np.array_equal(host[k, f].numpy(), want)


def test_tiny_translucent_overlaps_keep_submission_order(built):
    """Thousands of 1-20 pixel triangles, half of them translucent, piled on a small area: fragments
    of many triangles share one shading batch, and the same pixel occurs several times in a batch.
    Blending is order dependent, so any reordering inside the fragment queue shows up here."""
    rng = np.random.default_rng(2024)
    w, h, n = 96, 80, 6000
    c = rng.integers(8, [w - 8, h - 8], (n, 1, 2)).astype(np.float32)
    p = np.concatenate([c + rng.integers(-5, 6, (n, 3, 2)), rng.uniform(0, 255, (n, 3, 1))], 2).astype(np.float32)
    color = rng.random((n, 4)).astype(np.float32)
    color[::2, 3] = 1.0
    o, r = _oracle(w, h), _renderer(w, h)
    o.reset_counters()
    r.begin_frame(0)
    for t in (o, r):
        t.clear((0.2, 0.4, 0.6))
        t.triangles(p.reshape(n, 9), color, scenes.DEFAULT_TRIANGLE_TRANSFORM)
    col, z = r.end_frame(0)
    _assert_same(col, z, o.color(), o.zbuffer())
    assert r.stats()["setPixels"] == o.counters()[0]


def test_band_split_peer_write_two_gpus(built):
    """Sort-first bands over peer memory: the second GPU's raster kernel writes its band straight into
    the first GPU's frame planes; the assembled frame equals the single-GPU frame.  (Needs 2 GPUs.)"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    w, h = 1024, 768
    scene = scenes.fill_scene(w, h, 20000, seed=11) + scenes.cfg1_scene(w, h)[1:]
    _, full_c, full_z = _render_gpu(w, h, scene)
    from dtrenderer_b200 import api
    r0, r1 = api.Renderer(w, h, 1, 0), api.Renderer(w, h, 1, 1)
    r1.enable_peer_access(0)
    c0, z0 = r0.frame_device_ptrs(0)
    r1.set_output_planes(c0, z0)
    r0.set_band(0, 352)
    r1.set_band(352, h)
    for r in (r0, r1):
        r.begin_frame(0)
        scenes.replay(scene, r)
        r.flush()
    r1.sync()
    col, z = r0.end_frame(0)
    assert np.array_equal(col, full_c) and np.array_equal(z.view(np.uint32), full_z.view(np.uint32))
    assert r0.stats()["setPixels"] + r1.stats()["setPixels"] == _render_gpu(w, h, scene)[0].stats()["setPixels"]


def test_debug_marker_overlay_matches_reference_default_build(built):
    """SURVEY §8f rank 1: with dtr_b200_set_debug_markers the rectangle / bitmap calls also draw the
    DTR_DEBUG_RENDER overlay, and the frame equals the reference's DEFAULT build (markers on)."""
    from oracle import dtro
    if not dtro.available("reference_markers"):
        pytest.skip("oracle/_ref/libdtr_ref_markers.so not built")
    rng = np.random.default_rng(5)
    w, h = 640, 400
    texs = [scenes.random_texture(24, 17, 2, False), scenes.random_texture(40, 40, 3, True)]
    o = dtro.Oracle(w, h, "reference_markers")
    r = _renderer(w, h)
    r.set_debug_markers(True)
    r.begin_frame(0)
    o.reset_counters()
    for t in (o, r):
        t.clear((0.5, 0.0, 1.0))
    scene = scenes.cfg1_scene(w, h)[1:]
    scenes.replay(scene, o)
    scenes.replay(scene, r)
    for i in range(24):
        tr = scenes.transform7(float(rng.uniform(-2, 3)) if i % 3 else 0.0, (*rng.random(2), 0.0),
                               (float(rng.uniform(0.5, 3)), float(rng.uniform(0.5, 3)), 1.0))
        col = (*rng.random(3).tolist(), float(rng.choice([1.0, rng.random()])))
        if i % 2:
            mn = rng.uniform(-30, [w, h]).astype(np.float32)
            mx = mn + rng.uniform(1, 150, 2).astype(np.float32)
            for t in (o, r):
                t.rectangle(mn, mx, col, tr)
        else:
            pos = rng.uniform(-20, [w, h]).astype(np.float32)
            for t in (o, r):
                t.bitmap(texs[(i // 2) % 2], pos, tr, col)
    col, z = r.end_frame(0)
    _assert_same(col, z, o.color(), o.zbuffer())
    assert r.stats()["setPixels"] == o.counters()[0]


def test_device_premultiply_matches_asset_loader_pass(built):
    """SURVEY §8f rank 3: straight-alpha upload + device premultiply == DTRAsset_LoadBitmap's pass,
    over every (channel value, alpha) pair; and a bitmap drawn from it equals the oracle's."""
    from oracle import dtro
    kind = "reference" if dtro.available("reference") else "port"
    v, a = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8))
    rgba = np.ascontiguousarray(np.stack([v, v[::-1], v.T, a], -1))
    want = dtro.premultiply_bitmap(rgba, kind)
    r = _renderer(320, 300)
    tid = r.upload_bitmap_straight(rgba)
    assert np.array_equal(r.read_texture(tid, rgba.shape), want)
    o = _oracle(320, 300)
    r.begin_frame(0)
    for t in (o, r):
        t.clear((0.3, 0.6, 0.2))
    tr = scenes.transform7(0.2, (0.5, 0.5, 0.0), (1.1, 0.9, 1.0))
    o.bitmap(want, (20.0, 15.0), tr, (1.0, 0.9, 0.8, 0.9))
    r.bitmap_id(tid, (20.0, 15.0), tr, (1.0, 0.9, 0.8, 0.9))
    col, z = r.end_frame(0)
    _assert_same(col, z, o.color(), o.zbuffer())


@pytest.mark.parametrize("seed,size", [(1, (257, 131)), (2, (640, 360)), (3, (96, 1000)), (4, (1023, 65))])
def test_fuzz_mixed_primitives(built, seed, size):
    """Random interleavings of every primitive kind (exact and transformed triangles, textured
    triangles, mesh, rectangles, bitmaps, lines, text, clears in mid-frame) at awkward sizes, split
    over random flushes: the device frame, depth and SetPixels counter equal the oracle's."""
    rng = np.random.default_rng(1000 + seed)
    w, h = size
    texs = [scenes.random_texture(int(rng.integers(2, 48)), int(rng.integers(2, 48)), 10 + i, opaque=bool(i & 1)) for i in range(3)]
    font = scenes.synthetic_font(20 + seed)
    mesh = scenes.uv_sphere(14, 7)
    o, r = _oracle(w, h), _renderer(w, h)
    o.reset_counters()
    r.begin_frame(0)
    both = (o, r)
    for t in both:
        t.clear((0.2, 0.5, 0.4))
    for i in range(140):
        kind = int(rng.integers(0, 9))
        col = (*rng.random(3).tolist(), float(rng.choice([1.0, rng.random()])))
        tr = scenes.transform7(float(rng.uniform(-3, 3)) if rng.random() < 0.5 else 0.0, (*rng.random(2), 0.0),
                               (float(rng.uniform(0.4, 2.5)), float(rng.uniform(0.4, 2.5)), 1.0))
        if kind == 0:      # integer-vertex triangles (exact path), a small batch
            n = int(rng.integers(1, 40))
            c = rng.integers(-10, [w + 10, h + 10], (n, 1, 2))
            p = np.concatenate([c + rng.integers(-30, 31, (n, 3, 2)), rng.uniform(0, 255, (n, 3, 1))], 2).astype(np.float32)
            cols = rng.random((n, 4)).astype(np.float32)
            cols[rng.random(n) < 0.6, 3] = 1.0
            for t in both:
                t.triangles(p.reshape(n, 9), cols, scenes.DEFAULT_TRIANGLE_TRANSFORM)
        elif kind == 1:    # transformed triangle (sequential-accumulation path)
            p = np.concatenate([rng.uniform(-40, [w + 40, h + 40], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
            tri_tr = scenes.transform7(tr[0], tuple(rng.random(3)), (tr[4], tr[5], 1.0))
            for t in both:
                t.triangle(p.reshape(-1), col, tri_tr)
        elif kind == 2:
            p = np.concatenate([rng.integers(-20, [w + 20, h + 20], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
            uv = (rng.random(6) * 0.999).astype(np.float32)
            for t in both:
                t.textured_triangle(p.reshape(-1), uv, texs[i % 3], col, scenes.DEFAULT_TRIANGLE_TRANSFORM)
        elif kind == 3:
            mn = rng.uniform(-30, [w, h]).astype(np.float32)
            mx = mn + rng.uniform(1, 120, 2).astype(np.float32)
            for t in both:
                t.rectangle(mn, mx, col, tr)
        elif kind == 4:
            pos = rng.uniform(-30, [w, h]).astype(np.float32)
            for t in both:
                t.bitmap(texs[i % 3], pos, tr, col)
        elif kind == 5:
            a = rng.integers(-20, [w + 20, h + 20]).astype(np.int32)
            b = rng.integers(-20, [w + 20, h + 20]).astype(np.int32)
            for t in both:
                t.line(a, b, col)
        elif kind == 6:
            s = bytes(rng.integers(32, 127, int(rng.integers(1, 16))).astype(np.uint8))
            pos = rng.uniform(-15, [w, h + 8]).astype(np.float32)
            for t in both:
                t.text(font, pos, s, col)
        elif kind == 7 and i % 3 == 0:
            mode = int(rng.integers(0, 3))
            view = scenes.view_transforms(4096)[int(rng.integers(0, 4096))]
            for t in both:
                t.mesh(mesh, texs[1], mode, (1, -1, 1), (1, 1, 1, 1), (0.1, 0.0, 0.0), view)
        elif kind == 8 and rng.random() < 0.15:
            rgb = tuple(rng.random(3))
            for t in both:
                t.clear(rgb)
        if rng.random() < 0.1:
            r.flush()
    col_, z_ = r.end_frame(0)
    _assert_same(col_, z_, o.color(), o.zbuffer())
    assert r.stats()["setPixels"] == o.counters()[0]
