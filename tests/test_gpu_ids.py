"""Triangle id planes on the device (-m gpu): dtr_b200_set_id_output / read_ids / frame_id_ptr.

The id planes must equal the reference ids (tests/id_reference.py, derived from the CPU oracle) bit for bit,
in every opaque-stage mode, and turning them on must leave colour, depth and the work counters exactly as
they are with ids off.
"""
import ctypes as C

import numpy as np
import pytest

from dtrenderer_b200 import scenes
from golden_scenes import SCENES

pytestmark = pytest.mark.gpu

STAGES = (0, 1, 2)  # api.OPAQUE_SINGLE_KERNEL, OPAQUE_TWO_KERNELS, OPAQUE_ONE_KERNEL
ERR_ARG = -1


def _port(w, h):
    from id_reference import IdOracle
    o = IdOracle(w, h)
    o.reset_counters()
    return o


def _renderer(w, h, frames=1, ids=True, stage=2):
    from dtrenderer_b200 import api
    r = api.Renderer(w, h, frames, 0)
    r.set_opaque_stage(stage)
    if ids:
        r.set_id_output(True)
    return r


def _same_frame(a, b):
    (ca, za), (cb, zb) = a, b
    assert np.array_equal(ca, cb) and np.array_equal(za.view(np.uint32), zb.view(np.uint32))


def _stats(r):
    s = r.stats()
    return s["setPixels"], s["triangles"], s["primitives"], s["listEntries"], s["kernelLaunches"]


def _render(w, h, ops, ids, stage):
    """ops: (name, kwargs) draw calls and ("flush", None); returns (colour, depth), ids or None, counters."""
    r = _renderer(w, h, ids=ids, stage=stage)
    r.begin_frame(0)
    for name, kw in ops:
        if name == "flush":
            r.flush()
        else:
            getattr(r, name)(**kw)
    frame = r.end_frame(0)
    return frame, (r.read_ids(0, 1)[0] if ids else None), _stats(r)


def _check_against_reference(w, h, ops):
    o = _port(w, h)
    scenes.replay([op for op in ops if op[0] != "flush"], o)
    for stage in STAGES:
        off, _, st_off = _render(w, h, ops, False, stage)
        on, ids, st_on = _render(w, h, ops, True, stage)
        _same_frame(on, off)
        assert st_on == st_off, (stage, st_on, st_off)
        _same_frame(on, (o.color(), o.zbuffer()))
        assert np.array_equal(ids, o.ids()), f"stage {stage}: ids differ on {(ids != o.ids()).sum()} px"


@pytest.mark.parametrize("name", sorted(SCENES))
def test_parity_scene_ids_equal_reference(built, name):
    w, h, make = SCENES[name]
    _check_against_reference(w, h, make())


def _fuzz_ops(seed, size):
    """The draw-call mix of test_gpu_parity.test_fuzz_mixed_primitives (same seeds), flushes included."""
    rng = np.random.default_rng(1000 + seed)
    w, h = size
    texs = [scenes.random_texture(int(rng.integers(2, 48)), int(rng.integers(2, 48)), 10 + i, opaque=bool(i & 1)) for i in range(3)]
    font = scenes.synthetic_font(20 + seed)
    mesh = scenes.uv_sphere(14, 7)
    ops = [("clear", dict(rgb=(0.2, 0.5, 0.4)))]
    for i in range(140):
        kind = int(rng.integers(0, 9))
        col = (*rng.random(3).tolist(), float(rng.choice([1.0, rng.random()])))
        tr = scenes.transform7(float(rng.uniform(-3, 3)) if rng.random() < 0.5 else 0.0, (*rng.random(2), 0.0),
                               (float(rng.uniform(0.4, 2.5)), float(rng.uniform(0.4, 2.5)), 1.0))
        if kind == 0:
            n = int(rng.integers(1, 40))
            c = rng.integers(-10, [w + 10, h + 10], (n, 1, 2))
            p = np.concatenate([c + rng.integers(-30, 31, (n, 3, 2)), rng.uniform(0, 255, (n, 3, 1))], 2).astype(np.float32)
            cols = rng.random((n, 4)).astype(np.float32)
            cols[rng.random(n) < 0.6, 3] = 1.0
            ops.append(("triangles", dict(p=p.reshape(n, 9), color=cols, transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
        elif kind == 1:
            p = np.concatenate([rng.uniform(-40, [w + 40, h + 40], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
            ops.append(("triangle", dict(p=p.reshape(-1), color=col, transform=scenes.transform7(tr[0], tuple(rng.random(3)), (tr[4], tr[5], 1.0)))))
        elif kind == 2:
            p = np.concatenate([rng.integers(-20, [w + 20, h + 20], (3, 2)), rng.uniform(0, 255, (3, 1))], 1).astype(np.float32)
            uv = (rng.random(6) * 0.999).astype(np.float32)
            ops.append(("textured_triangle", dict(p=p.reshape(-1), uv=uv, tex=texs[i % 3], color=col, transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
        elif kind == 3:
            mn = rng.uniform(-30, [w, h]).astype(np.float32)
            ops.append(("rectangle", dict(mn=mn, mx=mn + rng.uniform(1, 120, 2).astype(np.float32), color=col, transform=tr)))
        elif kind == 4:
            ops.append(("bitmap", dict(tex=texs[i % 3], pos=rng.uniform(-30, [w, h]).astype(np.float32), transform=tr, color=col)))
        elif kind == 5:
            a = rng.integers(-20, [w + 20, h + 20]).astype(np.int32)
            b = rng.integers(-20, [w + 20, h + 20]).astype(np.int32)
            ops.append(("line", dict(a=a, b=b, color=col)))
        elif kind == 6:
            s = bytes(rng.integers(32, 127, int(rng.integers(1, 16))).astype(np.uint8))
            ops.append(("text", dict(font=font, pos=rng.uniform(-15, [w, h + 8]).astype(np.float32), text=s, color=col)))
        elif kind == 7 and i % 3 == 0:
            mode = int(rng.integers(0, 3))
            view = scenes.view_transforms(4096)[int(rng.integers(0, 4096))]
            ops.append(("mesh", dict(mesh=mesh, tex=texs[1], light_mode=mode, light_vector=(1, -1, 1), light_color=(1, 1, 1, 1),
                                     pos=(0.1, 0.0, 0.0), transform=view)))
        elif kind == 8 and rng.random() < 0.15:
            ops.append(("clear", dict(rgb=tuple(rng.random(3)))))
        if rng.random() < 0.1:
            ops.append(("flush", None))
    return ops


@pytest.mark.parametrize("seed,size", [(1, (257, 131)), (2, (640, 360)), (3, (96, 1000)), (4, (1023, 65))])
def test_fuzz_mixed_primitive_ids_equal_reference(built, seed, size):
    _check_against_reference(size[0], size[1], _fuzz_ops(seed, size))


def _sphere_views(n):
    mesh, tex = scenes.uv_sphere(), scenes.random_texture(64, 64, 1, True)
    return mesh, tex, scenes.view_transforms(4096)[200:200 + n], np.zeros((n, 3), np.float32)


def test_mesh_views_ids_are_face_indices(built):
    """64 views of the textured Gouraud sphere in one mesh_views call: each view is its own frame, so
    id - 1 is the face index; equal to the port view by view, and replays (overlapped or not) reproduce them."""
    w, h, n = 320, 240, 64
    mesh, tex, ts, pos = _sphere_views(n)
    expect = {}
    for f in range(0, n, 7):
        o = _port(w, h)
        o.clear((0.5, 0.0, 1.0))
        o.mesh(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), ts[f])
        expect[f] = o.ids().copy()
    for stage in STAGES:
        r = _renderer(w, h, n, stage=stage)
        for f in range(n):
            r.begin_frame(f)
            r.clear((0.5, 0.0, 1.0))
        r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), pos, ts, 0)
        ids = r.read_ids(0, n)
        for f, e in expect.items():
            assert np.array_equal(ids[f], e), (stage, f)
        assert 0 < ids.max() <= np.asarray(mesh["faces"]).size // 9
        for overlap in (True, False):
            r.set_replay_overlap(overlap)
            for _ in range(3):
                r.replay()
            assert np.array_equal(r.read_ids(0, n), ids)


def test_counter_continues_across_flushes_and_resets_at_begin_frame(built):
    """A frame drawn over two flushes numbers its triangles on from the first flush; begin_frame restarts
    the count; begin_frame with uploaded depth and colour zeroes the frame's ids."""
    w, h = 200, 120
    rng = np.random.default_rng(5)
    p = np.concatenate([rng.integers(0, [w, h], (60, 3, 2)), rng.uniform(0, 255, (60, 3, 1))], 2).astype(np.float32).reshape(60, 9)
    cols = np.ones((60, 4), np.float32)
    cols[:, :3] = rng.random((60, 3))
    o = _port(w, h)
    o.triangles(p[:25], cols[:25], scenes.DEFAULT_TRIANGLE_TRANSFORM)
    o.triangles(p[25:], cols[25:], scenes.DEFAULT_TRIANGLE_TRANSFORM)
    for stage in STAGES:
        r = _renderer(w, h, stage=stage)
        r.begin_frame(0)
        r.triangles(p[:25], cols[:25], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        r.flush()
        r.triangles(p[25:], cols[25:], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        assert np.array_equal(r.read_ids(0, 1)[0], o.ids())
        assert r.read_ids(0, 1).max() > 25
        # a new frame: numbering restarts at 1
        r.begin_frame(0)
        r.triangles(p[25:], cols[25:], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        o2 = _port(w, h)
        o2.triangles(p[25:], cols[25:], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        assert np.array_equal(r.read_ids(0, 1)[0], o2.ids())
        # uploaded depth and colour: ids reset to 0, then only the new triangles appear
        col0, z0 = r.end_frame(0)
        r.begin_frame(0, color=col0, z=z0)
        assert not r.read_ids(0, 1).any()
        r.triangle(p[0], cols[0], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        o2.reset_ids()
        o2.triangle(p[0], cols[0], scenes.DEFAULT_TRIANGLE_TRANSFORM)
        assert np.array_equal(r.read_ids(0, 1)[0], o2.ids())


def test_band_split_ids_equal_full_frame(built):
    w, h = 1024, 768
    scene = scenes.fill_scene(w, h, 30000, seed=5) + scenes.cfg1_scene(w, h)[1:]
    full = _renderer(w, h)
    full.begin_frame(0)
    scenes.replay(scene, full)
    ids_full = full.read_ids(0, 1)[0]
    bounds = [0, 192, 416, 768]
    for y0, y1 in zip(bounds[:-1], bounds[1:]):
        r = _renderer(w, h)
        r.set_band(y0, y1)
        r.begin_frame(0)
        scenes.replay(scene, r)
        ids = r.read_ids(0, 1)[0]
        assert np.array_equal(ids[y0:y1], ids_full[y0:y1])
        assert not ids[:y0].any() and not ids[y1:].any()


def test_foreign_output_planes_keep_ids_in_own_planes(built):
    """set_output_planes (one GPU): colour and depth go to the other context's planes, ids to this one's."""
    w, h = 320, 200
    scene = scenes.cfg1_scene(w, h) + scenes.mesh_scene(w, h, textured=True, tex_size=32)[1:]
    ref = _renderer(w, h)
    ref.begin_frame(0)
    scenes.replay(scene, ref)
    ref_frame, ref_ids = ref.end_frame(0), ref.read_ids(0, 1)
    for stage in STAGES:
        dst = _renderer(w, h, ids=False)
        dst.flush()  # its first frame's pending depth reset, now: a later flush of dst would reset what src wrote
        src = _renderer(w, h, stage=stage)
        c, z = dst.frame_device_ptrs(0)
        src.set_output_planes(c, z)
        src.begin_frame(0)
        scenes.replay(scene, src)
        src.flush()
        src.sync()
        assert np.array_equal(src.read_ids(0, 1), ref_ids)
        _same_frame(dst.end_frame(0), ref_frame)


def test_foreign_output_planes_two_gpus(built):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from dtrenderer_b200 import api
    w, h = 320, 200
    scene = scenes.cfg1_scene(w, h) + scenes.mesh_scene(w, h, textured=True, tex_size=32)[1:]
    ref = _renderer(w, h)
    ref.begin_frame(0)
    scenes.replay(scene, ref)
    ref_ids = ref.read_ids(0, 1)[0]
    dst = api.Renderer(w, h, 1, 0)
    src = api.Renderer(w, h, 1, 1)
    src.set_id_output(True)
    src.enable_peer_access(0)
    c, z = dst.frame_device_ptrs(0)
    src.set_output_planes(c, z)
    src.begin_frame(0)
    scenes.replay(scene, src)
    assert np.array_equal(src.read_ids(0, 1)[0], ref_ids)


def test_ids_off_allocates_nothing_and_readers_refuse(built):
    """Ids off: the readers return DTR_B200_ERR_ARG; enabling takes the planes' memory and disabling returns it;
    enabling adds no kernel launch to a flush or replay."""
    import torch
    w, h, n = 1920, 1080, 8
    planes = 4 * w * h * n
    r = _renderer(w, h, n, ids=False)
    out = np.empty((1, h, w), np.uint32)
    p = C.c_void_p()
    assert r.lib.dtr_b200_read_ids(r.ctx, 0, 1, out.ctypes.data_as(C.c_void_p)) == ERR_ARG
    assert r.lib.dtr_b200_frame_id_ptr(r.ctx, 0, C.byref(p)) == ERR_ARG
    mesh, tex, ts, pos = _sphere_views(n)

    def launches(ids):
        r.set_id_output(ids)
        r.reset_stats()
        for f in range(n):
            r.begin_frame(f)
            r.clear((0.5, 0.0, 1.0))
        r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), pos, ts, 0)
        r.flush()
        r.replay()
        r.sync()
        return r.stats()["kernelLaunches"]

    assert launches(True) == launches(False)
    free_off = torch.cuda.mem_get_info(0)[0]
    r.set_id_output(True)
    free_on = torch.cuda.mem_get_info(0)[0]
    assert r.lib.dtr_b200_read_ids(r.ctx, n, 1, out.ctypes.data_as(C.c_void_p)) == ERR_ARG
    assert r.lib.dtr_b200_read_ids(r.ctx, 0, 0, out.ctypes.data_as(C.c_void_p)) == ERR_ARG
    assert r.lib.dtr_b200_frame_id_ptr(r.ctx, n, C.byref(p)) == ERR_ARG
    assert r.frame_id_ptr(1) - r.frame_id_ptr(0) == 4 * w * h
    r.set_id_output(False)
    free_off2 = torch.cuda.mem_get_info(0)[0]
    assert r.lib.dtr_b200_frame_id_ptr(r.ctx, 0, C.byref(p)) == ERR_ARG
    slack = 16 << 20  # (the device is shared: other processes may allocate meanwhile)
    assert free_off - free_on >= planes - slack, (free_off, free_on)
    assert free_off2 - free_on >= planes - slack, (free_off2, free_on)
