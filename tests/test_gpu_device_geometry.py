"""Draw calls from device memory (-m gpu): dtr_b200_triangles_device / dtr_b200_mesh_views_device.

Every case draws the same arrays twice, once from torch CUDA tensors through the device entries and once from host
memory through the existing entries (dtr_b200_triangles, dtr_b200_textured_triangle per triangle, dtr_b200_mesh_views
on a mesh uploaded with the per-view vertices), each in a fresh context, in all three opaque-stage modes.  Frames,
depth bits, triangle ids, the stage that ran and every counter except uploadBytes must be equal.
"""
import ctypes as C

import numpy as np
import pytest

from dtrenderer_b200 import scenes

pytestmark = pytest.mark.gpu

STAGES = (0, 1, 2)  # api.OPAQUE_SINGLE_KERNEL, OPAQUE_TWO_KERNELS, OPAQUE_ONE_KERNEL
ERR_ARG = -1
T_TRI = scenes.DEFAULT_TRIANGLE_TRANSFORM
# bytes of the command block (dtr_records.h / dtr_kernels.h): FrameState, DrawItem, one u32 per setup CTA, GatherSegment
FRAME_STATE, DRAW_ITEM, GATHER_SEGMENT, SETUP_THREADS = 32, 192, 32, 64


def _torch():
    return pytest.importorskip("torch")


def _dev(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a, np.float32).reshape(-1)).to("cuda:0")


def _renderer(w, h, frames=1, stage=2):
    from dtrenderer_b200 import api
    r = api.Renderer(w, h, frames, 0)
    r.set_opaque_stage(stage)
    r.set_id_output(True)
    return r


def _render(w, h, frames, stage, script):
    """Run script(r), flush; returns (stage that ran, colour, depth bits, ids of every frame, stats, renderer)."""
    r = _renderer(w, h, frames, stage)
    script(r)
    r.flush()
    ran = r.last_pass_stage()
    col, z = zip(*[r.end_frame(f) for f in range(frames)])
    ids = r.read_ids(0, frames)
    return ran, np.stack(col), np.stack(z).view(np.uint32), ids, r.stats(), r


def _compare(w, h, frames, stage, host, device, what=""):
    """host(r) and device(r) must draw the same thing; returns the stage that ran and the device path's results."""
    hs, hc, hz, hi, hst, rh = _render(w, h, frames, stage, host)
    ds, dc, dz, di, dst, rd = _render(w, h, frames, stage, device)
    assert ds == hs, f"{what}: stage {ds} against the host path's {hs}"
    assert np.array_equal(dc, hc), f"{what}: colour differs at {(dc != hc).sum()} px"
    assert np.array_equal(dz, hz), f"{what}: depth differs at {(dz != hz).sum()} px"
    assert np.array_equal(di, hi), f"{what}: ids differ at {(di != hi).sum()} px"
    hst.pop("uploadBytes")
    up = dst.pop("uploadBytes")
    assert dst == hst, what
    rh.close()
    return ds, dc, di, up, rd


def _expect_stage(ran, stage, deferred):
    assert ran == (stage if deferred else 0), (ran, stage, deferred)


# ---- triangles ------------------------------------------------------------------------------------------------
def test_fill4k_million_triangles_take_the_deferred_stage():
    """scenes.small_triangles at 1 M triangles on 3840x2160: many 8192-primitive binning segments, all opaque."""
    w, h, n = 3840, 2160, 1 << 20
    p, color = scenes.small_triangles(w, h, n)
    tp, tc = _dev(p), _dev(color)

    def host(r):
        r.clear((0.0, 0.0, 0.0))
        r.triangles(p, color, T_TRI)

    def device(r):
        r.clear((0.0, 0.0, 0.0))
        r.triangles_device(tp, tc, transform=T_TRI)

    for stage in STAGES:
        ran, _, ids, up, rd = _compare(w, h, 1, stage, host, device, f"fill4k stage {stage}")
        _expect_stage(ran, stage, True)
        blocks = (n + SETUP_THREADS - 1) // SETUP_THREADS
        cmd = FRAME_STATE + DRAW_ITEM + 4 * blocks
        assert up == ((cmd + 15) & ~15) + 2 * GATHER_SEGMENT  # the command block alone: no payload
        rd.close()


def _random_tris(w, h, n, seed):
    p, color = scenes.small_triangles(w, h, n, seed=seed, max_edge=40)
    return p, color


@pytest.mark.parametrize("alpha", [0.5, float("nan")], ids=["translucent", "nan"])
def test_one_non_opaque_alpha_takes_the_single_kernel(alpha):
    """Random colours, all alpha 1 but one (0.5, or NaN, which counts as not opaque like the host loop)."""
    w, h, n = 640, 360, 5000
    p, color = _random_tris(w, h, n, 11)
    color[n // 3, 3] = alpha
    tp, tc = _dev(p), _dev(color)
    for stage in STAGES:
        ran, *_rest, rd = _compare(w, h, 1, stage, lambda r: (r.clear((0.1, 0.2, 0.3)), r.triangles(p, color, T_TRI)),
                                   lambda r: (r.clear((0.1, 0.2, 0.3)), r.triangles_device(tp, tc, transform=T_TRI)),
                                   f"alpha {alpha} stage {stage}")
        _expect_stage(ran, stage, False)
        rd.close()


TEXTURES = {
    "opaque": scenes.random_texture(37, 23, seed=5, opaque=True),
    "translucent": scenes.random_texture(37, 23, seed=6, opaque=False),
    "white": np.full((9, 13, 4), 255, np.uint8),
    "none": None,
}


@pytest.mark.parametrize("kind", sorted(TEXTURES))
def test_textured_batches_equal_textured_triangles(kind):
    """uv in [0, 1] with exact 0 and 1 corners; equal to dtr_b200_textured_triangle per triangle."""
    w, h, n = 480, 272, 1500
    p, color = _random_tris(w, h, n, 12)
    rng = np.random.default_rng(13)
    uv = rng.random((n, 6)).astype(np.float32)
    uv[::5] = np.round(uv[::5])  # corners at exactly 0 and 1
    uv[1::7] = 1.0
    tu = _dev(uv)
    tp, tc = _dev(p), _dev(color)
    tex = TEXTURES[kind]

    def tex_id(r):
        return r.upload_texture(tex) if tex is not None else -1

    def host(r):
        r.clear((0.3, 0.2, 0.1))
        tid = tex_id(r)
        for i in range(n):
            r.textured_triangle_id(p[i], uv[i], tid, color[i], T_TRI)

    def device(r):
        r.clear((0.3, 0.2, 0.1))
        r.triangles_device(tp, tc, tu, tex_id(r), T_TRI)

    for stage in STAGES:
        ran, *_rest, rd = _compare(w, h, 1, stage, host, device, f"{kind} stage {stage}")
        _expect_stage(ran, stage, kind != "translucent")
        rd.close()


def test_device_items_interleaved_with_host_draw_calls():
    """Device and host triangles, rectangles, bitmaps and text in one frame, across two frames and two flushes;
    the ids show the submission order."""
    w, h = 400, 300
    a = _random_tris(w, h, 700, 21)
    b = _random_tris(w, h, 900, 22)
    c = _random_tris(w, h, 500, 23)
    d = _random_tris(w, h, 300, 24)
    uv = np.random.default_rng(25).random((900, 6)).astype(np.float32)
    tex = scenes.random_texture(16, 16, seed=2, opaque=True)
    bmp = scenes.random_texture(40, 30, seed=3, opaque=False)
    font = scenes.synthetic_font(4)
    dev = {k: (_dev(v[0]), _dev(v[1])) for k, v in dict(b=b, d=d).items()}
    tuv = _dev(uv)

    def script(r, on_device):
        tid = r.upload_texture(tex)
        r.set_target(0)
        r.clear((0.5, 0.0, 1.0))
        r.triangles(*a, T_TRI)
        if on_device:
            r.triangles_device(*dev["b"], tuv, tid, T_TRI)
        else:
            for i in range(len(uv)):
                r.textured_triangle_id(b[0][i], uv[i], tid, b[1][i], T_TRI)
        r.rectangle((20, 20), (200, 120), (0.0, 1.0, 1.0, 0.6))
        r.bitmap(bmp, (150.0, 100.0), scenes.transform7(0.3, (0.5, 0.5, 0.5), (2.0, 2.0, 1.0)))
        r.set_target(1)
        r.clear((0.0, 0.0, 0.0))
        if on_device:
            r.triangles_device(*dev["d"], transform=T_TRI)
        else:
            r.triangles(*d, T_TRI)
        r.set_target(0)
        r.text(font, (10.0, 150.0), "device geometry", (1.0, 1.0, 0.0, 0.8))
        r.triangles(*c, T_TRI)
        r.flush()
        r.set_target(0)
        if on_device:
            r.triangles_device(*dev["d"], transform=T_TRI)
        else:
            r.triangles(*d, T_TRI)
        r.set_target(1)
        r.triangles(*a, T_TRI)

    for stage in STAGES:
        _, _, ids, _, rd = _compare(w, h, 2, stage, lambda r: script(r, False), lambda r: script(r, True),
                                    f"interleaved stage {stage}")
        # frame 0: a (1..700), b (701..1600), c (1601..2100), then d of the second flush (2101..2400)
        for lo, hi in ((1, 700), (701, 1600), (1601, 2100), (2101, 2400)):
            assert ((ids[0] >= lo) & (ids[0] <= hi)).any(), (lo, hi)
        for lo, hi in ((1, 300), (301, 1000)):
            assert ((ids[1] >= lo) & (ids[1] <= hi)).any(), (lo, hi)
        rd.close()


def test_misaligned_sources():
    """Tensor views starting 4 bytes into their storage (scalar path), and an odd byte address through the C ABI."""
    torch = _torch()
    w, h, n = 320, 240, 3001  # 36 n bytes: not a multiple of 16, several gather chunks
    p, color = _random_tris(w, h, n, 31)
    color[::97, 3] = 1.0
    uv = np.random.default_rng(32).random((n, 6)).astype(np.float32)
    tex = scenes.random_texture(8, 8, seed=9, opaque=True)

    def shifted(a):
        s = torch.zeros(a.size + 1, dtype=torch.float32, device="cuda:0")
        v = s[1:]
        v.copy_(torch.from_numpy(a.reshape(-1)))
        assert v.data_ptr() % 16 == 4 and v.is_contiguous()
        return v

    sp, sc, su = shifted(p), shifted(color), shifted(uv)

    def host(r):
        r.clear((0.0, 0.0, 0.0))
        tid = r.upload_texture(tex)
        for i in range(n):
            r.textured_triangle_id(p[i], uv[i], tid, color[i], T_TRI)

    def device(r):
        r.clear((0.0, 0.0, 0.0))
        r.triangles_device(sp, sc, su, r.upload_texture(tex), T_TRI)

    keep = []

    def odd_bytes(a):
        raw = np.frombuffer(np.ascontiguousarray(a, np.float32).tobytes(), np.uint8)
        s = torch.zeros(raw.size + 3, dtype=torch.uint8, device="cuda:0")
        s[1:1 + raw.size].copy_(torch.from_numpy(raw.copy()))
        keep.append(s)
        return C.c_void_p(s.data_ptr() + 1)

    from dtrenderer_b200 import api
    t = api.make_transform(T_TRI)

    def device_odd(r):
        r.clear((0.0, 0.0, 0.0))
        tid = r.upload_texture(tex)
        args = odd_bytes(p), odd_bytes(color), odd_bytes(uv)
        torch.cuda.synchronize()
        assert r.lib.dtr_b200_triangles_device(r.ctx, n, *args, tid, C.byref(t)) == 0

    for stage in STAGES:
        for device_path, what in ((device, "4-byte offset"), (device_odd, "odd address")):
            _, _, _, _, rd = _compare(w, h, 1, stage, host, device_path, f"{what} stage {stage}")
            rd.close()


def test_replay_renders_the_snapshot_after_the_tensors_changed():
    """A replay after the caller overwrote the tensors gives the first frame again; a later flush reads the new
    values.  The replay itself uploads nothing."""
    w, h, n = 512, 256, 4000
    p, color = _random_tris(w, h, n, 41)
    p2, color2 = _random_tris(w, h, n, 42)
    tp, tc = _dev(p), _dev(color)
    for stage in STAGES:
        r = _renderer(w, h, 1, stage)
        r.clear((0.2, 0.2, 0.2))
        r.triangles_device(tp, tc, transform=T_TRI)
        r.flush()
        first = r.end_frame(0)[0].copy()
        tp.copy_(_dev(p2))
        tc.copy_(_dev(color2))
        r.replay()
        again = r.end_frame(0)[0]
        assert np.array_equal(again, first), f"stage {stage}: the replay re-read the caller's arrays"
        # the new values, drawn by a new flush, equal the host path's drawing of them
        r.begin_frame(0)
        r.clear((0.2, 0.2, 0.2))
        r.triangles_device(tp, tc, transform=T_TRI)
        new = r.end_frame(0)[0]
        o = _renderer(w, h, 1, stage)
        o.clear((0.2, 0.2, 0.2))
        o.triangles(p2, color2, T_TRI)
        assert np.array_equal(new, o.end_frame(0)[0]), stage
        tp.copy_(_dev(p))
        tc.copy_(_dev(color))
        r.close()
        o.close()


def test_writes_on_another_torch_stream_are_ordered_before_the_flush():
    """The wrapper synchronises torch's current stream, so a kernel that fills the tensors on a side stream is seen."""
    torch = _torch()
    w, h, n = 320, 200, 20000
    p, color = _random_tris(w, h, n, 51)
    src_p, src_c = _dev(p), _dev(color)
    for stage in STAGES:
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            tp = torch.empty_like(src_p)
            tc = torch.empty_like(src_c)
            side.wait_stream(torch.cuda.default_stream())
            for _ in range(20):  # enough work that the copy is still running when the call returns
                tp.copy_(src_p * 1.0)
                tc.copy_(src_c * 1.0)
            *_rest, rd = _compare(w, h, 1, stage, lambda r: (r.clear((0, 0, 0)), r.triangles(p, color, T_TRI)),
                                  lambda r: (r.clear((0, 0, 0)), r.triangles_device(tp, tc, transform=T_TRI)),
                                  f"side stream stage {stage}")
        rd.close()


# ---- meshes ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_normals", [True, False], ids=["normals", "mesh-normals"])
def test_mesh_views_with_per_view_vertex_sets(with_normals):
    """The textured sphere with 64 deformed vertex sets, one per view and frame, against uploading each deformed
    mesh on the host and drawing it with dtr_b200_mesh_views into the same frame."""
    w, h, views = 200, 150, 64
    sphere = scenes.uv_sphere()
    tex = scenes.random_texture(64, 64, seed=1, opaque=True)
    rng = np.random.default_rng(61)
    nv = sphere["vertexes"].shape[0]
    verts = np.repeat(sphere["vertexes"][None], views, 0).copy()
    verts[..., :3] *= (0.6 + 0.5 * rng.random((views, 1, 3))).astype(np.float32)
    verts[..., :3] += (0.03 * rng.standard_normal((views, nv, 3))).astype(np.float32)
    verts[..., 3] = 1.0
    normals = np.repeat(sphere["normals"][None], views, 0) + (0.2 * rng.standard_normal((views, *sphere["normals"].shape)))
    normals = (normals / np.linalg.norm(normals, axis=-1, keepdims=True)).astype(np.float32)
    positions = np.zeros((views, 3), np.float32)
    transforms = scenes.view_transforms(views)
    tv, tn = _dev(verts), (_dev(normals) if with_normals else None)
    light = (scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1))

    def host(r):
        for v in range(views):
            r.set_target(v)
            r.clear((0.5, 0.0, 1.0))
        for v in range(views):
            mesh = dict(sphere, vertexes=verts[v], normals=normals[v] if with_normals else sphere["normals"])
            r.mesh_views(mesh, tex, *light, positions[v], [transforms[v]], first_frame=v)

    def device(r):
        for v in range(views):
            r.set_target(v)
            r.clear((0.5, 0.0, 1.0))
        mid = r.upload_mesh(sphere, r.upload_texture(tex))
        r.mesh_views_device(mid, *light, positions, transforms, tv, tn, first_frame=0)

    for stage in STAGES:
        ran, *_rest, rd = _compare(w, h, views, stage, host, device, f"mesh views stage {stage}")
        _expect_stage(ran, stage, True)
        rd.close()


# ---- argument errors ------------------------------------------------------------------------------------------
def _nothing_recorded(r):
    assert r.stats()["triangles"] == 0
    r.flush()
    assert r.stats()["primitives"] == 0


def test_argument_errors_record_nothing():
    torch = _torch()
    from dtrenderer_b200 import api
    r = _renderer(64, 64, 2)
    lib = r.lib
    n = 4
    p, color = _random_tris(64, 64, n, 71)
    tp, tc = _dev(p), _dev(color)
    pinned = torch.from_numpy(p.reshape(-1)).pin_memory()
    light = api.Light(2, (C.c_float * 3)(1, -1, 1), (C.c_float * 4)(1, 1, 1, 1))
    pos = (C.c_float * 6)()
    ts = (api.Transform * 2)(*[api.make_transform(t) for t in scenes.view_transforms(2)])
    sphere = scenes.uv_sphere(8, 4)
    mid = r.upload_mesh(sphere, r.upload_texture(scenes.WHITE_TEXTURE))
    tv = _dev(np.repeat(sphere["vertexes"][None], 2, 0))
    dptr = lambda t: C.c_void_p(t.data_ptr())
    # host pointers: pageable and pinned
    assert lib.dtr_b200_triangles_device(r.ctx, n, p.ctypes.data_as(C.c_void_p), dptr(tc), None, -1, None) == ERR_ARG
    assert lib.dtr_b200_triangles_device(r.ctx, n, dptr(pinned), dptr(tc), None, -1, None) == ERR_ARG
    assert lib.dtr_b200_triangles_device(r.ctx, n, dptr(tp), color.ctypes.data_as(C.c_void_p), None, -1, None) == ERR_ARG
    assert lib.dtr_b200_triangles_device(r.ctx, n, dptr(tp), dptr(tc), p.ctypes.data_as(C.c_void_p), 0, None) == ERR_ARG
    # texId out of range
    assert lib.dtr_b200_triangles_device(r.ctx, n, dptr(tp), dptr(tc), None, 99, None) == ERR_ARG
    # meshes: bad id, frame range, host vertexes / normals
    for m, nv, first in ((-1, 2, 0), (99, 2, 0), (mid, 2, 1), (mid, 2, -1), (mid, 3, 0)):
        assert lib.dtr_b200_mesh_views_device(r.ctx, m, C.byref(light), nv, pos, ts, first, dptr(tv), None) == ERR_ARG
    hv = np.repeat(sphere["vertexes"][None], 2, 0)
    assert lib.dtr_b200_mesh_views_device(r.ctx, mid, C.byref(light), 2, pos, ts, 0, hv.ctypes.data_as(C.c_void_p), None) == ERR_ARG
    hn = np.repeat(sphere["normals"][None], 2, 0)
    assert lib.dtr_b200_mesh_views_device(r.ctx, mid, C.byref(light), 2, pos, ts, 0, dptr(tv), hn.ctypes.data_as(C.c_void_p)) == ERR_ARG
    if torch.cuda.device_count() >= 2:
        other = torch.from_numpy(p.reshape(-1)).to("cuda:1")
        assert lib.dtr_b200_triangles_device(r.ctx, n, dptr(other), dptr(tc), None, -1, None) == ERR_ARG
        ov = tv.to("cuda:1")
        assert lib.dtr_b200_mesh_views_device(r.ctx, mid, C.byref(light), 2, pos, ts, 0, dptr(ov), None) == ERR_ARG
    _nothing_recorded(r)
    # nothing to draw: OK without drawing
    assert lib.dtr_b200_triangles_device(r.ctx, 0, dptr(tp), dptr(tc), None, -1, None) == 0
    assert lib.dtr_b200_triangles_device(r.ctx, n, None, dptr(tc), None, -1, None) == 0
    assert lib.dtr_b200_mesh_views_device(r.ctx, mid, C.byref(light), 2, pos, ts, 0, None, None) == 0
    _nothing_recorded(r)
    r.close()


def test_python_wrapper_rejects_what_it_would_have_to_copy():
    torch = _torch()
    r = _renderer(64, 64, 1)
    p, color = _random_tris(64, 64, 4, 81)
    tp, tc = _dev(p), _dev(color)
    bad = [
        (torch.from_numpy(p.reshape(-1)), tc),                 # CPU tensor
        (tp.double(), tc),                                      # float64
        (tp.view(4, 9).t(), tc),                                # not contiguous
        (tp, tc[:-1]),                                          # wrong element count
        (p, tc),                                                # numpy array
    ]
    for a, b in bad:
        with pytest.raises(ValueError):
            r.triangles_device(a, b)
    with pytest.raises(ValueError):
        r.triangles_device(tp, tc, uv=tc)
    _nothing_recorded(r)
    r.close()
