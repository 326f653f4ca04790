"""Supersampled readback on the device (-m gpu): dtr_b200_set_readback_resolve / dtr_b200_resolve_frames.

Every readback of a context with resolve factor k must equal, bit for bit, the numpy resolve
(tests/resolve_reference.py) of the frame at sample resolution: of the CPU oracle's frame, and of the device's
own k = 1 readback.
"""
import ctypes as C
import functools

import numpy as np
import pytest

from dtrenderer_b200 import scenes
from golden_scenes import SCENES
from resolve_reference import pack_bgr24, resolve_colour, resolve_depth, resolve_ids
from test_gpu_colour_range import CLEARS, _cleared_word

pytestmark = pytest.mark.gpu

STAGES = (0, 1, 2)  # api.OPAQUE_SINGLE_KERNEL, OPAQUE_TWO_KERNELS, OPAQUE_ONE_KERNEL
ERR_ARG = -1


def _renderer(w, h, frames=1, ids=False, stage=2, k=1):
    from dtrenderer_b200 import api
    r = api.Renderer(w, h, frames, 0)
    r.set_opaque_stage(stage)
    if ids:
        r.set_id_output(True)
    if k != 1:
        r.set_readback_resolve(k)
    return r


def _bits(z):
    return np.asarray(z, np.float32).view(np.uint32)


def _same(col, z, ref_col, ref_z, what=""):
    assert np.array_equal(col, ref_col), f"{what}: colour differs at {(col != ref_col).sum()} px"
    assert np.array_equal(_bits(z), _bits(ref_z)), f"{what}: depth differs at {(_bits(z) != _bits(ref_z)).sum()} px"


def _pinned(shape, dtype):
    import torch
    return torch.empty(shape, dtype=dtype, pin_memory=True)


@functools.lru_cache(maxsize=None)
def _golden_oracle(name):
    from oracle import dtro
    w, h, make = SCENES[name]
    o = dtro.Oracle(w, h, "port")
    scenes.replay(make(), o)
    return o.color().copy(), o.zbuffer().copy()


GOLDEN = [(name, k) for name in sorted(SCENES) for k in (2, 4) if SCENES[name][0] % k == 0 and SCENES[name][1] % k == 0]
GOLDEN.append(("cfg2_gouraud_1080p", 3))


@pytest.mark.parametrize("name,k", GOLDEN, ids=[f"{n}-k{k}" for n, k in GOLDEN])
def test_golden_scene_resolves_like_the_oracle(built, name, k):
    w, h, make = SCENES[name]
    col_o, z_o = _golden_oracle(name)
    ref_c, ref_z = resolve_colour(col_o, k), resolve_depth(z_o, k)
    for stage in STAGES:
        r = _renderer(w, h, stage=stage)
        r.begin_frame(0)
        scenes.replay(make(), r)
        col1, z1 = r.end_frame(0)
        r.set_readback_resolve(k)
        col, z = r.end_frame(0)
        assert col.shape == (h // k, w // k)
        _same(col, z, ref_c, ref_z, f"stage {stage} vs oracle")
        _same(col, z, resolve_colour(col1, k), resolve_depth(z1, k), f"stage {stage} vs own k=1")


def _mixed_scene(w, h):
    return scenes.cfg1_scene(w, h) + scenes.mesh_scene(w, h, textured=True, tex_size=32)[1:]


def _mesh_only(w, h):
    return scenes.mesh_scene(w, h, textured=True, tex_size=32)


# (width, height, k): 16-byte sample rows at k = 2 and 4; rows of 2 mod 4 samples and an odd output width at
# k = 2; output widths that end in a partial group of four in the 24-bit pack at k = 2, 3 and 4
PATH_SIZES = [(640, 360, 2), (322, 218, 2), (330, 219, 3), (648, 364, 4)]


@pytest.mark.parametrize("w,h,k", PATH_SIZES, ids=[f"{w}x{h}-k{k}" for w, h, k in PATH_SIZES])
def test_every_readback_path_agrees(built, w, h, k):
    """Two different frames read through end_frame, read_frames, read_frames_async, read_frames_bgr24_async,
    read_ids and resolve_frames_tensors: all equal the resolve of the reference frames (ids: tests/id_reference.py)."""
    import torch
    from id_reference import IdOracle
    ref = []
    for make in (_mixed_scene, _mesh_only):
        o = IdOracle(w, h)
        scenes.replay(make(w, h), o)
        c, z, i = o.color(), o.zbuffer(), o.ids()
        ref.append((resolve_colour(c, k), resolve_depth(z, k), resolve_ids(z, i, k)))
    ref_c = np.stack([x[0] for x in ref])
    ref_z = np.stack([x[1] for x in ref])
    ref_i = np.stack([x[2] for x in ref])
    oh, ow = h // k, w // k
    for stage in STAGES:
        r = _renderer(w, h, 2, ids=True, stage=stage, k=k)
        for f, make in enumerate((_mixed_scene, _mesh_only)):
            r.begin_frame(f)
            scenes.replay(make(w, h), r)
        for f in range(2):
            _same(*r.end_frame(f), ref_c[f], ref_z[f], f"end_frame {f}")
        col, z = np.empty((2, oh, ow), np.uint32), np.empty((2, oh, ow), np.float32)
        r.read_frames_ptr(0, 2, col.ctypes.data, z.ctypes.data)
        _same(col, z, ref_c, ref_z, "read_frames")
        hc, hz = _pinned((2, oh, ow), torch.int32), _pinned((2, oh, ow), torch.float32)
        r.read_frames_async_ptr(0, 2, hc.data_ptr(), hz.data_ptr())
        pitch = r.bgr24_pitch()
        assert pitch == (3 * ow + 3) & ~3
        hb = _pinned((2, oh, pitch), torch.uint8)
        hb.fill_(0x5A)  # the padding must be written too
        r.read_frames_bgr24_async_ptr(0, 2, hb.data_ptr())
        r.wait_reads()
        _same(hc.numpy().view(np.uint32), hz.numpy(), ref_c, ref_z, "read_frames_async")
        bgr = hb.numpy()
        assert np.array_equal(bgr[:, :, :3 * ow], pack_bgr24(ref_c, pitch)[:, :, :3 * ow]), "bgr24 pixels"
        assert (bgr[:, :, 3 * ow:] == 0).all(), "bgr24 row padding"
        assert np.array_equal(r.read_ids(0, 2), ref_i), "read_ids"
        tc, tz, ti = r.resolve_frames_tensors(0, 2, ids=True)
        assert tc.dtype == torch.int32 and tz.dtype == torch.float32 and ti.dtype == torch.int32
        assert tuple(tc.shape) == (2, oh, ow)
        _same(tc.cpu().numpy().view(np.uint32), tz.cpu().numpy(), ref_c, ref_z, "resolve_frames_tensors")
        assert np.array_equal(ti.cpu().numpy().view(np.uint32), ref_i), "resolve_frames_tensors ids"
        tc1, tz1 = r.resolve_frames_tensors(1, 1)
        _same(tc1.cpu().numpy().view(np.uint32), tz1.cpu().numpy(), ref_c[1:], ref_z[1:], "resolve_frames_tensors frame 1")


def _sphere_views(n):
    mesh, tex = scenes.uv_sphere(), scenes.random_texture(64, 64, 1, True)
    return mesh, tex, scenes.view_transforms(4096)[300:300 + n], np.zeros((n, 3), np.float32)


@pytest.mark.parametrize("k", [2, 3])
def test_mesh_views_resolve_like_their_k1_readback(built, k):
    """64 views of the textured Gouraud sphere rendered at k x a 160x120 output: resolved frames and ids equal the
    numpy resolve of the same context's k = 1 readback."""
    ow, oh, n = 160, 120, 64
    w, h = k * ow, k * oh
    mesh, tex, ts, pos = _sphere_views(n)
    r = _renderer(w, h, n, ids=True)
    for f in range(n):
        r.begin_frame(f)
        r.clear((0.5, 0.0, 1.0))
    r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), pos, ts, 0)
    col1, z1 = np.empty((n, h, w), np.uint32), np.empty((n, h, w), np.float32)
    r.read_frames_ptr(0, n, col1.ctypes.data, z1.ctypes.data)
    ids1 = r.read_ids(0, n)
    r.set_readback_resolve(k)
    col, z = np.empty((n, oh, ow), np.uint32), np.empty((n, oh, ow), np.float32)
    r.read_frames_ptr(0, n, col.ctypes.data, z.ctypes.data)
    _same(col, z, resolve_colour(col1, k), resolve_depth(z1, k), "mesh_views")
    assert np.array_equal(r.read_ids(0, n), resolve_ids(z1, ids1, k))


# ---- the rule at its edges -----------------------------------------------------------------------------------
def test_uniform_blocks_and_clear_words_resolve_to_themselves(built):
    from oracle import dtro
    k, ow, oh = 2, 96, 40
    rng = np.random.default_rng(11)
    words = rng.integers(0, 1 << 32, (oh, ow), dtype=np.uint64).astype(np.uint32)
    words[0, :4] = [0, 0xFFFFFFFF, 0x00FFFFFF, 0xFF000000]
    z = rng.standard_normal((oh, ow)).astype(np.float32)
    for kk in (2, 3, 4):
        r = _renderer(kk * ow, kk * oh, k=kk)
        r.begin_frame(0, color=np.repeat(np.repeat(words, kk, 0), kk, 1), z=np.repeat(np.repeat(z, kk, 0), kk, 1))
        _same(*r.end_frame(0), words, z, f"uploaded uniform blocks, k={kk}")
    w, h = k * ow, k * oh
    for rgb in CLEARS:
        word = _cleared_word(rgb)
        o = dtro.Oracle(w, h, "port")
        o.clear(rgb)
        r = _renderer(w, h, k=k)
        r.begin_frame(0)
        r.clear(rgb)
        col, z = r.end_frame(0)
        assert (col == np.uint32(word)).all(), (rgb, hex(word))
        _same(col, z, resolve_colour(o.color(), k), resolve_depth(o.zbuffer(), k), f"clear {rgb}")


def test_blocks_mixing_0_and_255(built):
    rng = np.random.default_rng(12)
    for k in (2, 3, 4):
        w, h = 60 * k, 36 * k
        col = rng.choice(np.array([0, 0xFFFFFFFF, 0x00FF00FF, 0xFF00FF00, 0x000000FF], np.uint32), (h, w))
        r = _renderer(w, h, k=k)
        r.begin_frame(0, color=col, z=np.zeros((h, w), np.float32))
        out, _ = r.end_frame(0)
        assert np.array_equal(out, resolve_colour(col, k)), k
        assert len(np.unique(out)) > 20


def _special_depths():
    f = np.float32
    nans = np.array([0x7FC00000, 0x7FC00001, 0xFFC00002, 0x7F800003], np.uint32).view(np.float32)
    return np.concatenate([np.array([0.0, -0.0, 1.0, 1.0, 2.0, np.inf, -np.inf, -3.4028234663852886e38, 3.4028234663852886e38,
                                     f(1e-45), f(-1e-45), 100.0], np.float32), nans])


def test_depth_ties_infinities_and_nans_keep_the_scan_order(built):
    """Uploaded depth planes of ties (+0 / -0 have different bits), +-inf and NaNs with distinct payloads: the chosen
    sample's bits tell which one the device picked.  Triangles drawn over them give the ids to check."""
    from id_reference import IdOracle
    rng = np.random.default_rng(13)
    vals = _special_depths()
    for k in (2, 3, 4):
        w, h = 64 * k, 40 * k
        z = rng.choice(vals, (h, w))
        col = rng.integers(0, 1 << 24, (h, w), dtype=np.uint32)
        n = 200
        c = rng.integers(0, [w, h], (n, 1, 2))
        p = np.concatenate([c + rng.integers(-20, 21, (n, 3, 2)), rng.uniform(-1, 255, (n, 3, 1))], 2).astype(np.float32)
        cols = rng.random((n, 4)).astype(np.float32)
        cols[:, 3] = 1.0
        o = IdOracle(w, h)
        o.upload(col, z)
        o.triangles(p.reshape(n, 9), cols, scenes.DEFAULT_TRIANGLE_TRANSFORM)
        for stage in STAGES:
            r = _renderer(w, h, ids=True, stage=stage, k=k)
            r.begin_frame(0, color=col, z=z)
            out, oz = r.end_frame(0)
            _same(out, oz, resolve_colour(col, k), resolve_depth(z, k), f"uploaded planes k={k}")
            r.triangles(p.reshape(n, 9), cols, scenes.DEFAULT_TRIANGLE_TRANSFORM)
            out, oz = r.end_frame(0)
            _same(out, oz, resolve_colour(o.color(), k), resolve_depth(o.zbuffer(), k), f"drawn over k={k} stage={stage}")
            ids = r.read_ids(0, 1)[0]
            assert np.array_equal(ids, resolve_ids(o.zbuffer(), o.ids(), k)), (k, stage)
            assert ids.any()


# ---- k = 1 and the rest of the context are untouched ----------------------------------------------------------
def test_factor_1_is_the_plain_readback_and_no_stat_changes(built):
    w, h = 320, 200
    scene = _mixed_scene(w, h)

    def run(toggle):
        r = _renderer(w, h, ids=True)
        r.begin_frame(0)
        scenes.replay(scene, r)
        r.flush()
        r.sync()
        before = r.stats()
        if toggle:
            r.set_readback_resolve(2)
            assert r.stats() == before
            r.end_frame(0)
            r.read_ids(0, 1)
            r.resolve_frames_tensors(0, 1, ids=True)
            assert r.stats() == before  # resolve kernels are not counted
            r.set_readback_resolve(1)
        col, z = r.end_frame(0)
        return col, z, r.read_ids(0, 1), r.stats()

    col0, z0, ids0, st0 = run(False)
    col1, z1, ids1, st1 = run(True)
    _same(col1, z1, col0, z0, "k back to 1")
    assert np.array_equal(ids1, ids0)
    assert st1 == st0
    assert col1.shape == (h, w)


def test_rendering_continues_after_a_resolved_read(built):
    """A frame drawn over two flushes with a resolved read between them still equals the oracle."""
    from oracle import dtro
    w, h, k = 640, 360, 2
    scene = _mixed_scene(w, h)
    cut = len(scene) // 2
    o1, o = dtro.Oracle(w, h, "port"), dtro.Oracle(w, h, "port")
    scenes.replay(scene[:cut], o1)
    scenes.replay(scene, o)
    for stage in STAGES:
        r = _renderer(w, h, stage=stage, k=k)
        r.begin_frame(0)
        scenes.replay(scene[:cut], r)
        _same(*r.end_frame(0), resolve_colour(o1.color(), k), resolve_depth(o1.zbuffer(), k), "first flush")
        scenes.replay(scene[cut:], r)
        _same(*r.end_frame(0), resolve_colour(o.color(), k), resolve_depth(o.zbuffer(), k), "second flush")
        r.set_readback_resolve(1)
        _same(*r.end_frame(0), o.color(), o.zbuffer(), "samples")


def test_alternating_async_reads_overlapped_with_the_next_flush(built):
    """The bench's end-to-end pattern: batches of views rendered into two halves of the frames, each half read
    back asynchronously (resolved, then resolved bgr24) into its own pinned buffer while the next batch renders."""
    import torch
    from oracle import dtro
    k, ow, oh, sub, batches = 2, 160, 120, 8, 6
    w, h = k * ow, k * oh
    mesh, tex, ts, pos = _sphere_views(sub * batches)
    expect = []
    for v in range(sub * batches):
        o = dtro.Oracle(w, h, "port")
        o.clear((0.5, 0.0, 1.0))
        o.mesh(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), (0, 0, 0), ts[v])
        expect.append(resolve_colour(o.color(), k))
    r = _renderer(w, h, 2 * sub, k=k)
    pitch = r.bgr24_pitch()
    host = _pinned((2, sub, oh, ow), torch.int32)
    host24 = _pinned((2, sub, oh, pitch), torch.uint8)
    for mode in ("u32", "bgr24"):
        for b in range(batches):
            half = b & 1
            for f in range(half * sub, half * sub + sub):
                r.begin_frame(f)
                r.clear((0.5, 0.0, 1.0))
            r.mesh_views(mesh, tex, scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1), pos[:sub], ts[b * sub:(b + 1) * sub], half * sub)
            if mode == "u32":
                r.read_frames_async_ptr(half * sub, sub, host[half].data_ptr())
            else:
                r.read_frames_bgr24_async_ptr(half * sub, sub, host24[half].data_ptr())
        r.wait_reads()
        for b in (batches - 2, batches - 1):
            want = np.stack(expect[b * sub:(b + 1) * sub])
            if mode == "u32":
                assert np.array_equal(host[b & 1].numpy().view(np.uint32), want), b
            else:
                got = host24[b & 1].numpy()[:, :, :3 * ow]
                assert np.array_equal(got, pack_bgr24(want, pitch)[:, :, :3 * ow]), b


def test_band_split_resolves_the_assembled_frame(built):
    """Two contexts on one GPU: the second renders its band into the first one's planes (set_output_planes);
    the resolved read on the owning context equals the resolve of a whole-frame render."""
    w, h = 640, 480
    scene = scenes.fill_scene(w, h, 8000, seed=5) + scenes.cfg1_scene(w, h)[1:]
    full = _renderer(w, h)
    full.begin_frame(0)
    scenes.replay(scene, full)
    col1, z1 = full.end_frame(0)
    for k in (2, 4):
        r0, r1 = _renderer(w, h, k=k), _renderer(w, h)
        c0, z0 = r0.frame_device_ptrs(0)
        r1.set_output_planes(c0, z0)
        r0.set_band(*r0.band_rows(2, 0))
        r1.set_band(*r1.band_rows(2, 1))
        for r in (r0, r1):
            r.begin_frame(0)
            scenes.replay(scene, r)
            r.flush()
        r1.sync()
        _same(*r0.end_frame(0), resolve_colour(col1, k), resolve_depth(z1, k), f"band split k={k}")


# ---- errors ---------------------------------------------------------------------------------------------------
def test_bad_arguments_are_refused_and_the_old_factor_stays(built):
    w, h = 320, 200
    scene = _mixed_scene(w, h)
    r = _renderer(w, h, 2, k=2)
    for f in range(2):
        r.begin_frame(f)
        scenes.replay(scene, r)
    ref = r.end_frame(0)
    lib, ctx = r.lib, r.ctx
    for bad in (0, 5, -1, 3):  # 3 divides neither 320 nor 200
        assert lib.dtr_b200_set_readback_resolve(ctx, bad) == ERR_ARG, bad
    col, z = np.empty((h // 2, w // 2), np.uint32), np.empty((h // 2, w // 2), np.float32)
    assert lib.dtr_b200_end_frame(ctx, 0, col.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p)) == 0
    _same(col, z, *ref, "factor kept")
    odd = _renderer(333, 217)
    for bad in (2, 3, 4):
        assert odd.lib.dtr_b200_set_readback_resolve(odd.ctx, bad) == ERR_ARG, bad
    assert odd.end_frame(0)[0].shape == (217, 333)
    import torch
    buf = torch.empty((2, h // 2, w // 2), dtype=torch.int32, device="cuda")
    p = C.c_void_p(buf.data_ptr())
    assert lib.dtr_b200_resolve_frames(ctx, 0, 1, p, None, p) == ERR_ARG  # ids without id output
    for first, n in ((0, 0), (-1, 1), (1, 2), (2, 1), (0, 3)):
        assert lib.dtr_b200_resolve_frames(ctx, first, n, p, None, None) == ERR_ARG, (first, n)
    assert lib.dtr_b200_end_frame(ctx, 0, col.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p)) == 0
    _same(col, z, *ref, "factor kept after resolve_frames errors")
