"""Render to texture on the device (-m gpu): dtr_b200_create_texture / dtr_b200_frames_to_textures.

A texture made from a frame on the device must be, bit for bit, the host conversion (tests/frame_texture_reference.py)
of the same frame, and drawing with it must equal drawing with that conversion uploaded as a texture: the CPU oracle
draws with the numpy texture.  The oracle reads past a texture at uv == 1 like the reference; it is handed the texture
as a view of a larger array whose next rows are opaque white, what the device's spare texels hold after a conversion.
"""
import ctypes as C
import functools

import numpy as np
import pytest

from dtrenderer_b200 import scenes
from frame_texture_reference import frame_texture, texels_of_words
from golden_scenes import SCENES
from test_gpu_colour_range import CLEARS, _cleared_word

pytestmark = pytest.mark.gpu

STAGES = (0, 1, 2)  # api.OPAQUE_SINGLE_KERNEL, OPAQUE_TWO_KERNELS, OPAQUE_ONE_KERNEL
ERR_ARG = -1
FRAME = "frame texture"  # stands for the texture made from a frame in the draw calls below
T7 = scenes.transform7


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


def _same(col, z, o, what=""):
    assert np.array_equal(col, o.color()), f"{what}: colour differs at {(col != o.color()).sum()} px"
    assert np.array_equal(_bits(z), _bits(o.zbuffer())), f"{what}: depth differs at {(_bits(z) != _bits(o.zbuffer())).sum()} px"


def _padded(tex, fill):
    """tex as a view of a larger array whose two following rows are `fill` (the device's spare texels)."""
    h, w = tex.shape[:2]
    buf = np.full((h + 2, w, 4), fill, np.uint8)
    buf[:h] = tex
    return buf[:h]


def _host_texture(color, k=1):
    """The host conversion of a frame as the oracle is given it: opaque, spare texels opaque white."""
    return _padded(frame_texture(color, k), 255)


def _read_tex(r, tid):
    return r.read_texture(tid, (*r.out_shape, 4))


def _issue(target, ops, tex=None, tid=None):
    """Replay ops on the oracle (FRAME -> the numpy texture tex) or on a Renderer (FRAME -> the device texture tid)."""
    for name, kw in ops:
        kw = dict(kw)
        if kw.get("tex") is not FRAME:
            getattr(target, name)(**kw)
        elif tid is None:
            kw["tex"] = tex
            getattr(target, name)(**kw)
        elif name == "bitmap":
            target.bitmap_id(tid, kw["pos"], kw["transform"], kw["color"])
        elif name == "textured_triangle":
            target.textured_triangle_id(kw["p"], kw["uv"], tid, kw["color"], kw["transform"])
        else:
            assert name == "mesh"
            target.mesh_id(target.upload_mesh(kw["mesh"], tid), kw["light_mode"], kw["light_vector"], kw["light_color"],
                           kw["pos"], kw["transform"])


def _oracle(w, h, ids=False):
    from id_reference import IdOracle
    from oracle import dtro
    return IdOracle(w, h) if ids else dtro.Oracle(w, h, "port")


# ---- 1. texels ----------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _golden_oracle(name):
    from oracle import dtro
    w, h, make = SCENES[name]
    o = dtro.Oracle(w, h, "port")
    scenes.replay(make(), o)
    return o.color().copy()


@pytest.mark.parametrize("name", sorted(SCENES))
def test_golden_scene_textures_are_the_host_conversion(built, name):
    """Every k in 1..4 that divides the scene's size, every opaque stage: the texels read back right after the
    conversion (no sync in between) equal the conversion of the oracle's frame."""
    w, h, make = SCENES[name]
    col_o = _golden_oracle(name)
    ks = [k for k in (1, 2, 3, 4) if w % k == 0 and h % k == 0]
    for stage in STAGES:
        r = _renderer(w, h, stage=stage)
        r.begin_frame(0)
        scenes.replay(make(), r)
        for k in ks:
            r.set_readback_resolve(k)
            (tid,) = r.frames_to_textures(0, 1)
            got = _read_tex(r, tid)
            ref = frame_texture(col_o, k)
            assert np.array_equal(got, ref), f"stage {stage} k={k}: {(got != ref).any(-1).sum()} texels differ"
        r.close()


# (width, height, k): 16-byte rows at k = 1, 2 and 4; rows of 2 mod 4 samples at k = 2; odd widths at k = 1 and 3
PATH_SIZES = [(336, 200, 1), (333, 217, 1), (644, 362, 2), (322, 218, 2), (330, 219, 3), (648, 364, 4)]


@pytest.mark.parametrize("w,h,k", PATH_SIZES, ids=[f"{w}x{h}-k{k}" for w, h, k in PATH_SIZES])
def test_every_kernel_path_converts_uploaded_planes(built, w, h, k):
    """Random colour words (X bytes set) uploaded into frames 1..3 of four, converted in one call starting at
    frame 1 into textures given in a shuffled order; the spare texels become opaque white."""
    rng = np.random.default_rng([w, h, k])
    words = rng.integers(0, 1 << 32, (3, h, w), dtype=np.uint64).astype(np.uint32)
    words[0, :k, :] = 0xFF000000  # only the X byte set
    r = _renderer(w, h, 4, k=k)
    for f in range(3):
        r.begin_frame(f + 1, color=words[f])
    oh, ow = r.out_shape
    tids = [r.create_texture(ow, oh) for _ in range(4)]
    order = [tids[2], tids[0], tids[3]]
    assert r.frames_to_textures(1, 3, order) == order
    for f in range(3):
        assert np.array_equal(_read_tex(r, order[f]), frame_texture(words[f], k)), f
    assert not _read_tex(r, tids[1]).any()  # not a target: still the created texture's zeros


# ---- 2. composition against the oracle ---------------------------------------------------------------------
def _scene_a(w, h, seed=3):
    return scenes.cfg1_scene(w, h, seed) + scenes.mesh_scene(w, h, textured=True, tex_size=32, seed=seed)[1:]


def _scene_b(w, h):
    """Bitmaps (rotated, scaled, colour-modulated, one translucent), textured triangles with uv exactly 0 and 1,
    and the sphere bound to the frame texture, lit with an alpha-1 and an alpha < 1 light colour."""
    sphere = scenes.uv_sphere()
    tri = scenes.DEFAULT_TRIANGLE_TRANSFORM
    return [
        ("clear", dict(rgb=(0.1, 0.2, 0.3))),
        ("bitmap", dict(tex=FRAME, pos=(w * .05, h * .1), transform=T7(0.3, (0.5, 0.5, 0.5), (0.6, 0.45, 1.0)), color=(1, 1, 1, 1))),
        ("bitmap", dict(tex=FRAME, pos=(w * .4, h * .3), transform=T7(-0.7, (0.5, 0.5, 0.5), (0.8, 1.3, 1.0)),
                        color=(0.9, 0.5, 0.25, 0.6))),
        ("textured_triangle", dict(p=np.array([w * .1, h * .5, 5, w * .6, h * .5, 5, w * .6, h * .95, 5], np.float32),
                                   uv=(0, 0, 1, 0, 1, 1), tex=FRAME, color=(1, 1, 1, 1), transform=tri)),
        ("textured_triangle", dict(p=np.array([w * .5, h * .05, 8, w * .95, h * .4, 8, w * .55, h * .6, 8], np.float32),
                                   uv=(0, 0, 0, 1, 1, 1), tex=FRAME, color=(0.8, 1.0, 0.6, 0.7), transform=tri)),
        ("mesh", dict(mesh=sphere, tex=FRAME, light_mode=scenes.SHADE_GOURAUD, light_vector=(1, -1, 1), light_color=(1, 1, 1, 1),
                      pos=(0.2, 0.0, 0.0), transform=T7(30.0, (0, 1, 0), (0.5, 0.5, 0.5)))),
        ("mesh", dict(mesh=sphere, tex=FRAME, light_mode=scenes.SHADE_FLAT, light_vector=(-1, -1, 1),
                      light_color=(1.0, 0.8, 0.6, 0.5), pos=(-0.3, 0.1, 0.0), transform=T7(-40.0, (0, 1, 0), (0.4, 0.4, 0.4)))),
    ]


def _opaque_pass(w, h):
    """Only opaque textured triangles on a cleared frame (uv corners, (1, 1) included) and the sphere under an
    alpha-1 light: with a frame texture this pass takes the deferred stage."""
    rng = np.random.default_rng(9)
    ops = [("clear", dict(rgb=(0.7, 0.1, 0.2)))]
    for _ in range(12):
        p = np.concatenate([rng.integers(0, [w, h], (3, 2)), rng.uniform(0, 9, (3, 1))], 1).astype(np.float32).reshape(-1)
        uv = rng.choice([0.0, 1.0], 6).astype(np.float32)
        ops.append(("textured_triangle", dict(p=p, uv=uv, tex=FRAME, color=(1, 1, 1, 1), transform=scenes.DEFAULT_TRIANGLE_TRANSFORM)))
    ops.append(("mesh", dict(mesh=scenes.uv_sphere(), tex=FRAME, light_mode=scenes.SHADE_GOURAUD, light_vector=(1, -1, 1),
                             light_color=(1, 1, 1, 1), pos=(0, 0, 0), transform=T7(10.0, (0, 1, 0), (0.7, 0.7, 0.7)))))
    return ops


COMPOSE = [(1, False), (1, True), (2, False), (2, True)]


@pytest.mark.parametrize("k,ids", COMPOSE, ids=[f"k{k}-{'ids' if i else 'noids'}" for k, i in COMPOSE])
def test_drawing_with_a_frame_texture_equals_drawing_with_its_host_conversion(built, k, ids):
    w, h = 320, 240
    oa = _oracle(w, h)
    _issue(oa, _scene_a(w, h))
    tex = _host_texture(oa.color(), k)
    ob = _oracle(w, h, ids)
    ob.reset_counters()  # the oracle's counters are process-global
    _issue(ob, _scene_b(w, h), tex)
    counts_b = ob.counters()
    oc = _oracle(w, h, ids)
    _issue(oc, _opaque_pass(w, h), tex)
    for stage in STAGES:
        r = _renderer(w, h, 3, ids, stage, k)
        r.begin_frame(0)
        _issue(r, _scene_a(w, h))
        (tid,) = r.frames_to_textures(0, 1)
        r.set_readback_resolve(1)  # frames B and C are compared sample for sample
        before = r.counters()
        r.begin_frame(1)
        _issue(r, _scene_b(w, h), tid=tid)
        col, z = r.end_frame(1)
        _same(col, z, ob, f"scene B, stage {stage}")
        after = r.counters()
        assert (after[0] - before[0], after[1] - before[1]) == counts_b, stage
        if ids:
            assert np.array_equal(r.read_ids(1, 1)[0], ob.ids()), f"ids of scene B, stage {stage}"
        r.begin_frame(2)
        _issue(r, _opaque_pass(w, h), tid=tid)
        col, z = r.end_frame(2)
        _same(col, z, oc, f"opaque pass, stage {stage}")
        assert r.last_pass_stage() == stage
        if ids:
            assert np.array_equal(r.read_ids(2, 1)[0], oc.ids()), f"ids of the opaque pass, stage {stage}"
        r.close()


def test_created_texture_draws_as_transparent_black(built):
    """Before any conversion a created texture is upload_texture of zeros: transparent, zero spare texels."""
    w, h = 160, 120
    r = _renderer(w, h)
    tid = r.create_texture(40, 30)
    assert not r.read_texture(tid, (30, 40, 4)).any()
    ops = _scene_b(w, h)
    o = _oracle(w, h)
    _issue(o, ops, _padded(np.zeros((30, 40, 4), np.uint8), 0))
    r.begin_frame(0)
    _issue(r, ops, tid=tid)
    _same(*r.end_frame(0), o, "zero texture")


# ---- 3. a batch of views --------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2])
def test_64_views_become_64_impostors_in_one_call(built, k):
    """64 mesh_views frames, one conversion into 64 new textures, drawn as 64 bitmaps in an 8 x 8 grid into the
    65th frame.  The conversion adds no counted launch and no set pixel."""
    n, ow, oh = 64, 256, 192
    w, h = k * ow, k * oh
    mesh, tex = scenes.uv_sphere(), scenes.random_texture(64, 64, 1, True)
    ts, pos = scenes.view_transforms(n), np.zeros((n, 3), np.float32)
    light = (scenes.SHADE_GOURAUD, (1, -1, 1), (1, 1, 1, 1))
    sprites = []
    for v in range(n):
        o = _oracle(w, h)
        o.clear((0.5, 0.0, 1.0))
        o.mesh(mesh, tex, *light, (0, 0, 0), ts[v])
        sprites.append(_host_texture(o.color(), k))
    cell = T7(0.0, (0.0, 0.0, 0.0), (0.125, 0.125, 1.0))
    place = [((v % 8) * w / 8, (v // 8) * h / 8) for v in range(n)]
    o = _oracle(w, h)
    o.clear((0.2, 0.2, 0.2))
    for v in range(n):
        o.bitmap(sprites[v], place[v], cell, (1, 1, 1, 1))
    r = _renderer(w, h, n + 1, k=k)
    for f in range(n):
        r.begin_frame(f)
        r.clear((0.5, 0.0, 1.0))
    r.mesh_views(mesh, tex, *light, pos, ts, 0)
    r.flush()
    before = r.stats()
    tids = r.frames_to_textures(0, n)
    assert r.stats() == before
    r.set_readback_resolve(1)
    r.begin_frame(n)
    r.clear((0.2, 0.2, 0.2))
    for v in range(n):
        r.bitmap_id(tids[v], place[v], cell, (1, 1, 1, 1))
    _same(*r.end_frame(n), o, f"impostors k={k}")
    for v in (0, 37, 63):
        assert np.array_equal(r.read_texture(tids[v], (oh, ow, 4)), sprites[v]), v


# ---- 4. overwriting textures that earlier passes used ----------------------------------------------------------
def test_overwritten_white_and_translucent_textures(built):
    """An all-white uploaded texture (its fetch is skipped when a draw call is recorded) and a translucent one
    (zero spare texels), both drawn by an earlier pass, are overwritten by frames.  Draw calls recorded afterwards,
    an opaque pass with uv == 1 under the deferred stages included, match the oracle; a replay is refused until
    the next flush."""
    w, h = 192, 128
    white = np.full((h, w, 4), 255, np.uint8)
    translucent = scenes.random_texture(w, h, 5, opaque=False)
    early = _scene_b(w, h)[:4]
    oa = [_oracle(w, h), _oracle(w, h)]
    _issue(oa[0], _scene_a(w, h, 3))
    _issue(oa[1], _scene_a(w, h, 4))
    conv = [_host_texture(o.color()) for o in oa]
    for stage in STAGES:
        r = _renderer(w, h, 4, stage=stage)
        lib, ctx = r.lib, r.ctx
        tw, tt = r.upload_texture(white), r.upload_texture(translucent)
        for f, (tid, t, fill) in enumerate(((tw, white, 255), (tt, translucent, 0))):
            o = _oracle(w, h)
            _issue(o, early, _padded(t, fill))
            r.begin_frame(2 + f)
            _issue(r, early, tid=tid)
            _same(*r.end_frame(2 + f), o, f"before the conversion, stage {stage}")
        for f in range(2):
            r.begin_frame(f)
            _issue(r, _scene_a(w, h, 3 + f))
        r.flush()
        assert lib.dtr_b200_replay(ctx) == 0
        r.frames_to_textures(0, 2, [tw, tt])
        assert lib.dtr_b200_replay(ctx) == ERR_ARG
        assert lib.dtr_b200_replay(ctx) == ERR_ARG
        for f, tid in ((2, tw), (3, tt)):
            t = conv[f - 2]
            for ops in (_scene_b(w, h), _opaque_pass(w, h)):
                o = _oracle(w, h)
                _issue(o, ops, t)
                r.begin_frame(f)
                _issue(r, ops, tid=tid)
                _same(*r.end_frame(f), o, f"after the conversion, stage {stage}")
            assert r.last_pass_stage() == stage
            assert lib.dtr_b200_replay(ctx) == 0
            _same(*r.end_frame(f), o, f"replayed, stage {stage}")
        r.close()


# ---- 5. ordering without host synchronisation ----------------------------------------------------------------
def test_render_convert_draw_convert_again_without_syncs(built):
    """Four iterations with replay overlap on and asynchronous readbacks in flight, no explicit sync:
    frame 0 gets scene A, becomes texture TA; frame 1 is drawn with TA (flush, then two replays) and read back
    asynchronously, and becomes TB while that read is in flight; TB is drawn into frame 0, and in iteration 2
    frame 0's own texture TA is drawn into frame 0 too; frame 0 is read back asynchronously.  Every read equals
    the oracle's frame of its iteration."""
    import torch
    w, h, iters = 256, 160, 4
    r = _renderer(w, h, 2)
    r.set_replay_overlap(True)
    ta, tb = r.create_texture(w, h), r.create_texture(w, h)
    host = torch.empty((iters, 2, h, w), dtype=torch.int32, pin_memory=True)
    spot = T7(0.2, (0.5, 0.5, 0.5), (0.3, 0.3, 1.0))
    expect = []
    for i in range(iters):
        o0, o1 = _oracle(w, h), _oracle(w, h)
        scene_a = _scene_a(w, h, 10 + i)
        _issue(o0, scene_a)
        r.begin_frame(0)
        _issue(r, scene_a)
        tex_a = _host_texture(o0.color())
        r.frames_to_textures(0, 1, [ta])
        _issue(o1, _scene_b(w, h), tex_a)
        r.begin_frame(1)
        _issue(r, _scene_b(w, h), tid=ta)
        r.flush()
        r.replay()
        r.replay()
        r.read_frames_async_ptr(1, 1, host[i, 1].data_ptr())
        tex_b = _host_texture(o1.color())
        r.frames_to_textures(1, 1, [tb])
        r.set_target(0)
        ops = [("bitmap", dict(tex=FRAME, pos=(20.0 + 10 * i, 15.0), transform=spot, color=(1, 1, 1, 1)))]
        _issue(o0, ops, tex_b)
        _issue(r, ops, tid=tb)
        if i == 2:
            ops = [("bitmap", dict(tex=FRAME, pos=(120.0, 60.0), transform=spot, color=(1, 0.5, 1, 0.8)))]
            _issue(o0, ops, tex_a)
            _issue(r, ops, tid=ta)
        r.read_frames_async_ptr(0, 1, host[i, 0].data_ptr())
        expect.append((o0.color().copy(), o1.color().copy()))
    r.wait_reads()
    got = host.numpy().view(np.uint32)
    for i in range(iters):
        for f in range(2):
            assert np.array_equal(got[i, f], expect[i][f]), f"iteration {i}, frame {f}"


# ---- 6. colour range ------------------------------------------------------------------------------------------
def test_clear_words_with_the_x_byte_give_opaque_texels(built):
    words = [_cleared_word(rgb) for rgb in CLEARS]
    assert any(wd >> 24 for wd in words)
    for k in (1, 2):
        w, h = 64 * k, 48 * k
        r = _renderer(w, h, len(CLEARS), k=k)
        for f, rgb in enumerate(CLEARS):
            r.begin_frame(f)
            r.clear(rgb)
        tids = r.frames_to_textures(0, len(CLEARS))
        for f, wd in enumerate(words):
            want = texels_of_words(np.uint32(wd))
            assert (_read_tex(r, tids[f]) == want).all(), (CLEARS[f], hex(wd), k)
            assert want[3] == 255 and want[0] == (wd >> 16) & 0xFF and want[2] == wd & 0xFF


# ---- 7. errors ------------------------------------------------------------------------------------------------
def test_bad_arguments_are_refused_and_enqueue_nothing(built):
    w, h = 128, 96
    r = _renderer(w, h, 2)
    lib, ctx = r.lib, r.ctx
    for f in range(2):
        r.begin_frame(f)
        _issue(r, _scene_a(w, h, 20 + f))
    good = r.frames_to_textures(0, 2)
    small = r.create_texture(w // 2, h // 2)
    other = r.create_texture(w - 1, h)
    n_tex = 1 << 20  # beyond every texture of the context
    for f in range(2):  # new content: a conversion that got through would change the targets
        r.begin_frame(f)
        _issue(r, _scene_a(w, h, 30 + f))
    snap = {t: r.read_texture(t, (h, w, 4)) for t in good}
    snap[small] = r.read_texture(small, (h // 2, w // 2, 4))

    def refused(first, n, tids):
        arr = (C.c_int * max(len(tids), 1))(*tids)
        assert lib.dtr_b200_frames_to_textures(ctx, first, n, arr) == ERR_ARG, (first, n, tids)
        assert lib.dtr_b200_last_error(ctx)

    for first, n in ((0, 0), (-1, 1), (1, 2), (2, 1), (0, 3), (0, -1)):
        refused(first, n, good + good)
    assert lib.dtr_b200_frames_to_textures(ctx, 0, 1, None) == ERR_ARG
    refused(0, 1, [-1])
    refused(0, 1, [n_tex])
    refused(0, 2, [good[0], n_tex])
    refused(0, 1, [other])              # (W-1) x H
    refused(0, 1, [small])              # (W/2) x (H/2) at k = 1
    refused(0, 2, [good[1], good[1]])   # the same texture twice
    refused(0, 2, [good[0], other])     # a bad entry after a good one
    r.set_readback_resolve(2)
    refused(0, 1, [good[0]])            # W x H no longer matches at k = 2
    for t, want in snap.items():
        assert np.array_equal(r.read_texture(t, want.shape), want), t
    assert r.frames_to_textures(0, 1, [small]) == [small]
    r.set_readback_resolve(1)
    # foreign output planes: the frames are in another context's planes
    owner = _renderer(w, h, 2)
    c0, z0 = owner.frame_device_ptrs(0)
    r.set_output_planes(c0, z0)
    refused(0, 1, [good[0]])
    assert np.array_equal(r.read_texture(good[0], (h, w, 4)), snap[good[0]])
    r.set_output_planes(0, 0)
    assert r.frames_to_textures(0, 2, good) == good
    col, _ = r.end_frame(1)
    assert np.array_equal(r.read_texture(good[1], (h, w, 4)), frame_texture(col))
    for bad in ((0, 4), (4, 0), (32768, 4), (4, 32768), (-1, 4)):
        tid = C.c_int(-7)
        assert lib.dtr_b200_create_texture(ctx, *bad, C.byref(tid)) == ERR_ARG and tid.value == -7, bad
