"""Render to texture without a GPU: the host conversion the GPU tests compare with, against its definition, and
the C ABI's render-to-texture entry points without a context."""
import ctypes as C

import numpy as np

from frame_texture_reference import frame_texture, texels_of_words
from resolve_reference import resolve_byte

EXTREME = np.array([0x00000000, 0xFFFFFFFF, 0x00FFFFFF, 0xFF000000, 0x00FF0000, 0x0000FF00, 0x000000FF,
                    0xFF123456, 0x80808080, 0x7F7F7F7F, 0x01FE01FE], np.uint32)


def _by_definition(color, k):
    """Texel (x, y) from the block [kx, kx+k) x [ky, ky+k), one pixel at a time in plain Python."""
    h, w = color.shape
    out = np.zeros((h // k, w // k, 4), np.uint8)
    for y in range(h // k):
        for x in range(w // k):
            block = [int(v) for v in color[k * y:k * y + k, k * x:k * x + k].reshape(-1)]
            word = 0
            for lane in range(4):
                s = sum(((v >> (8 * lane)) & 0xFF) ** 2 for v in block)
                word |= int(resolve_byte(s, k)) << (8 * lane)
            out[y, x] = ((word >> 16) & 0xFF, (word >> 8) & 0xFF, word & 0xFF, 0xFF)
    return out


def test_texel_layout_of_single_words():
    t = texels_of_words(EXTREME)
    for word, texel in zip(EXTREME.tolist(), t):
        r, g, b = (word >> 16) & 0xFF, (word >> 8) & 0xFF, word & 0xFF
        assert texel.tolist() == [r, g, b, 255], hex(word)
        assert int(texel.view(np.uint32)[0]) == r | g << 8 | b << 16 | 0xFF000000  # DTRBitmap's u32, little endian


def test_reference_conversion_against_its_definition():
    """k = 1..4 on hand-built words: random ones, the X byte set, and blocks of extreme bytes."""
    rng = np.random.default_rng(21)
    for k in range(1, 5):
        h, w = 3 * k, 5 * k
        color = rng.integers(0, 1 << 32, (h, w), dtype=np.uint64).astype(np.uint32)
        color[:k, :] = rng.choice(EXTREME, (k, w))
        color[k:2 * k, :k] = 0xFF000000  # a block whose only set byte is X
        t = frame_texture(color, k)
        assert t.shape == (h // k, w // k, 4)
        assert np.array_equal(t, _by_definition(color, k)), k
        assert (t[..., 3] == 255).all()
        assert (t[1, 0] == [0, 0, 0, 255]).all()


def test_uniform_blocks_keep_their_rgb_and_drop_x():
    for k in range(1, 5):
        up = np.repeat(np.repeat(EXTREME[None, :], k, 0), k, 1)
        assert np.array_equal(frame_texture(up, k)[0], texels_of_words(EXTREME))


def test_batches_convert_frame_by_frame():
    rng = np.random.default_rng(22)
    color = rng.integers(0, 1 << 32, (3, 8, 12), dtype=np.uint64).astype(np.uint32)
    for k in (1, 2, 4):
        t = frame_texture(color, k)
        for f in range(3):
            assert np.array_equal(t[f], frame_texture(color[f], k))


def test_entry_points_fail_loudly_without_a_context(built):
    from dtrenderer_b200 import api
    lib = api.load_library()
    tid = C.c_int(-7)
    assert lib.dtr_b200_create_texture(None, 4, 4, C.byref(tid)) == -1
    assert tid.value == -7
    ids = (C.c_int * 1)(0)
    assert lib.dtr_b200_frames_to_textures(None, 0, 1, ids) == -1
    assert lib.dtr_b200_frames_to_textures(None, 0, 1, None) == -1
