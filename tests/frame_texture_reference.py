"""numpy statement of render to texture (dtr_b200_frames_to_textures) that the device is compared with: the host
conversion of a readback into the texels dtr_b200_upload_texture would be given."""
import numpy as np

from resolve_reference import resolve_colour


def texels_of_words(words):
    """0x00RRGGBB words [..., H, W] -> RGBA8 texels [..., H, W, 4]: R, G, B from the word, A = 255 (X dropped)."""
    w = np.asarray(words, np.uint32)
    out = np.empty(w.shape + (4,), np.uint8)
    out[..., 0] = (w >> np.uint32(16)) & np.uint32(0xFF)
    out[..., 1] = (w >> np.uint32(8)) & np.uint32(0xFF)
    out[..., 2] = w & np.uint32(0xFF)
    out[..., 3] = 0xFF
    return out


def frame_texture(color, k=1):
    """The texture a frame's colour plane [..., H, W] at sample resolution becomes at resolve factor k:
    [..., H/k, W/k, 4] RGBA8, row 0 at the bottom like the frame."""
    return texels_of_words(resolve_colour(color, k))  # k = 1: every word resolves to itself
