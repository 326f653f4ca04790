"""numpy statement of the readback resolve (dtr_b200_set_readback_resolve) that the device is compared with.

Planes are [..., H, W] with row 0 at the bottom; output pixel (X, Y) is made from samples [kX, kX+k) x [kY, kY+k).
"""
import numpy as np


def resolve_byte(sums, k):
    """floor(sqrt(floor(sums / k^2))) for integer sums, exactly: a float root corrected by integer compares."""
    m = np.asarray(sums, np.int64) // (k * k)
    v = np.floor(np.sqrt(m.astype(np.float64))).astype(np.int64)
    v -= (v * v > m)
    v += ((v + 1) * (v + 1) <= m)
    return v


def _blocks(plane, k):
    """[..., H, W] -> [..., H/k, W/k, k*k]: each block's samples row by row from its bottom-left sample."""
    *lead, h, w = plane.shape
    b = plane.reshape(*lead, h // k, k, w // k, k)
    b = np.moveaxis(b, -3, -2)  # [..., H/k, W/k, k(rows), k(columns)]
    return b.reshape(*lead, h // k, w // k, k * k)


def resolve_colour(color, k):
    """Per byte of each 0x00RRGGBB word (the X byte too): the integer root of the mean of the squared bytes."""
    c = np.ascontiguousarray(color, np.uint32)
    out = np.zeros(c.shape[:-2] + (c.shape[-2] // k, c.shape[-1] // k), np.uint32)
    for lane in range(4):
        b = _blocks(((c >> np.uint32(8 * lane)) & np.uint32(0xFF)).astype(np.int64), k)
        out |= resolve_byte((b * b).sum(-1), k).astype(np.uint32) << np.uint32(8 * lane)
    return out


def pick_index(z, k):
    """Index into each block (row-major from its bottom-left) of the sample the depth rule chooses: the first,
    replaced only by a later sample whose depth compares > (IEEE) with the current choice."""
    b = _blocks(np.asarray(z, np.float32), k)
    best = b[..., 0].copy()
    at = np.zeros(best.shape, np.int64)
    for t in range(1, k * k):
        upd = b[..., t] > best
        best = np.where(upd, b[..., t], best)
        at = np.where(upd, t, at)
    return at


def pick(plane, at, k):
    """The chosen sample of each block of `plane` (any 4-byte dtype; bits are kept)."""
    return np.take_along_axis(_blocks(np.asarray(plane), k), at[..., None], -1)[..., 0]


def resolve_depth(z, k):
    """Depth bits of the chosen sample (float32, NaN payloads as they are)."""
    z = np.asarray(z, np.float32)
    return pick(z.view(np.uint32), pick_index(z, k), k).view(np.float32)


def resolve_ids(z, ids, k):
    return pick(np.asarray(ids, np.uint32), pick_index(z, k), k)


def pack_bgr24(color, pitch):
    """[n, H, W] u32 colour -> [n, H, pitch] bytes of 24-bit DIB rows (B, G, R per pixel, zero padding)."""
    c = np.ascontiguousarray(color, np.uint32)
    n, h, w = c.shape
    out = np.zeros((n, h, pitch), np.uint8)
    out[:, :, :3 * w] = c.view(np.uint8).reshape(n, h, w, 4)[..., :3].reshape(n, h, 3 * w)
    return out
