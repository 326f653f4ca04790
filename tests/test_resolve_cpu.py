"""Readback resolve without a GPU: the numpy rule the GPU tests compare with, and the C ABI's resolve entry
points without a context."""
import ctypes as C
import re

import numpy as np

from resolve_reference import pick_index, resolve_byte, resolve_colour, resolve_depth


def test_resolve_byte_is_the_largest_root_of_the_block_sum():
    """floor(sqrt(floor(S / k^2))) == the largest v with v^2 k^2 <= S, for every S a k x k block of bytes can give."""
    for k in range(1, 5):
        s = np.arange(0, k * k * 255 * 255 + 1, dtype=np.int64)
        v = resolve_byte(s, k)
        kk = k * k
        assert (v * v * kk <= s).all() and ((v + 1) * (v + 1) * kk > s).all(), k
        assert v.min() == 0 and v.max() == 255


def test_uniform_blocks_resolve_to_themselves():
    rng = np.random.default_rng(7)
    words = rng.integers(0, 1 << 32, (3, 6, 5), dtype=np.uint64).astype(np.uint32)
    words[0, 0, :4] = [0, 0xFFFFFFFF, 0x00FFFFFF, 0xFF000000]  # clears with the X byte set included
    z = rng.standard_normal((3, 6, 5)).astype(np.float32)
    for k in range(1, 5):
        up = np.repeat(np.repeat(words, k, 1), k, 2)
        assert np.array_equal(resolve_colour(up, k), words)
        uz = np.repeat(np.repeat(z, k, 1), k, 2)
        assert not pick_index(uz, k).any()  # ties keep the first sample
        assert np.array_equal(resolve_depth(uz, k).view(np.uint32), z.view(np.uint32))


def test_depth_rule_scans_rows_from_the_bottom_left():
    nan = np.float32("nan")
    z = np.array([[1, 2], [2, 0]], np.float32)  # row 0 (bottom) first: the tie in row 1 keeps (1, 0)
    assert pick_index(z, 2)[0, 0] == 1
    z = np.array([[nan, 5], [7, 9]], np.float32)  # nothing compares > with NaN: the first sample stays
    assert pick_index(z, 2)[0, 0] == 0
    z = np.array([[-np.inf, nan], [np.inf, np.inf]], np.float32)
    assert pick_index(z, 2)[0, 0] == 2


def test_resolve_entry_points_fail_loudly_without_a_context(built):
    from dtrenderer_b200 import api
    lib = api.load_library()
    assert lib.dtr_b200_set_readback_resolve(None, 2) == -1
    assert lib.dtr_b200_set_readback_resolve(None, 1) == -1
    assert lib.dtr_b200_resolve_frames(None, 0, 1, None, None, None) == -1
    assert lib.dtr_b200_resolve_frames(None, 0, 1, C.c_void_p(16), None, None) == -1


def test_resolve_symbols_are_bound_as_declared(built):
    import os
    from dtrenderer_b200 import api
    header = open(os.path.join(os.path.dirname(api._HERE), "include", "dtr_b200.h")).read()
    bound = {s[0]: s for s in api.SYMBOLS}
    for name, nargs in (("dtr_b200_set_readback_resolve", 2), ("dtr_b200_resolve_frames", 6)):
        decl = re.search(r"int\s+" + name + r"\s*\(([^)]*)\)", header)
        assert decl and len(decl.group(1).split(",")) == nargs
        assert name in bound and bound[name][1] is C.c_int and len(bound[name][2]) == nargs
