"""Draw calls from device memory without a GPU: the C ABI's device entry points without a context."""
import ctypes as C


def test_entry_points_fail_loudly_without_a_context(built):
    from dtrenderer_b200 import api
    lib = api.load_library()
    buf = (C.c_float * 36)()
    assert lib.dtr_b200_triangles_device(None, 1, buf, buf, None, -1, None) == -1
    assert lib.dtr_b200_triangles_device(None, 0, None, None, None, -1, None) == -1
    light = api.Light(0, (C.c_float * 3)(), (C.c_float * 4)(1, 1, 1, 1))
    t = (api.Transform * 1)(api.make_transform(None) or api.Transform())
    assert lib.dtr_b200_mesh_views_device(None, 0, C.byref(light), 1, buf, t, 0, buf, None) == -1
    assert lib.dtr_b200_mesh_views_device(None, 0, None, 0, None, None, 0, None, None) == -1
