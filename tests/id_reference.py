"""Reference triangle id planes for the tests, derived from the CPU oracle without changing it.

The oracle port draws one triangle at a time and writes a pixel's depth exactly when a fragment passes the
strict `>` test, so a pass always changes the depth's bits.  IdOracle therefore issues every triangle of a
draw call as a call of its own (a batch as single triangles with the same transform, a mesh as one-face
meshes through the same viewport matrix) and gives the pixels whose depth bits changed the id 1 + that
triangle's position since the last reset_ids().  Colour, depth and counters are the oracle's own: splitting
changes nothing, the oracle runs the same per-triangle code in the same order either way.
"""
import ctypes as C

import numpy as np

from oracle import dtro


class IdOracle:
    def __init__(self, width, height):
        self.o = dtro.Oracle(width, height, "port")
        self._z = self.o.zbuffer().view(np.uint32)  # live view of the oracle's depth plane
        self._ids = np.zeros((height, width), np.uint32)
        self._seen = self._z.copy()
        self._n = 0

    # ---- planes -------------------------------------------------------------------------------
    def ids(self):
        return self._ids

    def reset_ids(self):
        """Zero the id plane and the triangle count (where the device side calls begin_frame)."""
        self._ids[:] = 0
        self._n = 0

    def upload(self, color, z):
        """Start from caller-supplied planes, as begin_frame(color=, z=) does: the ids and the count restart."""
        self.o.color()[:] = color
        self._z[:] = np.asarray(z, np.float32).view(np.uint32)  # bit copy: NaN payloads stay as they are
        self._seen[:] = self._z
        self.reset_ids()

    def _after_triangle(self):
        self._n += 1
        changed = self._z != self._seen
        self._ids[changed] = self._n
        self._seen[changed] = self._z[changed]

    def __getattr__(self, name):  # color, zbuffer, counters, reset_counters and the blits
        return getattr(self.o, name)

    # ---- the draw calls that submit triangles ------------------------------------------------
    def triangle(self, p, color, transform=dtro.DEFAULT_TRIANGLE_TRANSFORM):
        self.o.triangle(p, color, transform)
        self._after_triangle()

    def triangles(self, p, color, transform=dtro.DEFAULT_TRIANGLE_TRANSFORM):
        p = np.asarray(p, np.float32).reshape(-1, 9)
        color = np.asarray(color, np.float32).reshape(-1, 4)
        for k in range(len(p)):  # == dtro_triangles, which loops dtro_triangle
            self.triangle(p[k], color[k], transform)

    def textured_triangle(self, p, uv, tex, color, transform=dtro.DEFAULT_TRIANGLE_TRANSFORM):
        self.o.textured_triangle(p, uv, tex, color, transform)
        self._after_triangle()

    def mesh(self, mesh, tex, light_mode, light_vector, light_color, pos=(0, 0, 0), transform=dtro.DEFAULT_TRANSFORM):
        fa, fp = dtro._fa, dtro._fp
        v, t, n = fa(mesh["vertexes"]), fa(mesh["texUV"]), fa(mesh["normals"])
        f = np.ascontiguousarray(mesh["faces"], dtype=np.int32).reshape(-1, 9)
        tex = np.ascontiguousarray(tex, dtype=np.uint8)
        h, w = tex.shape[:2]
        lv, lc, ps, tr = fa(light_vector, 3), fa(light_color, 4), fa(pos, 3), fa(transform, 7)
        for k in range(len(f)):  # one face per call: dtro_mesh builds the same matrix and loops the faces
            self.o.lib.dtro_mesh(self.o.ctx, fp(v), v.size // 4, fp(t), t.size // 3, fp(n), n.size // 3,
                                 C.cast(f.ctypes.data + f.strides[0] * k, C.POINTER(C.c_int32)), 1,
                                 tex.ctypes.data_as(C.POINTER(C.c_uint8)), w, h, int(light_mode),
                                 fp(lv), fp(lc), fp(ps), fp(tr))
            self._after_triangle()
