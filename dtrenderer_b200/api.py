"""ctypes binding of include/dtr_b200.h plus a thin host-side mirror of the renderer's draw calls.

``Renderer`` exposes the reference's draw-call set (DTRendererRender.h:91-98) with the same
argument meaning -- clear / triangle / textured_triangle / mesh / rectangle / bitmap / line -- on
top of the C ABI, so a scene written against the reference's API replays unchanged.  There is no
CPU fallback: if libdtr_b200.so is missing or no CUDA device is present, construction raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# DTR_B200_LIB: developer override used to compare experimental builds of the same C ABI
LIB_PATH = os.environ.get("DTR_B200_LIB") or os.path.join(_HERE, "libdtr_b200.so")

SHADE_FULLBRIGHT, SHADE_FLAT, SHADE_GOURAUD = 0, 1, 2
OPAQUE_SINGLE_KERNEL, OPAQUE_TWO_KERNELS, OPAQUE_ONE_KERNEL = 0, 1, 2  # dtr_b200_set_opaque_stage

_f = C.POINTER(C.c_float)
_u8 = C.POINTER(C.c_uint8)
_i32 = C.POINTER(C.c_int32)
_u32 = C.POINTER(C.c_uint32)


class Transform(C.Structure):
    """dtr_b200_transform == DTRRenderTransform (DTRendererRender.h:28-33)."""
    _fields_ = [("rotation", C.c_float), ("anchor", C.c_float * 3), ("scale", C.c_float * 3)]


class Light(C.Structure):
    """dtr_b200_light == DTRRenderLight (DTRendererRender.h:72-77)."""
    _fields_ = [("mode", C.c_int32), ("vector", C.c_float * 3), ("color", C.c_float * 4)]


class MeshDesc(C.Structure):
    _fields_ = [("vertexes", _f), ("numVertexes", C.c_uint32), ("texUV", _f), ("numTexUV", C.c_uint32),
                ("normals", _f), ("numNormals", C.c_uint32), ("faces", _i32), ("numFaces", C.c_uint32)]


class MeshFace(C.Structure):
    """dtr_b200_mesh_face == DTRMeshFace (DTRendererAsset.h:16-26): three host pointers + counts."""
    _fields_ = [("vertexIndex", C.c_void_p), ("numVertexIndex", C.c_uint32), ("texIndex", C.c_void_p),
                ("numTexIndex", C.c_uint32), ("normalIndex", C.c_void_p), ("numNormalIndex", C.c_uint32)]


class MeshFacesDesc(C.Structure):
    _fields_ = [("vertexes", _f), ("numVertexes", C.c_uint32), ("texUV", _f), ("numTexUV", C.c_uint32),
                ("normals", _f), ("numNormals", C.c_uint32), ("faces", C.POINTER(MeshFace)), ("numFaces", C.c_uint32),
                ("arena", C.c_void_p), ("arenaBytes", C.c_size_t)]


class Stats(C.Structure):
    _fields_ = [("setPixels", C.c_uint64), ("triangles", C.c_uint64), ("primitives", C.c_uint64),
                ("listEntries", C.c_uint64), ("kernelLaunches", C.c_uint64), ("uploadBytes", C.c_uint64)]


# every symbol include/dtr_b200.h declares: (name, restype, argtypes)
_T = C.POINTER(Transform)
_L = C.POINTER(Light)
SYMBOLS = [
    ("dtr_b200_create", C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("dtr_b200_destroy", None, [C.c_void_p]),
    ("dtr_b200_last_error", C.c_char_p, [C.c_void_p]),
    ("dtr_b200_version", C.c_char_p, []),
    ("dtr_b200_set_stream", C.c_int, [C.c_void_p, C.c_void_p]),
    ("dtr_b200_set_band", C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ("dtr_b200_upload_texture", C.c_int, [C.c_void_p, _u8, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    ("dtr_b200_upload_bitmap_straight", C.c_int, [C.c_void_p, _u8, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    ("dtr_b200_read_texture", C.c_int, [C.c_void_p, C.c_int, _u8]),
    ("dtr_b200_upload_mesh", C.c_int, [C.c_void_p, C.POINTER(MeshDesc), C.c_int, C.POINTER(C.c_int)]),
    ("dtr_b200_upload_mesh_faces", C.c_int, [C.c_void_p, C.POINTER(MeshFacesDesc), C.c_int, C.POINTER(C.c_int)]),
    ("dtr_b200_update_texture", C.c_int, [C.c_void_p, C.c_int, _u8]),
    ("dtr_b200_tile_height", C.c_int, []),
    ("dtr_b200_band_rows", C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("dtr_b200_band_comm_unique_id", C.c_int, [_u8]),
    ("dtr_b200_band_comm_init", C.c_int, [C.c_void_p, _u8, C.c_int, C.c_int]),
    ("dtr_b200_band_comm_attach", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    ("dtr_b200_gather_bands", C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ("dtr_b200_band_barrier", C.c_int, [C.c_void_p]),
    ("dtr_b200_set_target", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_begin_frame", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    ("dtr_b200_flush", C.c_int, [C.c_void_p]),
    ("dtr_b200_replay", C.c_int, [C.c_void_p]),
    ("dtr_b200_set_replay_overlap", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_sync", C.c_int, [C.c_void_p]),
    ("dtr_b200_end_frame", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    ("dtr_b200_read_frames", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("dtr_b200_read_frames_async", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("dtr_b200_wait_reads", C.c_int, [C.c_void_p]),
    ("dtr_b200_read_frames_bgr24_async", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    ("dtr_b200_set_readback_resolve", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_resolve_frames", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("dtr_b200_create_texture", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    ("dtr_b200_frames_to_textures", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    ("dtr_b200_export_frames", C.c_int, [C.c_void_p, _u8, _u8]),
    ("dtr_b200_open_peer_frames", C.c_int, [C.c_void_p, _u8, _u8]),
    ("dtr_b200_set_output_planes", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    ("dtr_b200_enable_peer_access", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_frame_device_ptrs", C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    ("dtr_b200_set_id_output", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_read_ids", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    ("dtr_b200_frame_id_ptr", C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    ("dtr_b200_get_stats", C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    ("dtr_b200_reset_stats", C.c_int, [C.c_void_p]),
    ("dtr_b200_last_pass_deferred", C.c_int, [C.c_void_p]),
    ("dtr_b200_set_opaque_stage", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_set_profiling", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_get_stage_ms", C.c_int, [C.c_void_p, C.POINTER(C.c_float * 4), C.POINTER(C.c_int)]),
    ("dtr_b200_get_raster_split_ms", C.c_int, [C.c_void_p, C.POINTER(C.c_float * 2), C.POINTER(C.c_int)]),
    ("dtr_b200_reset_stage_ms", C.c_int, [C.c_void_p]),
    ("dtr_b200_selftest", C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("dtr_b200_clear", C.c_int, [C.c_void_p, _f]),
    ("dtr_b200_triangle", C.c_int, [C.c_void_p, _f, _f, _f, _f, _T]),
    ("dtr_b200_triangles", C.c_int, [C.c_void_p, C.c_int, _f, _f, _T]),
    ("dtr_b200_textured_triangle", C.c_int, [C.c_void_p, _f, _f, _f, _f, _f, _f, C.c_int, _f, _T]),
    ("dtr_b200_mesh", C.c_int, [C.c_void_p, C.c_int, _L, _f, _T]),
    ("dtr_b200_mesh_views", C.c_int, [C.c_void_p, C.c_int, _L, C.c_int, _f, _T, C.c_int]),
    ("dtr_b200_triangles_device", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, _T]),
    ("dtr_b200_mesh_views_device", C.c_int, [C.c_void_p, C.c_int, _L, C.c_int, _f, _T, C.c_int, C.c_void_p, C.c_void_p]),
    ("dtr_b200_rectangle", C.c_int, [C.c_void_p, _f, _f, _f, _T]),
    ("dtr_b200_bitmap", C.c_int, [C.c_void_p, C.c_int, _f, _T, _f]),
    ("dtr_b200_line", C.c_int, [C.c_void_p, _i32, _i32, _f]),
    ("dtr_b200_set_debug_markers", C.c_int, [C.c_void_p, C.c_int]),
    ("dtr_b200_upload_font", C.c_int, [C.c_void_p, _u8, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    ("dtr_b200_text", C.c_int, [C.c_void_p, C.c_int, _f, C.c_char_p, _f, C.c_int]),
]

_lib = None


def load_library():
    """dlopen libdtr_b200.so and bind every symbol; raises if the CUDA module was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(this back end has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _fa(x, n=None):
    a = np.ascontiguousarray(x, dtype=np.float32).reshape(-1)
    if n is not None and a.size != n:
        raise ValueError(f"expected {n} floats, got {a.size}")
    return a


def _fp(a):
    return a.ctypes.data_as(_f)


def make_transform(t):
    """Accept a Transform, a 7-float array (rotation, anchor.xyz, scale.xyz) or None."""
    if t is None or isinstance(t, Transform):
        return t
    a = _fa(t, 7)
    return Transform(float(a[0]), (C.c_float * 3)(*a[1:4]), (C.c_float * 3)(*a[4:7]))


class DtrError(RuntimeError):
    pass


class Renderer:
    """One rendering context on one GPU: ``num_frames`` colour+depth targets in HBM."""

    def __init__(self, width, height, num_frames=1, device=0):
        self.lib = load_library()
        self.width, self.height, self.num_frames, self.device = width, height, num_frames, device
        h = C.c_void_p()
        rc = self.lib.dtr_b200_create(device, width, height, num_frames, C.byref(h))
        if rc != 0:
            raise DtrError(f"dtr_b200_create failed ({rc}): {self.lib.dtr_b200_last_error(None).decode()}")
        self.ctx = h
        self.resolve = 1  # readback resolve factor (set_readback_resolve)
        self._tex = {}    # id(array) -> (texId, array)
        self._mesh = {}   # (id(mesh dict), texId) -> meshId
        self._font = {}   # id(atlas) -> (fontId, font)
        self._mesh_counts = {}  # meshId -> (numVertexes, numNormals), for the device draw calls' size checks
        self._stream = None     # what set_stream was given (None: the context's own stream)
        self._device_inputs = []  # tensors recorded by the device draw calls, kept alive until a flush has read them

    # ---- plumbing ----------------------------------------------------------------------------
    def _ck(self, rc):
        if rc != 0:
            raise DtrError(f"dtr_b200 error {rc}: {self.lib.dtr_b200_last_error(self.ctx).decode()}")

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.dtr_b200_destroy(self.ctx)
            self.ctx = None
            self._device_inputs = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream):
        self._ck(self.lib.dtr_b200_set_stream(self.ctx, C.c_void_p(cuda_stream)))
        self._stream = cuda_stream or None
        self._device_inputs = []  # (set_stream flushes)

    def set_band(self, y0, y1):
        self._ck(self.lib.dtr_b200_set_band(self.ctx, y0, y1))

    def upload_texture(self, tex):
        key = id(tex)
        if key in self._tex:
            return self._tex[key][0]
        a = np.ascontiguousarray(tex, dtype=np.uint8)
        h, w = a.shape[:2]
        tid = C.c_int(-1)
        self._ck(self.lib.dtr_b200_upload_texture(self.ctx, a.ctypes.data_as(_u8), w, h, 4, C.byref(tid)))
        self._tex[key] = (tid.value, tex)
        return tid.value

    def upload_bitmap_straight(self, rgba):
        """Straight-alpha RGBA8 -> premultiplied texture (DTRAsset_LoadBitmap's pass, on the device)."""
        a = np.ascontiguousarray(rgba, dtype=np.uint8)
        h, w = a.shape[:2]
        tid = C.c_int(-1)
        self._ck(self.lib.dtr_b200_upload_bitmap_straight(self.ctx, a.ctypes.data_as(_u8), w, h, C.byref(tid)))
        return tid.value

    def read_texture(self, tex_id, shape):
        out = np.empty(shape, np.uint8)
        self._ck(self.lib.dtr_b200_read_texture(self.ctx, tex_id, out.ctypes.data_as(_u8)))
        return out

    def create_texture(self, w, h):
        """A device-only texture of w x h texels, all zero (dtr_b200_create_texture); returns its id."""
        tid = C.c_int(-1)
        self._ck(self.lib.dtr_b200_create_texture(self.ctx, int(w), int(h), C.byref(tid)))
        return tid.value

    def frames_to_textures(self, first=0, n=1, tex_ids=None):
        """Flush, then turn frames [first, first + n) into textures on the device, stream-ordered
        (dtr_b200_frames_to_textures): frame first + i into tex_ids[i], each of out_shape.  With tex_ids None, n
        new textures of out_shape are created.  Returns the texture ids."""
        if tex_ids is None:
            oh, ow = self.out_shape
            tex_ids = [self.create_texture(ow, oh) for _ in range(n)]
        tex_ids = [int(t) for t in tex_ids]
        if len(tex_ids) != n:
            raise ValueError(f"expected {n} texture ids, got {len(tex_ids)}")
        self._ck(self.lib.dtr_b200_frames_to_textures(self.ctx, first, n, (C.c_int * n)(*tex_ids)))
        self._device_inputs = []
        return tex_ids

    def upload_mesh(self, mesh, tex_id):
        key = (id(mesh), tex_id)
        if key in self._mesh:
            return self._mesh[key][0]
        v, t, n = _fa(mesh["vertexes"]), _fa(mesh["texUV"]), _fa(mesh["normals"])
        f = np.ascontiguousarray(mesh["faces"], dtype=np.int32).reshape(-1)
        d = MeshDesc(_fp(v), v.size // 4, _fp(t), t.size // 3, _fp(n), n.size // 3,
                     f.ctypes.data_as(_i32), f.size // 9)
        mid = C.c_int(-1)
        self._ck(self.lib.dtr_b200_upload_mesh(self.ctx, C.byref(d), tex_id, C.byref(mid)))
        self._mesh[key] = (mid.value, mesh)
        self._mesh_counts[mid.value] = (v.size // 4, n.size // 3)
        return mid.value

    def upload_mesh_faces(self, mesh, faces, arena, tex_id):
        """DTRMesh as the reference's loader leaves it: ``faces`` is a ctypes array of MeshFace whose
        pointers lead into the numpy byte block ``arena``; the index table is flattened on the device."""
        v, t, n = _fa(mesh["vertexes"]), _fa(mesh["texUV"]), _fa(mesh["normals"])
        d = MeshFacesDesc(_fp(v), v.size // 4, _fp(t), t.size // 3, _fp(n), n.size // 3, faces, len(faces),
                          C.c_void_p(arena.ctypes.data), arena.nbytes)
        mid = C.c_int(-1)
        self._ck(self.lib.dtr_b200_upload_mesh_faces(self.ctx, C.byref(d), tex_id, C.byref(mid)))
        self._mesh_counts[mid.value] = (v.size // 4, n.size // 3)
        return mid.value

    def update_texture(self, tex_id, tex):
        """Re-upload a texture the host changed in place (same dimensions)."""
        a = np.ascontiguousarray(tex, dtype=np.uint8)
        self._ck(self.lib.dtr_b200_update_texture(self.ctx, tex_id, a.ctypes.data_as(_u8)))

    def mesh_id(self, mesh_id, light_mode, light_vector, light_color, pos=(0, 0, 0), transform=None):
        """DTRRender_Mesh with a mesh that is already on the device."""
        light = self._light(light_mode, light_vector, light_color)
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_mesh(self.ctx, mesh_id, C.byref(light), _fp(_fa(pos, 3)), C.byref(t) if t else None))

    # ---- sort-first bands (C ABI: partition, NCCL exchange, barrier) ---------------------------
    def tile_height(self):
        return int(self.lib.dtr_b200_tile_height())

    def band_rows(self, nranks, rank):
        y0, y1 = C.c_int(0), C.c_int(0)
        self._ck(self.lib.dtr_b200_band_rows(self.height, nranks, rank, C.byref(y0), C.byref(y1)))
        return y0.value, y1.value

    def band_comm_init(self, unique_id, nranks, rank):
        """ncclCommInitRank inside the library (unique_id: the 128 bytes rank 0 got from band_comm_unique_id)."""
        buf = (C.c_uint8 * 128)(*unique_id)
        self._ck(self.lib.dtr_b200_band_comm_init(self.ctx, buf, nranks, rank))

    def band_comm_unique_id(self):
        buf = (C.c_uint8 * 128)()
        self._ck(self.lib.dtr_b200_band_comm_unique_id(buf))
        return bytes(buf)

    def band_comm_init_torch(self, dist, group=None):
        """Bootstrap the library's own NCCL communicator over an existing torch.distributed group:
        rank 0's ncclUniqueId is broadcast, every rank calls dtr_b200_band_comm_init."""
        import torch
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        buf = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            buf.copy_(torch.tensor(list(self.band_comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(buf, src=0, group=group)
        self.band_comm_init(bytes(buf.cpu().tolist()), world, rank)

    def gather_bands(self, frame=0, dst=0):
        """dtr_b200_gather_bands: grouped ncclSend/ncclRecv of every rank's band rows into rank dst's planes."""
        self._ck(self.lib.dtr_b200_gather_bands(self.ctx, frame, dst))

    def band_barrier(self):
        self._ck(self.lib.dtr_b200_band_barrier(self.ctx))

    # ---- frame -------------------------------------------------------------------------------
    def set_target(self, frame):
        self._ck(self.lib.dtr_b200_set_target(self.ctx, frame))

    def begin_frame(self, frame=0, color=None, z=None):
        cp = color.ctypes.data_as(C.c_void_p) if color is not None else None
        zp = z.ctypes.data_as(C.c_void_p) if z is not None else None
        self._ck(self.lib.dtr_b200_begin_frame(self.ctx, frame, cp, zp))

    def flush(self):
        self._ck(self.lib.dtr_b200_flush(self.ctx))
        self._device_inputs = []

    def replay(self):
        self._ck(self.lib.dtr_b200_replay(self.ctx))

    def set_replay_overlap(self, enable=True):
        self._ck(self.lib.dtr_b200_set_replay_overlap(self.ctx, 1 if enable else 0))

    def sync(self):
        self._ck(self.lib.dtr_b200_sync(self.ctx))

    @property
    def out_shape(self):
        """(rows, columns) of a frame as the readbacks return it: the sample size over the resolve factor."""
        return self.height // self.resolve, self.width // self.resolve

    def set_readback_resolve(self, k):
        """Every readback returns frames of (W/k) x (H/k), each pixel resolved on the device from a k x k block of
        samples (see dtr_b200_set_readback_resolve); draw calls, uploads and device pointers stay at W x H."""
        self._ck(self.lib.dtr_b200_set_readback_resolve(self.ctx, int(k)))
        self.resolve = int(k)

    def resolve_frames_tensors(self, first=0, n=1, ids=False):
        """Resolved colour (int32, the view multigpu.frame_tensors uses), depth (float32) and, with ids=True, ids
        (int32) of frames [first, first + n) as new torch tensors [n, H/k, W/k] on this context's device, filled in
        stream order on the context's stream (dtr_b200_resolve_frames)."""
        import torch
        dev = torch.device("cuda", self.device)
        shape = (n, *self.out_shape)
        col = torch.empty(shape, dtype=torch.int32, device=dev)
        dep = torch.empty(shape, dtype=torch.float32, device=dev)
        idp = torch.empty(shape, dtype=torch.int32, device=dev) if ids else None
        self._ck(self.lib.dtr_b200_resolve_frames(self.ctx, first, n, C.c_void_p(col.data_ptr()), C.c_void_p(dep.data_ptr()),
                                                  C.c_void_p(idp.data_ptr()) if ids else None))
        self._device_inputs = []
        self.sync()
        return (col, dep, idp) if ids else (col, dep)

    def end_frame(self, frame=0, want_z=True, color_out=None, z_out=None):
        """Flush and read the frame back: returns (colour u32[H/k,W/k], depth f32[H/k,W/k] or None)."""
        col = color_out if color_out is not None else np.empty(self.out_shape, np.uint32)
        z = z_out if z_out is not None else (np.empty(self.out_shape, np.float32) if want_z else None)
        self._ck(self.lib.dtr_b200_end_frame(self.ctx, frame, col.ctypes.data_as(C.c_void_p),
                                             z.ctypes.data_as(C.c_void_p) if z is not None else None))
        self._device_inputs = []
        return col, z

    def end_frame_ptr(self, frame, color_ptr, z_ptr=None):
        """end_frame into caller-owned (e.g. pinned) host memory given as raw addresses."""
        self._ck(self.lib.dtr_b200_end_frame(self.ctx, frame, C.c_void_p(color_ptr),
                                             C.c_void_p(z_ptr) if z_ptr else None))
        self._device_inputs = []

    def read_frames_ptr(self, first, n, color_ptr, z_ptr=None):
        """Flush and copy n consecutive frames into caller-owned host memory (raw addresses)."""
        self._ck(self.lib.dtr_b200_read_frames(self.ctx, first, n, C.c_void_p(color_ptr),
                                               C.c_void_p(z_ptr) if z_ptr else None))
        self._device_inputs = []

    def read_frames_async_ptr(self, first, n, color_ptr, z_ptr=None):
        """Flush and enqueue the readback of n frames on the copy stream (page-locked host memory);
        returns at once.  wait_reads() blocks until every outstanding readback has landed."""
        self._ck(self.lib.dtr_b200_read_frames_async(self.ctx, first, n, C.c_void_p(color_ptr),
                                                     C.c_void_p(z_ptr) if z_ptr else None))
        self._device_inputs = []

    def bgr24_pitch(self):
        """Row pitch in bytes of the 24-bit DIB rows written by read_frames_bgr24_async_ptr."""
        return (3 * (self.width // self.resolve) + 3) & ~3

    def read_frames_bgr24_async_ptr(self, first, n, bgr_ptr):
        """Flush, pack n colour planes into 24-bit bottom-up DIBs on the device and enqueue their
        readback (n * bgr24_pitch() * out_shape[0] bytes of page-locked memory); wait_reads() completes it."""
        self._ck(self.lib.dtr_b200_read_frames_bgr24_async(self.ctx, first, n, C.c_void_p(bgr_ptr)))
        self._device_inputs = []

    def wait_reads(self):
        self._ck(self.lib.dtr_b200_wait_reads(self.ctx))

    def upload_font(self, font):
        """font = (atlas u8[h, w], packedchars (scenes.PACKEDCHAR), cpMin, cpMax) -- a flattened DTRFont."""
        key = id(font[0])
        if key in self._font:
            return self._font[key][0]
        atlas, chars, cp_min, cp_max = font
        a = np.ascontiguousarray(atlas, dtype=np.uint8)
        ch = np.ascontiguousarray(chars)
        if ch.dtype.itemsize != 28 or ch.size != cp_max - cp_min:
            raise ValueError("packedchars must be 28-byte stbtt_packedchar records, one per codepoint")
        fid = C.c_int(-1)
        self._ck(self.lib.dtr_b200_upload_font(self.ctx, a.ctypes.data_as(_u8), a.shape[1], a.shape[0],
                                               ch.ctypes.data_as(C.c_void_p), cp_min, cp_max, C.byref(fid)))
        self._font[key] = (fid.value, font)
        return fid.value

    def text(self, font, pos, text, color, length=-1):
        """DTRRender_Text (DTRendererRender.h:91)."""
        fid = self.upload_font(font)
        raw = text.encode("latin-1") if isinstance(text, str) else text
        self._ck(self.lib.dtr_b200_text(self.ctx, fid, _fp(_fa(pos, 2)), raw, _fp(_fa(color, 4)), length))

    def set_debug_markers(self, enable=True):
        """Emit the overlay of the reference's default (DTR_DEBUG_RENDER 1) build from rectangle/bitmap."""
        self._ck(self.lib.dtr_b200_set_debug_markers(self.ctx, 1 if enable else 0))

    def export_frames(self):
        """CUDA IPC handles (2 x 64 bytes) of this context's colour and depth planes."""
        hc, hz = (C.c_uint8 * 64)(), (C.c_uint8 * 64)()
        self._ck(self.lib.dtr_b200_export_frames(self.ctx, hc, hz))
        return bytes(hc), bytes(hz)

    def open_peer_frames(self, color_handle, depth_handle):
        """Render into the frames another process exported (sort-first bands over NVLink)."""
        hc, hz = (C.c_uint8 * 64)(*color_handle), (C.c_uint8 * 64)(*depth_handle)
        self._ck(self.lib.dtr_b200_open_peer_frames(self.ctx, hc, hz))

    def set_output_planes(self, color_ptr, depth_ptr):
        self._ck(self.lib.dtr_b200_set_output_planes(self.ctx, C.c_void_p(color_ptr), C.c_void_p(depth_ptr)))

    def enable_peer_access(self, peer_device):
        self._ck(self.lib.dtr_b200_enable_peer_access(self.ctx, peer_device))

    def frame_device_ptrs(self, frame=0):
        c, z = C.c_void_p(), C.c_void_p()
        self._ck(self.lib.dtr_b200_frame_device_ptrs(self.ctx, frame, C.byref(c), C.byref(z)))
        return c.value, z.value

    # ---- triangle id planes (see dtr_b200_set_id_output) ----------------------------------------
    def set_id_output(self, on=True):
        """Keep a u32 id plane per frame: 1 + the frame position of the triangle whose fragment last wrote
        a pixel's depth since the frame's begin_frame, 0 where none did (for one mesh call: face index + 1)."""
        self._ck(self.lib.dtr_b200_set_id_output(self.ctx, 1 if on else 0))

    def read_ids(self, first=0, n=1):
        """Flush and read the id planes of frames [first, first + n): u32[n, H/k, W/k]."""
        out = np.empty((n, *self.out_shape), np.uint32)
        self._ck(self.lib.dtr_b200_read_ids(self.ctx, first, n, out.ctypes.data_as(C.c_void_p)))
        self._device_inputs = []
        return out

    def frame_id_ptr(self, frame=0):
        """Device address of a frame's id plane (u32[H*W])."""
        p = C.c_void_p()
        self._ck(self.lib.dtr_b200_frame_id_ptr(self.ctx, frame, C.byref(p)))
        return p.value

    def stats(self):
        s = Stats()
        self._ck(self.lib.dtr_b200_get_stats(self.ctx, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in Stats._fields_}

    def last_pass_deferred(self):
        """True when the last flush / replay used the deferred raster stage (a pass that can never blend:
        visibility first, every visible pixel shaded once) -- in one kernel or in two, see last_pass_stage()."""
        return bool(self.lib.dtr_b200_last_pass_deferred(self.ctx))

    def last_pass_stage(self):
        """OPAQUE_SINGLE_KERNEL (0), OPAQUE_TWO_KERNELS (1) or OPAQUE_ONE_KERNEL (2): what the last pass ran."""
        return int(self.lib.dtr_b200_last_pass_deferred(self.ctx))

    def set_opaque_stage(self, mode):
        """How passes made only of opaque triangles onto cleared frames run from now on (dtr_b200_set_opaque_stage)."""
        self._ck(self.lib.dtr_b200_set_opaque_stage(self.ctx, int(mode)))

    def reset_stats(self):
        self._ck(self.lib.dtr_b200_reset_stats(self.ctx))

    def set_profiling(self, on=True):
        self._ck(self.lib.dtr_b200_set_profiling(self.ctx, int(on)))

    def reset_stage_ms(self):
        self._ck(self.lib.dtr_b200_reset_stage_ms(self.ctx))

    def stage_ms(self):
        """Summed device ms of (setup, scan, bin, raster) and the number of pipelines timed."""
        ms, runs = (C.c_float * 4)(), C.c_int(0)
        self._ck(self.lib.dtr_b200_get_stage_ms(self.ctx, C.byref(ms), C.byref(runs)))
        return dict(setup=ms[0], scan=ms[1], bin=ms[2], raster=ms[3]), runs.value

    def raster_split_ms(self):
        """Summed device ms of the raster stage's kernels: (first kernel = the single raster kernel, the
        one-kernel opaque stage or the visibility kernel; resolve kernel, ~0 unless the stage is two kernels),
        and the number of pipelines timed."""
        ms, runs = (C.c_float * 2)(), C.c_int(0)
        self._ck(self.lib.dtr_b200_get_raster_split_ms(self.ctx, C.byref(ms), C.byref(runs)))
        return (ms[0], ms[1]), runs.value

    def selftest(self):
        """Mismatches of the device arithmetic self-test (must be 0)."""
        n = C.c_uint64(1)
        self._ck(self.lib.dtr_b200_selftest(self.ctx, C.byref(n)))
        return int(n.value)

    def counters(self):
        s = self.stats()
        return (s["setPixels"], s["triangles"])

    # ---- draw calls (names and argument meaning of DTRendererRender.h:91-98) ------------------
    def clear(self, rgb):
        self._ck(self.lib.dtr_b200_clear(self.ctx, _fp(_fa(rgb, 3))))

    def triangle(self, p, color, transform=None):
        p = _fa(p, 9)
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_triangle(self.ctx, _fp(p[0:3]), _fp(p[3:6]), _fp(p[6:9]), _fp(_fa(color, 4)),
                                            C.byref(t) if t else None))

    def triangles(self, p, color, transform=None):
        p = _fa(p)
        n = p.size // 9
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_triangles(self.ctx, n, _fp(p), _fp(_fa(color, 4 * n)),
                                             C.byref(t) if t else None))

    def textured_triangle(self, p, uv, tex, color, transform=None):
        p, uv = _fa(p, 9), _fa(uv, 6)
        tid = self.upload_texture(tex) if tex is not None else -1
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_textured_triangle(self.ctx, _fp(p[0:3]), _fp(p[3:6]), _fp(p[6:9]),
                                                     _fp(uv[0:2]), _fp(uv[2:4]), _fp(uv[4:6]), tid,
                                                     _fp(_fa(color, 4)), C.byref(t) if t else None))

    def textured_triangle_id(self, p, uv, tex_id, color, transform=None):
        """DTRRender_TexturedTriangle with a texture that is already on the device (tex_id < 0: untextured)."""
        p, uv = _fa(p, 9), _fa(uv, 6)
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_textured_triangle(self.ctx, _fp(p[0:3]), _fp(p[3:6]), _fp(p[6:9]),
                                                     _fp(uv[0:2]), _fp(uv[2:4]), _fp(uv[4:6]), int(tex_id),
                                                     _fp(_fa(color, 4)), C.byref(t) if t else None))

    @staticmethod
    def _light(light_mode, light_vector, light_color):
        return Light(int(light_mode), (C.c_float * 3)(*_fa(light_vector, 3)), (C.c_float * 4)(*_fa(light_color, 4)))

    def mesh(self, mesh, tex, light_mode, light_vector, light_color, pos=(0, 0, 0), transform=None):
        tid = self.upload_texture(tex)
        mid = self.upload_mesh(mesh, tid)
        light = self._light(light_mode, light_vector, light_color)
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_mesh(self.ctx, mid, C.byref(light), _fp(_fa(pos, 3)), C.byref(t) if t else None))

    def mesh_views(self, mesh, tex, light_mode, light_vector, light_color, positions, transforms, first_frame=0):
        tid = self.upload_texture(tex)
        mid = self.upload_mesh(mesh, tid)
        light = self._light(light_mode, light_vector, light_color)
        n = len(transforms)
        arr = (Transform * n)(*[make_transform(t) for t in transforms])
        self._ck(self.lib.dtr_b200_mesh_views(self.ctx, mid, C.byref(light), n, _fp(_fa(positions, 3 * n)), arr,
                                              first_frame))

    # ---- draw calls from device memory (dtr_b200_triangles_device / dtr_b200_mesh_views_device) ---------------
    def _device_tensor(self, t, n, what):
        """Address of t, a contiguous float32 torch tensor of n elements on this renderer's device (no copy is made)."""
        import torch
        if not isinstance(t, torch.Tensor) or t.device != torch.device("cuda", self.device):
            raise ValueError(f"{what} must be a torch tensor on cuda:{self.device}")
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"{what} must be contiguous float32, got {t.dtype} (contiguous: {t.is_contiguous()})")
        if t.numel() != n:
            raise ValueError(f"{what}: expected {n} elements, got {t.numel()}")
        return t.data_ptr()

    def _record_device(self, tensors):
        """Order torch's work on the tensors before the flush that reads them, and keep them alive until then."""
        import torch
        cur = torch.cuda.current_stream(self.device)
        if self._stream is None or cur.cuda_stream != self._stream:
            cur.synchronize()
        self._device_inputs.extend(t for t in tensors if t is not None)

    def triangles_device(self, p, color, uv=None, tex_id=-1, transform=None):
        """dtr_b200_triangles_device: n triangles from torch CUDA tensors p (n*9), color (n*4) and uv (n*6) or None,
        read by the next flush; bit for bit triangles() (textured_triangle_id() per triangle with uv and tex_id >= 0)."""
        n = p.numel() // 9 if hasattr(p, "numel") else 0
        pp = self._device_tensor(p, 9 * n, "p")
        cp = self._device_tensor(color, 4 * n, "color")
        up = self._device_tensor(uv, 6 * n, "uv") if uv is not None else None
        t = make_transform(transform)
        self._record_device((p, color, uv))
        self._ck(self.lib.dtr_b200_triangles_device(self.ctx, n, C.c_void_p(pp), C.c_void_p(cp),
                                                    C.c_void_p(up) if up else None, int(tex_id), C.byref(t) if t else None))

    def mesh_views_device(self, mesh_id, light_mode, light_vector, light_color, positions, transforms, vertexes,
                          normals=None, first_frame=0):
        """dtr_b200_mesh_views_device: view i is mesh mesh_id with vertex set i of vertexes (torch CUDA tensor of
        n_views * numVertexes * 4 floats) and normal set i of normals (n_views * numNormals * 3, or None: the mesh's
        own), drawn into frame first_frame + i."""
        if mesh_id not in self._mesh_counts:
            raise ValueError(f"mesh {mesh_id} was not uploaded through this renderer")
        nv, nn = self._mesh_counts[mesh_id]
        n = len(transforms)
        vp = self._device_tensor(vertexes, n * nv * 4, "vertexes")
        np_ = self._device_tensor(normals, n * nn * 3, "normals") if normals is not None else None
        light = self._light(light_mode, light_vector, light_color)
        arr = (Transform * n)(*[make_transform(t) for t in transforms])
        self._record_device((vertexes, normals))
        self._ck(self.lib.dtr_b200_mesh_views_device(self.ctx, mesh_id, C.byref(light), n, _fp(_fa(positions, 3 * n)), arr,
                                                     first_frame, C.c_void_p(vp), C.c_void_p(np_) if np_ else None))

    def rectangle(self, mn, mx, color, transform=None):
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_rectangle(self.ctx, _fp(_fa(mn, 2)), _fp(_fa(mx, 2)), _fp(_fa(color, 4)),
                                             C.byref(t) if t else None))

    def bitmap(self, tex, pos, transform=None, color=(1, 1, 1, 1)):
        tid = self.upload_texture(tex)
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_bitmap(self.ctx, tid, _fp(_fa(pos, 2)), C.byref(t) if t else None,
                                          _fp(_fa(color, 4))))

    def bitmap_id(self, tex_id, pos, transform=None, color=(1, 1, 1, 1)):
        """DTRRender_Bitmap with a texture that is already on the device (see upload_bitmap_straight)."""
        t = make_transform(transform)
        self._ck(self.lib.dtr_b200_bitmap(self.ctx, tex_id, _fp(_fa(pos, 2)), C.byref(t) if t else None,
                                          _fp(_fa(color, 4))))

    def line(self, a, b, color):
        a = np.ascontiguousarray(a, dtype=np.int32)
        b = np.ascontiguousarray(b, dtype=np.int32)
        self._ck(self.lib.dtr_b200_line(self.ctx, a.ctypes.data_as(_i32), b.ctypes.data_as(_i32), _fp(_fa(color, 4))))
