/* dtr_b200.h -- C ABI of the B200 (sm_100a) rasterisation back end for DTRenderer's draw path.
 *
 * This is the drop-in boundary: one shared library (libdtr_b200.so), `extern "C"`, plain
 * pointers and sizes, no C++/torch types.  Each draw entry replaces one reference draw call
 * (reference paths are relative to /root/reference/src):
 *
 *   dtr_b200_clear              <- DTRRender_Clear             DTRendererRender.h:98,  .cpp:1793-1815
 *   dtr_b200_triangle           <- DTRRender_Triangle          DTRendererRender.h:95,  .cpp:1587-1594
 *   dtr_b200_textured_triangle  <- DTRRender_TexturedTriangle  DTRendererRender.h:96,  .cpp:1358-1365
 *   dtr_b200_mesh               <- DTRRender_Mesh              DTRendererRender.h:94,  .cpp:1395-1585
 *   dtr_b200_rectangle          <- DTRRender_Rectangle         DTRendererRender.h:93,  .cpp:415-513
 *   dtr_b200_bitmap             <- DTRRender_Bitmap            DTRendererRender.h:97,  .cpp:1596-1791
 *   dtr_b200_line               <- DTRRender_Line              DTRendererRender.h:92,  .cpp:294-356
 *   dtr_b200_begin_frame        <- per-frame z-buffer reset    DTRenderer.cpp:967-978
 *   dtr_b200_end_frame          <- hand-back of the DTRRenderBuffer (DTRendererRender.h:14-25)
 *   dtr_b200_upload_mesh/_texture <- DTRMesh / DTRBitmap as produced by DTRendererAsset
 *                                    (DTRendererAsset.h:9-42); the loaders stay on the host.
 *   dtr_b200_upload_mesh_faces  <- DTRMesh with its per-face index arrays as they lie in the asset
 *                                    arena (DTRendererAsset.h:16-26, .cpp:509-578): flattened on the device
 *   dtr_b200_gather_bands / dtr_b200_band_barrier <- replace the reference's only parallel mode, the
 *                                    per-triangle job fan-out with its per-pixel lock
 *                                    (DTRendererRender.cpp:1367-1393, 1162-1171), for sort-first bands
 *
 * Semantics.  Draw calls are RECORDED and executed in submission order per frame: the result of
 * a flush is the reference's single-threaded (`multithread=false`) in-order result -- coverage,
 * depth decisions and depth values bit-exact, colour bit-exact in practice (tolerance 1/255).
 * Arguments have the reference's meaning: colours are sRGB in [0,1] (gamma 2.0), transform
 * rotation is RADIANS for 2D calls and DEGREES about the axis `anchor` for dtr_b200_mesh
 * (DTRendererRender.cpp:282 vs :1410), buffers are row-major with row 0 at the bottom, colour
 * pixels are 0x00RRGGBB and depth is f32 with larger = nearer, reset value -FLT_MAX.
 * Inputs the reference would assert on (w != 1, uv > 1, colours outside [0,1], w_clip <= 0)
 * are undefined here too.
 *
 * Errors.  Every call returns 0 on success or a negative dtr_b200_status; NULL/invalid
 * arguments that the reference silently ignores (DTRendererRender.cpp:128,420,1402,1601,1796)
 * return DTR_B200_OK without drawing.  There is NO CPU fallback: without a CUDA device
 * dtr_b200_create fails with DTR_B200_ERR_CUDA.
 *
 * Threading.  One host thread per context; all work is enqueued on the context's CUDA stream.
 */
#ifndef DTR_B200_H
#define DTR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dtr_b200_ctx dtr_b200_ctx;

typedef enum dtr_b200_status
{
	DTR_B200_OK           = 0,
	DTR_B200_ERR_ARG      = -1, /* out-of-range id / frame / size */
	DTR_B200_ERR_CUDA     = -2, /* CUDA runtime error, see dtr_b200_last_error */
	DTR_B200_ERR_NOMEM    = -3,
	DTR_B200_ERR_OVERFLOW = -4, /* more than 2^31 primitives / list entries in one flush */
} dtr_b200_status;

/* Layout-compatible with DTRRenderTransform (DTRendererRender.h:28-33): 7 floats. */
typedef struct dtr_b200_transform
{
	float rotation;
	float anchor[3];
	float scale[3];
} dtr_b200_transform;

/* DTRRenderShadingMode (DTRendererRender.h:63-68) */
enum
{
	DTR_B200_SHADE_FULLBRIGHT = 0,
	DTR_B200_SHADE_FLAT       = 1,
	DTR_B200_SHADE_GOURAUD    = 2,
};

/* Layout-compatible with DTRRenderLight (DTRendererRender.h:72-77). */
typedef struct dtr_b200_light
{
	int32_t mode;
	float   vector[3];
	float   color[4];
} dtr_b200_light;

/* DTRMesh flattened (DTRendererAsset.h:16-41): the per-face index arrays become one
 * i32[numFaces*9] = {v0,v1,v2, t0,t1,t2, n0,n1,n2}. */
typedef struct dtr_b200_mesh_desc
{
	const float   *vertexes; /* f32[numVertexes*4], w must be 1 */
	uint32_t       numVertexes;
	const float   *texUV;    /* f32[numTexUV*3] */
	uint32_t       numTexUV;
	const float   *normals;  /* f32[numNormals*3] */
	uint32_t       numNormals;
	const int32_t *faces;    /* i32[numFaces*9] */
	uint32_t       numFaces;
} dtr_b200_mesh_desc;

typedef struct dtr_b200_stats
{
	uint64_t setPixels;    /* fragments that passed coverage and the z-test == DTRDebugCounter_SetPixels */
	uint64_t triangles;    /* triangles submitted == DTRDebugCounter_RenderTriangle */
	uint64_t primitives;   /* primitives in the last flush */
	uint64_t listEntries;  /* (primitive, tile) pairs in the last flush */
	uint64_t kernelLaunches; /* kernels launched by this context so far */
	uint64_t uploadBytes;  /* host->device bytes of the last flush (command block + payload) */
} dtr_b200_stats;

/* ---- context ------------------------------------------------------------------------------ */
/* numFrames colour+depth targets of width x height live in HBM; draw calls go to the current
 * target (dtr_b200_set_target), so one flush can render a whole batch of frames/viewpoints. */
int         dtr_b200_create(int device, int width, int height, int numFrames, dtr_b200_ctx **out);
void        dtr_b200_destroy(dtr_b200_ctx *ctx);
const char *dtr_b200_last_error(const dtr_b200_ctx *ctx); /* ctx may be NULL: last create error */
const char *dtr_b200_version(void);
/* Use an existing cudaStream_t (e.g. the caller's current stream) instead of the context's own. */
int         dtr_b200_set_stream(dtr_b200_ctx *ctx, void *cudaStream);
/* Sort-first band split: only rows [y0,y1) are rasterised by this context (tile aligned: both
 * multiples of dtr_b200_tile_height() or y1 == height).  Default is the whole frame. */
int         dtr_b200_set_band(dtr_b200_ctx *ctx, int y0, int y1);
/* Height in pixels of a screen tile of this build (32): the granularity of bands. */
int         dtr_b200_tile_height(void);
/* THE band partition: tile-aligned rows [*y0, *y1) of rank `rank` out of `nranks`; the bands tile
 * [0, height) exactly, trailing ranks get an empty band when there are fewer tile rows than ranks. */
int         dtr_b200_band_rows(int height, int nranks, int rank, int *y0, int *y1);

/* ---- assets (device resident until destroy) ----------------------------------------------- */
int dtr_b200_upload_texture(dtr_b200_ctx *ctx, const uint8_t *texels, int width, int height,
                            int bytesPerPixel /* must be 4 */, int *texId);
/* The step before the hot path (SURVEY.md §8f rank 3): DTRAsset_LoadBitmap's per-pixel pass
 * (DTRendererAsset.cpp:816-843) on the device.  `rgba` is what stb_image hands the reference
 * (straight alpha, R in the low byte, rows already flipped by stbi_set_flip_vertically_on_load);
 * the stored texture is premultiplied in sRGB space, bit for bit what DTRBitmap::memory holds after
 * DTRAsset_LoadBitmap.  dtr_b200_read_texture copies a texture back (tests, tools). */
int dtr_b200_upload_bitmap_straight(dtr_b200_ctx *ctx, const uint8_t *rgba, int width, int height, int *texId);
int dtr_b200_read_texture(dtr_b200_ctx *ctx, int texId, uint8_t *rgba);
int dtr_b200_upload_mesh(dtr_b200_ctx *ctx, const dtr_b200_mesh_desc *mesh, int texId, int *meshId);
/* The other half of SURVEY.md §8f rank 3: DTRMesh as DTRAsset_LoadWavefrontObj leaves it
 * (DTRendererAsset.cpp:509-578) -- an array of DTRMeshFace, each pointing at three separately
 * allocated i32 index arrays inside the asset arena -- flattened ON THE DEVICE.  `faces` is the
 * DTRMeshFace array itself (dtr_b200_mesh_face is layout compatible with DTRMeshFace,
 * DTRendererAsset.h:16-26); [arena, arena + arenaBytes) is the host memory block that contains every
 * index array the faces point to (the reference's assetStack block).  The block and the face array are
 * uploaded with one copy each and a gather kernel chases the (rebased) pointers into i32[numFaces][9];
 * no per-face host loop.  Faces whose pointers leave the arena, whose counts are not 3/>=3/3 (the
 * reference asserts, DTRendererRender.cpp:1440-1441) or whose indices are out of range make the call
 * fail with DTR_B200_ERR_ARG. */
typedef struct dtr_b200_mesh_face
{
	const int32_t *vertexIndex;
	uint32_t       numVertexIndex;
	const int32_t *texIndex;
	uint32_t       numTexIndex;
	const int32_t *normalIndex;
	uint32_t       numNormalIndex;
} dtr_b200_mesh_face;
typedef struct dtr_b200_mesh_faces_desc
{
	const float              *vertexes; /* f32[numVertexes*4], w must be 1 */
	uint32_t                  numVertexes;
	const float              *texUV;    /* f32[numTexUV*3] */
	uint32_t                  numTexUV;
	const float              *normals;  /* f32[numNormals*3] */
	uint32_t                  numNormals;
	const dtr_b200_mesh_face *faces;    /* DTRMeshFace[numFaces] */
	uint32_t                  numFaces;
	const void               *arena;    /* host block containing every index array */
	size_t                    arenaBytes;
} dtr_b200_mesh_faces_desc;
int dtr_b200_upload_mesh_faces(dtr_b200_ctx *ctx, const dtr_b200_mesh_faces_desc *mesh, int texId, int *meshId);
/* Forget cached device copies after the host changed a texture in place: the texture keeps its id, its
 * contents are uploaded again (same dimensions required).  A mesh's vertexes and normals can change per draw
 * call instead, from device memory: dtr_b200_mesh_views_device. */
int dtr_b200_update_texture(dtr_b200_ctx *ctx, int texId, const uint8_t *texels);

/* ---- frame -------------------------------------------------------------------------------- */
int dtr_b200_set_target(dtr_b200_ctx *ctx, int frame);
/* Start a frame on `frame`: depth is reset to -FLT_MAX (hostZ == NULL) or uploaded; colour is
 * kept from the previous frame (hostColor == NULL, as the reference's platform buffer is) or
 * uploaded.  Host buffers are W*H elements, caller owned, only read here. */
int dtr_b200_begin_frame(dtr_b200_ctx *ctx, int frame, const uint32_t *hostColor, const float *hostZ);
/* Execute everything recorded so far (asynchronous on the context's stream). */
int dtr_b200_flush(dtr_b200_ctx *ctx);
/* Re-execute the last flushed command list from its device-resident copy (no host->device
 * traffic): every frame it touched is re-initialised the way it was before that flush. */
int dtr_b200_replay(dtr_b200_ctx *ctx);
/* Consecutive replays are pipelined by default: setup / scan / bin of replay i+1 run on a second
 * stream with their own buffer set while the raster kernel of replay i is finishing (its tail
 * leaves SMs idle); the raster kernels stay ordered.  Results are unaffected.  Disable (0) to time
 * the stages in isolation: with the overlap on, the per-stage times of dtr_b200_get_stage_ms
 * include the time a stage waited for free SMs. */
int dtr_b200_set_replay_overlap(dtr_b200_ctx *ctx, int enable);
int dtr_b200_sync(dtr_b200_ctx *ctx);
/* Flush, then copy the frame back (either pointer may be NULL) and wait for it. */
int dtr_b200_end_frame(dtr_b200_ctx *ctx, int frame, uint32_t *hostColor, float *hostZ);
/* Flush, then copy n consecutive frames back in one transfer per plane (either pointer may be
 * NULL): hostColor u32[n*W*H], hostZ f32[n*W*H]; waits for completion. */
int dtr_b200_read_frames(dtr_b200_ctx *ctx, int firstFrame, int n, uint32_t *hostColor, float *hostZ);
/* Presentation hand-off without stalling the renderer (the step after the hot path, SURVEY.md §8f
 * rank 4; the reference presents with StretchDIBits, Win32DTRenderer.cpp:267-284): flush, then
 * enqueue the same copies on the context's copy stream, ordered after the rendering submitted so
 * far, and return.  Rendering into OTHER frames may be submitted while the copies are in flight (a
 * flush that touches a frame still being read waits for the copy on the device).  The host
 * buffers must be page-locked for the copy to overlap; they are valid after dtr_b200_wait_reads. */
int dtr_b200_read_frames_async(dtr_b200_ctx *ctx, int firstFrame, int n, uint32_t *hostColor, float *hostZ);
int dtr_b200_wait_reads(dtr_b200_ctx *ctx);
/* The same hand-off with an on-device encode (SURVEY.md §8f rank 4, "on-device encode"): the X
 * byte of DTRRenderBuffer's 0x00RRGGBB pixels (DTRendererRender.h:14-25) is always 0, so the n
 * colour planes are packed on the device into 24-bit bottom-up DIBs -- B,G,R per pixel, row pitch
 * ((3*W + 3) & ~3) bytes, rows bottom first like the planes -- which StretchDIBits
 * (Win32DTRenderer.cpp:267-284) presents with biBitCount = 24, and 3/4 of the bytes cross PCIe.
 * hostBgr: n * pitch * H bytes, page-locked; valid after dtr_b200_wait_reads.  The frames may be
 * rendered into again at once (the pack runs in stream order, the transfer reads a staging copy). */
int dtr_b200_read_frames_bgr24_async(dtr_b200_ctx *ctx, int firstFrame, int n, uint8_t *hostBgr);
/* Supersampled output: a context has a READBACK RESOLVE FACTOR k, default 1.  Render into a kW x kH
 * context and every host readback -- dtr_b200_end_frame, dtr_b200_read_frames, dtr_b200_read_frames_async,
 * dtr_b200_read_frames_bgr24_async (pitch ((3*W/k + 3) & ~3)) and dtr_b200_read_ids -- returns frames of
 * (W/k) x (H/k), row 0 at the bottom as before.  Output pixel (X, Y) is made on the device from the block of
 * samples [kX, kX+k) x [kY, kY+k) of the frame's planes:
 *   colour  each of the four bytes of the 0x00RRGGBB word separately (the X byte too, which clear colours
 *           outside [0, 1] can set): the integer square root of the integer mean, rounded down, of the squared
 *           sample bytes, floor(sqrt(floor(sum(b^2) / k^2))) -- the largest v with v^2 k^2 <= sum(b^2).  This is
 *           the mean in the reference's gamma-2 linear space, encoded back with truncation; a block of equal
 *           words resolves to that word.
 *   depth   one sample per block: scanning the block row by row from its bottom-left sample, the first sample
 *   and id  is taken and replaced only by a sample whose depth compares > (IEEE) with the current one (ties
 *           and NaN keep the earlier sample).  Depth is the chosen sample's bits, the id the chosen sample's
 *           id: both always come from the same fragment.
 * k = 1 is the plain readback (the same copies, no resolve kernel).  Uploads (dtr_b200_begin_frame), device
 * pointers (dtr_b200_frame_device_ptrs, dtr_b200_frame_id_ptr), every draw call and dtr_b200_get_stats stay at
 * sample resolution: setPixels counts samples, and resolve kernels are not counted in kernelLaunches.
 * A resolved asynchronous readback resolves into a device staging buffer on the context's stream and copies
 * from there, so the frames may be rendered into again at once.
 *   dtr_b200_set_readback_resolve  k in 1..4 dividing width and height, else DTR_B200_ERR_ARG and the old factor
 *                                  stays.  Applies to readbacks issued after the call.
 *   dtr_b200_resolve_frames        flush, then write the resolved planes of frames [firstFrame, firstFrame + n)
 *                                  into caller-owned DEVICE memory (u32 / f32 / u32 [n][H/k][W/k], each may be
 *                                  NULL), stream-ordered on the context's stream: the zero-copy path.  ids without
 *                                  id output (dtr_b200_set_id_output) or a bad range: DTR_B200_ERR_ARG. */
int dtr_b200_set_readback_resolve(dtr_b200_ctx *ctx, int k);
int dtr_b200_resolve_frames(dtr_b200_ctx *ctx, int firstFrame, int n, void *color, void *z, void *ids);
/* Render to texture: frames become textures on the device, with no host round trip.  Converting frame f of a
 * W x H context with readback resolve factor k gives a texture of (W/k) x (H/k) texels, row 0 at the bottom
 * (frames and textures share it: no flip).  Texel (x, y) comes from w, the frame's resolved colour word at
 * (x, y) -- the sample itself at k = 1, the resolve rule above per byte at k > 1 -- in the DTRBitmap layout:
 * bytes R, G, B, A = (w >> 16) & 0xFF, (w >> 8) & 0xFF, w & 0xFF, 0xFF, i.e. the u32 R | G<<8 | B<<16 | 0xFF000000.
 * The X byte is dropped; A = 255, so the texel is trivially premultiplied and the texture opaque.  Drawing with
 * such a texture is bit for bit drawing with dtr_b200_upload_texture / dtr_b200_update_texture of the same
 * conversion done on the host from a readback issued at that point.
 *   dtr_b200_create_texture     a device-only texture (no host bytes, no upload), dimensions in [1, 32767].
 *                               Its contents and flags are those of dtr_b200_upload_texture with all-zero
 *                               texels: transparent black, neither white nor opaque.
 *   dtr_b200_frames_to_textures flush (the conversion sees every draw call submitted before it), then write frame
 *                               firstFrame + i into texture texIds[i] for every i < n: one kernel, stream-ordered
 *                               on the context's stream, no host synchronisation.  Draw calls recorded afterwards
 *                               sample the new texels; a replay needs a flush first (DTR_B200_ERR_ARG until then).
 *                               DTR_B200_ERR_ARG, with nothing enqueued, for a bad frame range or n < 1, a texId
 *                               out of range, a texture that is not (W/k) x (H/k), a texId given twice, or
 *                               foreign output planes (dtr_b200_set_output_planes / dtr_b200_open_peer_frames):
 *                               the frames are then not in this context's planes.  Like the resolve kernels the
 *                               conversion is not counted in kernelLaunches.
 * dtr_b200_read_texture waits for the conversions enqueued before it. */
int dtr_b200_create_texture(dtr_b200_ctx *ctx, int width, int height, int *texId);
int dtr_b200_frames_to_textures(dtr_b200_ctx *ctx, int firstFrame, int n, const int *texIds);
/* Sort-first screen bands WITHOUT a gather step (SURVEY.md §8e): every rank rasterises its band
 * (dtr_b200_set_band) but writes the finished regions straight into the gathering rank's frame
 * planes over NVLink, from inside the raster kernel's write-back -- the transfer overlaps the
 * rasterisation tile by tile and nothing is copied afterwards.  The planes have the layout of
 * DTRRenderBuffer (DTRendererRender.h:14-25), F frames back to back.
 *   dtr_b200_export_frames        rank 0: CUDA IPC handles of its colour / depth planes
 *   dtr_b200_open_peer_frames     other ranks (other processes): map them and render into them
 *   dtr_b200_set_output_planes    same-process variant: raw pointers of another context's planes
 *                                 (after dtr_b200_enable_peer_access); NULL, NULL = own planes again
 * The caller orders "all ranks finished" before reading the frames (a barrier / stream event). */
#define DTR_B200_IPC_HANDLE_BYTES 64
int dtr_b200_export_frames(dtr_b200_ctx *ctx, uint8_t *colorHandle, uint8_t *depthHandle);
int dtr_b200_open_peer_frames(dtr_b200_ctx *ctx, const uint8_t *colorHandle, const uint8_t *depthHandle);
int dtr_b200_set_output_planes(dtr_b200_ctx *ctx, void *color, void *depth);
int dtr_b200_enable_peer_access(dtr_b200_ctx *ctx, int peerDevice);
/* Sort-first bands from a C/C++ host, no Python: the exchange step and its barrier behind the C ABI
 * (SURVEY.md §8b/§8e).  NCCL is bound at run time (dlopen of libnccl.so.2 -- the copy already loaded
 * into the process if there is one -- so the library has no link-time NCCL dependency).
 *   dtr_b200_band_comm_unique_id  rank 0: a fresh ncclUniqueId (128 bytes) to hand to the other ranks
 *   dtr_b200_band_comm_init       every rank: ncclCommInitRank on this context's device
 *   dtr_b200_band_comm_attach     alternative: use a communicator the host already owns (an
 *                                 ncclComm_t passed as void *; not destroyed with the context)
 *   dtr_b200_gather_bands         flush, then one grouped ncclSend/ncclRecv on the context's stream:
 *                                 every rank's band rows (dtr_b200_band_rows of its rank) of colour and
 *                                 depth of `frame` land in the same rows of rank dstRank's planes.
 *                                 The baseline exchange; the fused peer-memory write-back above is faster.
 *   dtr_b200_band_barrier         stream-ordered barrier (a 4-byte ncclAllReduce on the context's
 *                                 stream): after it completes on rank r, every rank's work enqueued
 *                                 before its own barrier call -- e.g. the raster kernel that writes its
 *                                 band into r's planes -- has finished. */
#define DTR_B200_NCCL_ID_BYTES 128
int dtr_b200_band_comm_unique_id(uint8_t id[DTR_B200_NCCL_ID_BYTES]);
int dtr_b200_band_comm_init(dtr_b200_ctx *ctx, const uint8_t id[DTR_B200_NCCL_ID_BYTES], int nranks, int rank);
int dtr_b200_band_comm_attach(dtr_b200_ctx *ctx, void *ncclComm, int nranks, int rank);
int dtr_b200_gather_bands(dtr_b200_ctx *ctx, int frame, int dstRank);
int dtr_b200_band_barrier(dtr_b200_ctx *ctx);
/* Device pointers of a frame's planes (u32[W*H], f32[W*H]) for zero-copy consumers
 * (NCCL / peer access / torch views). */
int dtr_b200_frame_device_ptrs(dtr_b200_ctx *ctx, int frame, void **color, void **z);
/* Triangle id planes: a third plane per frame, u32[F][H][W], row 0 at the bottom like the depth plane.
 * A pixel holds 0 when no triangle fragment has written its depth since the frame's depth was last reset
 * or uploaded (dtr_b200_begin_frame), else 1 + n, n the 0-based position in the frame of the triangle
 * whose fragment last wrote depth there.  Triangles are counted in submission order since the frame's
 * begin_frame, across flushes, every submitted one included: triangle / textured_triangle 1, triangles n,
 * mesh and each view of mesh_views numFaces (face order).  The id changes exactly when depth does
 * (translucent fragments write depth too); rectangles, bitmaps, lines, text and clears never touch it.
 * With a band (set_band) only the band's rows are written; with foreign output planes
 * (set_output_planes / open_peer_frames) the ids still go to this context's own planes.
 *   dtr_b200_set_id_output  enable: allocate and zero the planes (DTR_B200_ERR_NOMEM if that fails);
 *                           0: free them.  Applies to every later flush and replay.
 *   dtr_b200_read_ids       flushes, copies frames [firstFrame, firstFrame + n) and waits
 *   dtr_b200_frame_id_ptr   device pointer of a frame's id plane
 * Both readers return DTR_B200_ERR_ARG when ids are off or the frame range is bad. */
int dtr_b200_set_id_output(dtr_b200_ctx *ctx, int enable);
int dtr_b200_read_ids(dtr_b200_ctx *ctx, int firstFrame, int n, uint32_t *hostIds);
int dtr_b200_frame_id_ptr(dtr_b200_ctx *ctx, int frame, void **ids);
int dtr_b200_get_stats(dtr_b200_ctx *ctx, dtr_b200_stats *out); /* syncs */
/* How the raster stage of a pass made ONLY of opaque triangles onto frames cleared on chip runs (nothing
 * can ever be blended there: a pixel's colour is the shading of the last fragment that passed the depth
 * test, DTRendererRender.cpp:124-191 with alpha 1).  Results are identical in every mode; every other pass
 * takes the single raster kernel whatever the mode.
 *   DTR_B200_OPAQUE_ONE_KERNEL (default)  visibility (depth test, primitive tags) and the shading of each
 *                                         finished region's visible pixels in one kernel
 *   DTR_B200_OPAQUE_TWO_KERNELS           visibility kernel, then a resolve kernel over the busy tiles
 *   DTR_B200_OPAQUE_SINGLE_KERNEL         the general raster kernel (shades every fragment that passes)
 * Environment (defaults of new contexts): DTR_B200_FUSED=0 -> TWO_KERNELS, DTR_B200_DEFER=0 -> SINGLE_KERNEL. */
enum
{
	DTR_B200_OPAQUE_SINGLE_KERNEL = 0,
	DTR_B200_OPAQUE_TWO_KERNELS   = 1,
	DTR_B200_OPAQUE_ONE_KERNEL    = 2
};
int dtr_b200_set_opaque_stage(dtr_b200_ctx *ctx, int mode);
/* Which of them the last flush / replay ran: 0 = the single raster kernel (the pass could blend, or the mode
 * says so), DTR_B200_OPAQUE_TWO_KERNELS, DTR_B200_OPAQUE_ONE_KERNEL. */
int dtr_b200_last_pass_deferred(const dtr_b200_ctx *ctx);
int dtr_b200_reset_stats(dtr_b200_ctx *ctx);
/* Per-stage device timing with CUDA events on the context's stream (the ncu/nsys replacement of
 * the reference's rdtsc region counters, DTRendererDebug.h:42-78).  While enabled, every
 * flush/replay records 7 events; dtr_b200_get_stage_ms syncs and returns the SUMS in ms of
 * {setup, scan, bin, raster} over the pipelines run since the last reset, and their number. */
int dtr_b200_set_profiling(dtr_b200_ctx *ctx, int enable);
int dtr_b200_get_stage_ms(dtr_b200_ctx *ctx, float ms[4], int *runs);
/* The raster stage of the same runs, split at the event between its kernels: ms[0] = the stage's first
 * kernel (the single raster kernel, the one-kernel opaque stage, or the visibility kernel of the two-kernel
 * stage), ms[1] = the resolve kernel (~0 when the stage is one kernel).  ms[0] + ms[1] = the raster entry
 * of get_stage_ms. */
int dtr_b200_get_raster_split_ms(dtr_b200_ctx *ctx, float ms[2], int *runs);
int dtr_b200_reset_stage_ms(dtr_b200_ctx *ctx);

/* Device self-test of the arithmetic shortcuts: the blend's branch-free square root is compared
 * with IEEE sqrtf on every float in [2^-60, 4).  *mismatches must come back 0. */
int dtr_b200_selftest(dtr_b200_ctx *ctx, uint64_t *mismatches);

/* ---- draw calls --------------------------------------------------------------------------- */
int dtr_b200_clear(dtr_b200_ctx *ctx, const float rgb[3]);
int dtr_b200_triangle(dtr_b200_ctx *ctx, const float p1[3], const float p2[3], const float p3[3],
                      const float color[4], const dtr_b200_transform *transform);
/* n triangles sharing one transform, submitted in order: p f32[n*9], color f32[n*4] */
int dtr_b200_triangles(dtr_b200_ctx *ctx, int n, const float *p, const float *color,
                       const dtr_b200_transform *transform);
int dtr_b200_textured_triangle(dtr_b200_ctx *ctx, const float p1[3], const float p2[3],
                               const float p3[3], const float uv1[2], const float uv2[2],
                               const float uv3[2], int texId /* <0: untextured */,
                               const float color[4], const dtr_b200_transform *transform);
int dtr_b200_mesh(dtr_b200_ctx *ctx, int meshId, const dtr_b200_light *light, const float pos[3],
                  const dtr_b200_transform *transform);
/* nViews DTRRender_Mesh calls, view i drawn into frame firstFrame + i (frame/viewpoint
 * parallel batch): pos f32[nViews*3], transforms[nViews]. */
int dtr_b200_mesh_views(dtr_b200_ctx *ctx, int meshId, const dtr_b200_light *light, int nViews,
                        const float *pos, const dtr_b200_transform *transforms, int firstFrame);
/* Draw calls whose arrays live in DEVICE memory of the context's device (device or managed allocations, e.g. torch
 * CUDA tensors): geometry made on the GPU is drawn without a round trip over the host link.
 *   dtr_b200_triangles_device   n triangles: p f32[n*9], color f32[n*4], uv f32[n*6] or NULL; texId < 0 or uv == NULL:
 *                               untextured.  Same meaning, transform handling, triangle ids and counters as
 *                               dtr_b200_triangles (and, when textured, dtr_b200_textured_triangle per triangle).
 *   dtr_b200_mesh_views_device  dtr_b200_mesh_views with per-view vertex sets: vertexes f32[nViews][numVertexes][4]
 *                               (w must be 1, as for dtr_b200_upload_mesh), normals f32[nViews][numNormals][3] or NULL
 *                               (the mesh's own normals); texUV, faces and texture come from the uploaded mesh.  View i
 *                               is mesh meshId with vertex set i, drawn into frame firstFrame + i.
 * Equivalence: drawing with these calls is bit for bit drawing the same values through dtr_b200_triangles /
 * dtr_b200_textured_triangle, or through dtr_b200_mesh_views on a mesh uploaded with those vertexes and normals --
 * colour, depth, ids, setPixels, triangles and the opaque stage that runs (dtr_b200_last_pass_deferred).  Only
 * uploadBytes differs: the arrays never cross the host link.
 * When the arrays are read: on the context's stream, by the flush that executes the call (any entry that flushes).
 * Whatever writes them must be ordered before that flush on that stream.  Once that flush returns the library no
 * longer reads them (a flush waits on the host for its list total): the caller may then free or overwrite them.
 * Replay: dtr_b200_replay renders what that flush read, from the library's own device snapshot; it never re-reads
 * the caller's arrays.
 * Errors: DTR_B200_ERR_ARG, with nothing recorded, for a pointer that cudaPointerGetAttributes does not report as
 * device or managed memory of the context's device (host memory, pinned or not, included), and for meshId, texId or
 * the frame range out of range.  n <= 0 or NULL p / color / vertexes (or light / pos / transforms) return
 * DTR_B200_OK without drawing.  The arrays need no particular alignment. */
int dtr_b200_triangles_device(dtr_b200_ctx *ctx, int n, const float *p, const float *color, const float *uv,
                              int texId, const dtr_b200_transform *transform);
int dtr_b200_mesh_views_device(dtr_b200_ctx *ctx, int meshId, const dtr_b200_light *light, int nViews,
                               const float *pos, const dtr_b200_transform *transforms, int firstFrame,
                               const float *vertexes, const float *normals);
int dtr_b200_rectangle(dtr_b200_ctx *ctx, const float min[2], const float max[2],
                       const float color[4], const dtr_b200_transform *transform);
int dtr_b200_bitmap(dtr_b200_ctx *ctx, int texId, const float pos[2],
                    const dtr_b200_transform *transform, const float color[4]);
int dtr_b200_line(dtr_b200_ctx *ctx, const int32_t a[2], const int32_t b[2], const float color[4]);
/* DTRRender_Text (DTRendererRender.h:91, DTRendererRender.cpp:193-273; SURVEY.md §8f rank 2).
 * A font is the reference's DTRFont flattened (DTRendererAsset.h:44-52): the 1-byte-per-pixel atlas
 * and one packed-char entry per codepoint of [codepointMin, codepointMax) -- dtr_b200_packedchar
 * has the layout of stbtt_packedchar (external/stb_truetype.h:522-527), i.e. DTRFont::atlas can be
 * passed as is.  dtr_b200_text lays the string out on the host exactly like the reference
 * (stbtt_GetPackedQuad with align_to_integer) and records one glyph primitive per character;
 * len == -1 means strlen(text).  Characters outside the font's range are an argument error (the
 * reference asserts). */
typedef struct dtr_b200_packedchar
{
	uint16_t x0, y0, x1, y1; /* glyph box in the atlas */
	float    xoff, yoff, xadvance, xoff2, yoff2;
} dtr_b200_packedchar;
int dtr_b200_upload_font(dtr_b200_ctx *ctx, const uint8_t *atlas, int atlasWidth, int atlasHeight,
                         const dtr_b200_packedchar *chars, int codepointMin, int codepointMax, int *fontId);
int dtr_b200_text(dtr_b200_ctx *ctx, int fontId, const float pos[2], const char *text, const float color[4], int len);
/* DTR_DEBUG_RENDER parity (SURVEY.md §8f rank 1): when enabled, dtr_b200_rectangle and
 * dtr_b200_bitmap also emit the overlay of the reference's DEFAULT build -- bounding-box lines,
 * the green outline of rotated rectangles, and for bitmaps the red bounding box plus a 10x10
 * rectangle per corner (DTRendererRender.cpp:492-512, 719-771, 1783-1790).  Off by default
 * (== the reference compiled with DTR_DEBUG_RENDER 0). */
int dtr_b200_set_debug_markers(dtr_b200_ctx *ctx, int enable);

#ifdef __cplusplus
}
#endif
#endif /* DTR_B200_H */
