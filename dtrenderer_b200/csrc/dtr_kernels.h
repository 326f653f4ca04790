// dtr_kernels.h -- parameter blocks and launchers of the sm_100a kernels (dtr_kernels.cu).
#pragma once
#include <cuda_runtime_api.h>

#include "dtr_records.h"

namespace dtr
{

constexpr int SETUP_THREADS = 64; // 64 x 48 registers fit next to five resident raster CTAs: setup of the next replay runs DURING the raster kernel

struct SetupParams
{
	const DrawItem *items;
	const uint32_t *blockItem; // [ceil(numPrims / SETUP_THREADS)] item of each CTA's first primitive
	int             numItems;
	uint32_t        numPrims;
	PrimRecord     *prims;
	PrimBounds     *bounds;
	int32_t        *primZ;     // per primitive: depth_key of an upper bound of its depths (INT_MAX: unknown / not a depth-tested triangle)
	uint32_t       *segCount;  // [numFrames * bandTiles * segs] primitives per (tile, segment); == tile counts when segs == 1
	const FrameState *frames;
	const TexDesc  *textures; // texture table: pointer and size are copied into textured records
	Geometry        g;
	uint32_t       *primId;   // null, or per primitive: 1 + its triangle's position in its frame (0: not a triangle) -- the id planes' value
};

constexpr int SCAN_THREADS = 64;    // small CTAs (64 x 32 registers) fit next to five resident raster CTAs
constexpr int SCAN_CHUNK   = SCAN_THREADS * 4; // counts scanned per CTA

struct ScanParams
{
	const uint32_t     *counts;   // per-tile counts [n]
	uint32_t           *offsets;  // [n + 1]
	uint32_t            n;
	uint4              *order;    // [2n] raster work order (busy tiles first, untouched last), 32 bytes per tile:
	                              // {tile, list length, list offset, plane index} {clear colour, init flags, tx | ty << 16, -}
	const FrameState   *frames;
	uint32_t            bandTiles, tilesX, bandTileY0;
	unsigned long long *status;   // [chunks] look-back words, zeroed before the launch
	unsigned long long *totals;   // [0] list total
	uint32_t           *workCounter;
	uint32_t           *numBusy;  // number of tiles with primitives
};

// one look-back word per chunk plus one more: the ticket counter that hands out chunk ids
inline uint32_t scan_status_words(uint32_t n) { return (n + SCAN_CHUNK - 1) / SCAN_CHUNK + 1; }

// segs > 1 only: per tile, the exclusive prefix of its segment counts and their sum
struct TileSumParams
{
	const uint32_t *segCount;  // [numTiles * segs]
	uint32_t       *segRel;    // [numTiles * segs]
	uint32_t       *tileCount; // [numTiles]
	uint32_t        numTiles, segs;
};

struct BinParams
{
	const PrimBounds *bounds;
	const FrameState *frames;
	const uint32_t   *segCount;   // [numTiles * segs]
	const uint32_t   *segRel;     // [numTiles * segs] offset of a segment's entries inside its tile list (segs > 1)
	const uint32_t   *tileOffset; // [numTiles + 1]
	uint32_t         *lists;
	uint2            *listBounds; // [listCapacity] bbox of every list entry, same positions
	const int32_t    *primZ;      // per primitive depth bound (see SetupParams)
	int32_t          *listZ;      // [listCapacity] ... and its depth bound
	uint32_t          listCapacity;
	int32_t           groupRows; // tile rows per CTA, filled by launch_bin
	Geometry          g;
};

struct RasterParams
{
	uint32_t           *color; // [F][H][W]
	float              *depth;
	uint32_t           *tagColor; // two-kernel deferred stage: where the visibility kernel leaves the colour tiles of busy tiles (pending
	                              // tags included) for the resolve kernel -- the context's OWN colour planes; == color unless
	                              // the output planes are foreign (another GPU's memory)
	const FrameState   *frames;
	const PrimRecord   *prims;
	const PrimBounds   *bounds;
	const uint32_t     *tileCount;
	const uint32_t     *tileOffset;
	const uint4        *order; // work order + tile descriptors written by scan_kernel
	const uint32_t     *lists;
	const uint2        *listBounds;
	const int32_t      *listZ;
	const TexDesc      *textures;
	unsigned long long *setPixels;
	uint32_t           *workCounter;    // zeroed by scan_kernel; items handed out by atomicAdd
	const uint32_t     *numBusy;        // written by scan_kernel
	const unsigned long long *listTotal; // (primitive, tile) pairs of the pass, written by scan_kernel
	uint32_t           *zeroBase;       // counters + look-back words to clear for the next pass (may be null)
	size_t              zeroWords;
	uint32_t            anyTextured;    // some primitive of this pass samples a texture: raster_tex_kernel
	uint32_t            numTiles;       // filled by launch_raster
	uint32_t            smallTilesMin;  // filled by launch_raster: busy tiles rasterised as fine-grained items
	Geometry            g;
	// Triangle id planes (appended: the fields above keep their offsets).  ids == null: off, and the kernels
	// without id logic run; otherwise the IDS variants keep ids[F][H][W] next to the depth plane (every depth
	// write also stores primId[] of the triangle that wrote it; a depth reset stores 0)
	uint32_t           *ids;
	const uint32_t     *primId;
};

// Per-device launch limits, queried once per context (dtr_b200_create) on ITS device: a process may
// hold contexts on several GPUs.
struct LaunchLimits
{
	int sms          = 148;
	int residentCtas = 148; // raster CTAs resident on the whole device (sms x CTAs per SM)
	int residentCtasVis = 148; // ... of the deferred pass's visibility kernel
	int residentCtasVisRes = 148; // ... of the one-kernel form of the deferred pass (raster_visres_kernel)
	// ... of the id-plane variants of the three (more shared memory per CTA: fewer of them per SM)
	int residentCtasIds = 148, residentCtasVisIds = 148, residentCtasVisResIds = 148;
};
LaunchLimits query_launch_limits(int device);
void         launch_init_tables(cudaStream_t s); // per-device lookup tables of the raster kernel (once per context)

// DTRMesh's per-face index arrays (DTRendererAsset.h:16-26) flattened on the device: faces[] holds
// HOST pointers into the arena block, which was uploaded as one copy (see dtr_b200_upload_mesh_faces).
struct FlattenParams
{
	const uint8_t *faces;      // device copy of DTRMeshFace[numFaces] (48 bytes each)
	const uint8_t *arena;      // device copy of the host arena block
	uint64_t       hostArena;  // host address of the block
	uint64_t       arenaBytes;
	uint32_t       numFaces, numVertexes, numTexUV, numNormals;
	int32_t       *out;        // i32[numFaces][9]
	uint32_t      *error;      // != 0: some face was malformed
};
void launch_flatten_faces(const FlattenParams &P, cudaStream_t s);

struct ResolveParams
{
	uint32_t         *color;   // [F][H][W]: the output colour planes
	const uint32_t   *tags;    // [F][H][W]: finished colours and pending primitive tags of the busy tiles (== color, or the
	                           // context's own planes when the output planes are foreign: every pixel of a busy tile is
	                           // then stored to `color`, pending or not)
	const PrimRecord *prims;
	const uint4      *order;   // tile descriptors in work order: the busy tiles are the first *numBusy
	const uint32_t   *numBusy;
	uint32_t          numTiles; // tiles of the pass (busy + untouched).  Not read by resolve_kernel; it keeps g.width at
	                            // 4 mod 8 bytes, where the kernel loads it with the instruction schedule that was measured
	Geometry          g;
};

void launch_setup(const SetupParams &P, cudaStream_t s);
// Scans the tile counts (-> totals[0]); the offsets array gets one extra trailing entry holding the
// total.  Also zeroes the raster work counter and writes the work order.
void launch_scan(const ScanParams &P, cudaStream_t s);
void launch_tile_sum(const TileSumParams &P, cudaStream_t s);
void launch_selftest_sqrt(unsigned long long *mismatches, cudaStream_t s);
void launch_bin(const BinParams &P, const LaunchLimits &L, cudaStream_t s);
void launch_raster(const RasterParams &P, const LaunchLimits &L, cudaStream_t s);
// the deferred variant of the raster stage (dtr_deferred.cuh): oneKernel = raster_opaque_kernel<true> (visibility with the
// resolve done in place, region by region), else raster_opaque_kernel<false> (visibility) + resolve_kernel.
// `between` (may be null) is called after the first kernel has been launched: the profiling event
void launch_raster_deferred(const RasterParams &P, const LaunchLimits &L, cudaStream_t s, bool oneKernel, void (*between)(void *, cudaStream_t) = nullptr,
                            void *betweenArg = nullptr);
void launch_premultiply(uint32_t *pixels, size_t count, cudaStream_t s);
void launch_pack_bgr24(const uint32_t *color, uint32_t *out, int width, size_t rows, int pitchWords, cudaStream_t s);

// Readback resolve of n frames at factor k (2..4, dividing width and height): resolve_frames_kernel<k, ...>
struct FrameResolveParams
{
	const uint32_t *color; // sample planes [frames][height][width] (read where the matching output is wanted)
	const float    *depth; // read when outDepth or outIds is wanted
	const uint32_t *ids;   // read when outIds is wanted
	uint32_t       *outColor; // [frames][height/k][width/k], each may be null
	float          *outDepth;
	uint32_t       *outIds;
	int             width, height, frames;
};
void launch_resolve_frames(const FrameResolveParams &P, int k, cudaStream_t s);
// resolve_pack_bgr24_kernel<k, ...>: the colour of outRows output rows resolved and packed as launch_pack_bgr24 packs
void launch_resolve_pack_bgr24(const uint32_t *color, uint32_t *out, int width, int k, size_t outRows, int pitchWords, cudaStream_t s);

// Render to texture of n frames at factor k (1..4, dividing width and height): frames_to_textures_kernel<k, ...>
struct FrameTextureParams
{
	const uint32_t *color;    // colour planes [frames][height][width]
	const int32_t  *texIds;   // [frames] destination texture of each frame, (width/k) x (height/k), no two equal
	const TexDesc  *textures; // the context's texture table
	int             width, height, frames;
};
void launch_frames_to_textures(const FrameTextureParams &P, int k, cudaStream_t s);

// Snapshot of the device-resident draw-call inputs of a flush (gather_device_inputs_kernel): segment i copies
// `bytes` (a multiple of 4) from src to dst (16-byte aligned) and covers chunks [firstChunk, next firstChunk) of
// gather_chunks(bytes) each.  color: the segment is f32[n][4] colours whose alphas are checked.
constexpr int      GATHER_THREADS = 256;
constexpr uint32_t GATHER_CHUNK   = GATHER_THREADS * 64; // bytes of one segment a CTA copies per step
struct GatherSegment
{
	uint64_t src, dst, bytes;
	uint32_t firstChunk, color;
};
inline uint32_t gather_chunks(uint64_t bytes) { return (uint32_t)((bytes + GATHER_CHUNK - 1) / GATHER_CHUNK); }
struct GatherParams
{
	const GatherSegment *segs; // [numSegs], firstChunk ascending
	uint32_t             numSegs, numChunks;
	unsigned long long  *translucent; // set to 1 when some colour alpha is not 1.0f; zeroed by the host
};
void launch_gather_device_inputs(const GatherParams &P, const LaunchLimits &L, cudaStream_t s);

} // namespace dtr
