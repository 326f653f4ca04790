// dtr_records.h -- POD records shared by the host recorder and the sm_100a kernels.
//
// Data layout in HBM (see DESIGN.md §3):
//   frames        colour u32[F][H][W] (0x00RRGGBB) and depth f32[F][H][W], row 0 = bottom --
//                 exactly DTRRenderBuffer's planes (DTRendererRender.h:14-25), one pair per frame;
//                 optionally triangle ids u32[F][H][W] (dtr_b200_set_id_output), same layout.
//   DrawItem[]    one per recorded draw call (tiny), uploaded per flush.
//   PrimRecord[]  one 160-byte record per primitive in submission order, written by the setup
//                 kernel, read by the raster kernel as ten 128-bit broadcast loads.
//   PrimBounds[]  8 bytes per primitive (pixel bbox, half open) -- what binning scans.
//   tile lists    u32 primitive indices per (frame, tile), ascending = submission order.
#pragma once
#include <stdint.h>

namespace dtr
{

// Screen tile = the unit of binning.  The raster kernel hands 32x32-pixel regions of a tile to
// single warps; a region is 32 sub-blocks of 8x4 pixels (one sub-block per lane when a triangle is
// classified against the region, one pixel per lane when a sub-block is rasterised).
constexpr int TILE_W      = 64;
constexpr int TILE_H      = 32; // the only height the round-2 raster kernel supports, see its static_assert
constexpr int REGION_W    = 32;
constexpr int REGION_H    = TILE_H;
constexpr int SUB_W       = 8;
constexpr int SUB_H       = 4;
// A raster CTA is four warps, each with its own region (see WarpSmem in dtr_kernels.cu); five CTAs per SM
constexpr int RASTER_THREADS = 128;
constexpr int RASTER_TAIL_PERCENT = 10; // share of the untouched tiles kept for the end of the launch
constexpr int RASTER_SMALL_PERCENT = 5; // share of the busy tiles rasterised as four 32x16 items
constexpr int RASTER_CTAS_PER_SM = 5; // 5 x 4 warps per SM, each warp with 10.4 KB of shared memory
// Frames with many primitives are binned in segments of BIN_SEG primitives: the setup kernel counts
// per (tile, segment), so that one CTA per (frame, tile row, segment) can write its part of every
// tile list independently and the lists still come out in submission order.
constexpr int BIN_SEG = 8192;

enum PrimType : uint32_t
{
	PRIM_TRI       = 0, // edge-function triangle (DTRendererRender.cpp:1071-1236)
	PRIM_RECT_FILL = 1, // axis-aligned rectangle fill (:472-483)
	PRIM_RECT_ROT  = 2, // rotated rectangle, 4-edge inside test (:442-471)
	PRIM_BITMAP    = 3, // bilinear bitmap blit (:1596-1791)
	PRIM_CLEAR     = 4, // colour-only clear (:1793-1815)
	PRIM_LINE      = 5, // integer DDA line (:294-356)
	PRIM_GLYPH     = 6, // one character of DTRRender_Text: 1-byte-per-pixel atlas x colour (:193-273)
};

enum PrimFlags : uint32_t
{
	PF_TYPE_MASK    = 0xF,
	PF_EXACT        = 1u << 4, // integer-valued edge setup: direct evaluation == sequential adds
	PF_IGNORE_LIGHT = 1u << 5,
	PF_TEXTURED     = 1u << 6,
	PF_GREY         = 1u << 7, // linear base colour has r == g == b (so have the three light products)
};

// 40 words = ten 128-bit quads.  Triangle layout: quads 0-3 are the GEOMETRY part (read once per
// (triangle, region) by one lane), quads 3-9 the SHADING part (copied verbatim into a shared-memory
// slot that the fragments of the triangle refer to).
enum TriWord
{
	TW_FLAGS = 0, TW_TEX = 1, TW_MIN = 2 /* minx | miny<<16 */, TW_MAX = 3 /* maxx | maxy<<16 */,
	TW_E0 = 4 /*3*/, TW_DX = 7 /*3*/, TW_DY = 10 /*3*/,
	TW_TEXELS = 13 /*2: device pointer*/, TW_TEXDIM = 15 /* w | h << 16 */,
	TW_INV_AREA = 16, TW_Z1 = 17, TW_DZ2 = 18, TW_DZ3 = 19,
	TW_COLOR = 20 /*4: linear premultiplied rgba*/,
	TW_LIGHT_R = 24 /*3: red light product of vertex 1,2,3*/, TW_FLAGS_TEX = 27 /* (flags & 0xFF) | texId << 8 */,
	TW_LIGHT_G = 28 /*3*/, TW_LIGHT_B = 31 /*3*/,
	TW_UV1 = 34 /*2*/, TW_DUV2X = 36, TW_DUV2Y = 37, TW_DUV3X = 38, TW_DUV3Y = 39,
};
constexpr int TRI_SHADE_QUAD0 = 3; // first quad of the shading part (quad 3 carries the texture)
constexpr int TRI_SHADE_QUADS = 7;
// Word indices of the quad layout (rectangle / bitmap / clear / line):
enum QuadWord
{
	QW_FLAGS = 0, QW_TEX = 1, QW_MIN = 2, QW_MAX = 3,
	QW_P = 4 /*8: Basis, XAxis, Point, YAxis (x,y)*/, QW_COLOR = 12 /*4*/, QW_INVX = 16, QW_INVY = 17,
	QW_TEXDIM = 18 /* w | h<<16 */, QW_PACKED = 19 /* PRIM_CLEAR: packed 0x00RRGGBB */,
	QW_LINE = 20 /*6: ax, ay, run, dist, delta, steep */,
	QW_GLYPH = 20 /*10: atlas lo, atlas hi, fontOffset, pitch, fontWidth, fontHeight, screen x (f32), screen y (f32),
	                    fontHeightOffset (f32), atlas size in bytes */,
};

struct alignas(16) PrimRecord
{
	uint32_t w[40];
};
static_assert(sizeof(PrimRecord) == 160, "PrimRecord must be ten 128-bit words");

struct PrimBounds
{
	uint32_t mn; // minx | miny << 16
	uint32_t mx; // maxx | maxy << 16 (exclusive); mx <= mn component-wise means "never binned"
};

enum ItemType : uint32_t
{
	ITEM_TRIS = 0, // count triangles from host arrays p/color(/uv)
	ITEM_MESH = 1, // count faces of an uploaded mesh through one host-built matrix
	ITEM_RAW  = 2, // count == 1: a PrimRecord computed on the host (rectangle, bitmap, clear, line)
};

struct alignas(16) DrawItem
{
	uint32_t type;
	uint32_t frame;
	uint32_t primBase; // global index of this item's first primitive
	uint32_t count;
	int32_t  texId; // < 0: untextured
	uint32_t lightMode;
	uint32_t triBase; // ITEM_TRIS / ITEM_MESH: position of the item's first triangle in its frame (triangle id planes)
	uint32_t pad1;
	// ITEM_TRIS: device pointers to p f32[count*9], color f32[count*4], uv f32[count*6] (or 0)
	// ITEM_MESH: vertexes, texUV, normals, faces
	// ITEM_RAW : record
	uint64_t ptr[4];
	float xAxis[2], yAxis[2]; // host cosf/sinf * scale (DTRendererRender.cpp:282-285)
	float anchor[2];
	float pad2[2];
	float m[16];              // ITEM_MESH: viewport*persp*view*model, e[col][row]
	float lightVec[3];
	float pad3;
	float color[4];
};
static_assert(sizeof(DrawItem) % 16 == 0, "DrawItem must stay 16-byte aligned");

struct TexDesc
{
	const uint32_t *texels;
	int32_t         w, h;
};

enum FrameInit : uint32_t
{
	FI_Z_RESET     = 1u << 0, // depth starts at -FLT_MAX, generated on chip (no read)
	FI_COLOR_CLEAR = 1u << 1, // colour starts at clearPacked, generated on chip (no read)
};

// The deferred opaque stage (dtr_deferred.cuh) tells a pixel whose shading is still pending from a finished
// one by bit 31 of its colour word: 0x80000000 | primitive index.  Shaded colours never have it (their top
// byte is 0).  A clear colour can: DTRRender_Clear packs (int32)(c * 255) with shifts, so a channel at or
// below -1/255 reaches bit 31, and so do some large ones (red 130; blue 1e10, +-inf or NaN).
// The host runs a pass whose frames clear to such a colour through the single raster kernel.
constexpr uint32_t VIS_PENDING = 0x80000000u;

struct FrameState
{
	uint32_t init;
	uint32_t clearPacked;
	uint32_t primBegin, primEnd; // this frame's contiguous primitive range in the flush
	uint32_t frameIndex;         // which colour/depth plane pair this active slot renders into
	uint32_t pad[3];
};

struct Geometry
{
	int32_t width, height;
	int32_t tilesX, tilesY;     // tiles over the whole frame
	int32_t bandTileY0, bandTileY1; // tile rows rasterised by this context
	int32_t bandTiles;          // tilesX * (bandTileY1 - bandTileY0)
	int32_t numFrames;          // ACTIVE frames of this flush (slots into FrameState[])
	int32_t segs;               // binning segments per frame (1: a frame's primitives are binned in one go)
	int32_t pad[3];
};

} // namespace dtr
