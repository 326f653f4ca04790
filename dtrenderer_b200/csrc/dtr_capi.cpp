// dtr_capi.cpp -- implementation of the C ABI in include/dtr_b200.h.
//
// Host side of the back end: records draw calls, evaluates the once-per-call host arithmetic
// (dtr_host_math.h), uploads one command block per flush and launches
//     setup_kernel -> (tile_sum_kernel) -> scan_kernel -> bin_rows_kernel -> raster_kernel
// on the context's stream.  There is no CPU rendering path in this file: if CUDA is not
// available dtr_b200_create fails.  Compiled with -ffp-contract=off.
#include <cuda_runtime_api.h>

#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/dtr_b200.h"
#include "dtr_host_math.h"
#include "dtr_kernels.h"
#include "dtr_nccl.h"
#include "dtr_records.h"

using namespace dtr;

namespace
{

std::string g_createError;

struct DevBuf
{
	void  *p   = nullptr;
	size_t cap = 0;
};

struct MeshAsset
{
	float   *vertexes = nullptr, *texUV = nullptr, *normals = nullptr;
	int32_t *faces    = nullptr;
	uint32_t numFaces = 0, numVertexes = 0, numNormals = 0;
	int      texId    = -1;
};

struct RecItem
{
	DrawItem item;
	uint32_t frame;      // real frame index
	uint32_t order;      // submission order (stable sort key)
	size_t   payload[3]; // byte offsets into the payload buffer (valid where relocate[j])
	bool     relocate[3];
	size_t   snap[3];    // byte offsets into the device snapshot buffer (valid where fromSnap[j]): ptr[j] read from device memory
	bool     fromSnap[3];
	bool     opaque;     // triangles whose every fragment has alpha 1 (colour alpha 1, no texture or an opaque one)
};

struct FrameHost
{
	uint32_t pendingInit = 0; // FrameInit bits to apply at the next flush
	uint32_t clearPacked = 0;
	uint32_t recorded    = 0; // items recorded for this frame since the last flush
	uint32_t triangles   = 0; // triangles submitted since the frame's last dtr_b200_begin_frame: the next one's id is this + 1
};

} // namespace

struct dtr_b200_ctx
{
	int          device = 0, width = 0, height = 0, numFrames = 0;
	cudaStream_t stream = nullptr, ownStream = nullptr;
	// asynchronous readback (dtr_b200_read_frames_async): a copy stream ordered after the rendering
	// by renderDone; copyDone lets a later flush that renders into frames still being read wait
	cudaStream_t copyStream = nullptr;
	cudaEvent_t  renderDone = nullptr, copyDone = nullptr;
	// 24-bit presentation readback (dtr_b200_read_frames_bgr24_async) and resolved readbacks: two device
	// staging buffers used in turn, so that packing the next batch does not wait for the previous transfer
	DevBuf       packStage[2];
	cudaEvent_t  packFree[2] = {nullptr, nullptr}; // the D2H copy out of packStage[k] has finished
	int          packTurn    = 0;
	int          readLo = 0, readHi = 0; // frames [readLo, readHi) have reads in flight
	int          resolve = 1; // readback resolve factor k (dtr_b200_set_readback_resolve)
	struct FontHost
	{
		uint8_t                         *dAtlas = nullptr;
		int                              w = 0, h = 0, cpMin = 0, cpMax = 0;
		std::vector<dtr_b200_packedchar> chars;
	};
	std::vector<FontHost> fonts;
	bool         debugMarkers = false;  // emit the reference's DTR_DEBUG_RENDER overlay (dtr_b200_set_debug_markers)
	uint32_t    *dColor = nullptr; // this context's own frame planes
	float       *dDepth = nullptr;
	// where the frames are rendered: the own planes, or planes of a peer GPU (sort-first bands that
	// write straight into the gathering rank's frames over NVLink, dtr_b200_open_peer_frames)
	uint32_t    *outColor = nullptr;
	float       *outDepth = nullptr;
	uint32_t    *dIds = nullptr; // triangle id planes u32[F][H][W] (dtr_b200_set_id_output), always this context's own; null: off
	void        *ipcColor = nullptr, *ipcDepth = nullptr; // mappings opened from IPC handles
	Geometry     geom{};
	int          target = 0;
	LaunchLimits limits{}; // this context's device: SM count and resident raster CTAs (queried at create)
	int          opaqueStage = DTR_B200_OPAQUE_ONE_KERNEL; // how a pass of opaque triangles onto cleared frames runs (dtr_b200_set_opaque_stage)
	// sort-first band exchange behind the C ABI (dtr_b200_band_comm_init / _attach)
	NcclComm     comm = nullptr;
	bool         ownComm = false;
	int          commRanks = 0, commRank = -1;
	float       *dToken = nullptr; // the barrier's 4-byte all-reduce buffer

	std::vector<FrameHost> frames;
	std::vector<RecItem>   rec;
	uint8_t               *payload = nullptr; // pinned
	size_t                 payloadCap = 0, payloadUsed = 0;
	uint8_t               *staging = nullptr; // pinned: FrameState[] + DrawItem[]
	size_t                 stagingCap = 0;
	// arrays of draw calls recorded from device memory (dtr_b200_triangles_device / _mesh_views_device): where they
	// are, and where the flush's snapshot of them goes in dSnap (16-byte aligned offsets, like the payload's)
	struct DeviceArray
	{
		const void *src;
		size_t      at, bytes;
		bool        color; // f32[n][4] triangle colours: their alphas decide the opaque stage on the device
	};
	std::vector<DeviceArray> devArrays;
	size_t                   snapUsed = 0;

	std::vector<MeshAsset> meshes;
	std::vector<TexDesc>   textures;
	std::vector<uint8_t>   texIsWhite; // every texel 0xFFFFFFFF: sampling multiplies by exactly 1.0f
	std::vector<uint8_t>   texIsOpaque; // every texel has alpha 255: a textured fragment keeps its colour's alpha
	DevBuf                 dTextures;
	DevBuf                 dTexIds; // the texIds of the last dtr_b200_frames_to_textures, read by its kernel

	DevBuf dCmd, dPayload;
	DevBuf dSnap; // the last flush's snapshot of its device arrays (replays render from it)
	// Intermediate buffers of one pass of the pipeline.  PIPE_SETS sets: a flush uses set 0; replays
	// take them in turn, so that setup / scan / bin of a later replay (on preStream) run while the
	// raster kernels of earlier replays occupy the main stream.  With THREE sets the pre-raster stages
	// run two replays ahead: setup and scan of replay i+2 (small CTAs) co-run with raster i, bin i+2
	// takes the SM slots that free up at the end of raster i and runs beside the START of raster i+1,
	// which depends only on bin i+1 (long finished) and therefore launches back to back with raster i.
	// (With two sets raster i+1 had to wait for bin i+1, which could not start before raster i ended.)
	struct PipeSet
	{
		DevBuf              prims, bounds, primZ, tileCount, tileOffset, order, lists, listBounds, listZ, segRel;
		DevBuf              primId; // ids on: per primitive, its triangle id (setup_kernel)
		unsigned long long *counters = nullptr; // [1] list total, [3] work counter, [4] busy tiles
		cudaEvent_t         preDone = nullptr, rasterDone = nullptr;
		bool                rasterPending = false; // rasterDone has been recorded: the set may still be read
		size_t              cleanBytes = 0;        // the first cleanBytes of tileCount were zeroed by the last raster kernel
	};
	static constexpr int PIPE_SETS = 3;
	PipeSet             sets[PIPE_SETS];
	int                 nextReplaySet = 1;
	bool                replayOverlap = true; // dtr_b200_set_replay_overlap
	cudaStream_t        preStream = nullptr;
	unsigned long long *dSetPixels = nullptr; // [0] SetPixel count of every raster launch so far
	uint64_t            triangles = 0, launches = 0, uploadBytes = 0;
	bool                     profiling = false;
	std::vector<cudaEvent_t> events;     // EVENTS_PER_RUN per profiled pipeline
	std::vector<cudaEvent_t> eventPool;  // recycled

	// last flush, for replay
	struct
	{
		bool     valid = false;
		uint32_t numActive = 0, numItems = 0, numPrims = 0, maxFramePrims = 0;
		uint64_t listTotal = 0, triangles = 0;
		bool     anyTextured = false; // some triangle item of the flush samples a (non-white) texture
		bool     deferred    = false; // every primitive an opaque triangle, every frame cleared on chip: visibility + resolve
		bool     oneKernel   = false; // ... as ONE kernel (the resolve done in place, region by region)
		Geometry g{};
	} last;

	std::string err;
};

namespace
{

int fail(dtr_b200_ctx *c, int code, const char *what, cudaError_t e = cudaSuccess)
{
	char buf[512];
	if (e != cudaSuccess) snprintf(buf, sizeof(buf), "%s: %s", what, cudaGetErrorString(e));
	else snprintf(buf, sizeof(buf), "%s", what);
	if (c) c->err = buf;
	else g_createError = buf;
	return code;
}

#define CU(call)                                                              \
	do                                                                        \
	{                                                                         \
		cudaError_t e_ = (call);                                              \
		if (e_ != cudaSuccess) return fail(c, DTR_B200_ERR_CUDA, #call, e_);  \
	} while (0)

int ensure_dev(dtr_b200_ctx *c, DevBuf &b, size_t bytes)
{
	if (bytes <= b.cap) return 0;
	size_t want = std::max(bytes, b.cap + b.cap / 2);
	want        = (want + 255) & ~(size_t)255;
	// buffers may still be in use by enqueued work
	CU(cudaStreamSynchronize(c->stream));
	if (b.p) CU(cudaFree(b.p));
	b.p   = nullptr;
	b.cap = 0;
	CU(cudaMalloc(&b.p, want));
	b.cap = want;
	return 0;
}

int ensure_pinned(dtr_b200_ctx *c, uint8_t *&p, size_t &cap, size_t used, size_t bytes)
{
	if (bytes <= cap) return 0;
	size_t   want = std::max(bytes, cap * 2);
	want          = std::max<size_t>(want, 1 << 16);
	uint8_t *n    = nullptr;
	CU(cudaHostAlloc((void **)&n, want, cudaHostAllocDefault));
	if (p)
	{
		if (used) memcpy(n, p, used);
		cudaFreeHost(p);
	}
	p   = n;
	cap = want;
	return 0;
}

// append `bytes` to the pinned payload, 16-byte aligned; returns the byte offset
int payload_push(dtr_b200_ctx *c, const void *src, size_t bytes, size_t *off)
{
	size_t at = (c->payloadUsed + 15) & ~(size_t)15;
	int    rc = ensure_pinned(c, c->payload, c->payloadCap, c->payloadUsed, at + bytes);
	if (rc) return rc;
	memcpy(c->payload + at, src, bytes);
	c->payloadUsed = at + bytes;
	*off           = at;
	return 0;
}

void set_geometry(dtr_b200_ctx *c, int y0, int y1)
{
	Geometry &g  = c->geom;
	g.width      = c->width;
	g.height     = c->height;
	g.tilesX     = (c->width + TILE_W - 1) / TILE_W;
	g.tilesY     = (c->height + TILE_H - 1) / TILE_H;
	g.bandTileY0 = y0 / TILE_H;
	g.bandTileY1 = (y1 + TILE_H - 1) / TILE_H;
	g.bandTiles  = g.tilesX * (g.bandTileY1 - g.bandTileY0);
	g.numFrames  = 0;
}

const dtr_b200_transform kDefaultTransform         = {0.0f, {0.5f, 0.5f, 0.5f}, {1.0f, 1.0f, 1.0f}};
const dtr_b200_transform kDefaultTriangleTransform = {0.0f, {0.33f, 0.33f, 0.33f}, {1.0f, 1.0f, 1.0f}};

RecItem &new_item(dtr_b200_ctx *c, uint32_t type, uint32_t frame, uint32_t count)
{
	c->rec.emplace_back();
	RecItem &r = c->rec.back();
	memset(&r, 0, sizeof(r));
	r.item.type  = type;
	r.item.count = count;
	r.item.texId = -1;
	r.frame      = frame;
	r.order      = (uint32_t)c->rec.size() - 1;
	c->frames[frame].recorded++;
	if (type != ITEM_RAW)
	{
		// triangles are numbered per frame in submission order, across flushes (triangle id planes)
		r.item.triBase = c->frames[frame].triangles;
		c->frames[frame].triangles += count;
	}
	return r;
}

int record_raw(dtr_b200_ctx *c, const PrimRecord &rec)
{
	size_t off;
	int    rc = payload_push(c, &rec, sizeof(rec), &off);
	if (rc) return rc;
	RecItem &r    = new_item(c, ITEM_RAW, (uint32_t)c->target, 1);
	r.payload[0]  = off;
	r.relocate[0] = true;
	return 0;
}

// An ITEM_TRIS item of n triangles on the current target; the caller says where its arrays are.  opaque: the
// texture's part of the decision (the caller adds the colours')
RecItem &new_tris_item(dtr_b200_ctx *c, int n, int texId, const dtr_b200_transform *t)
{
	if (!t) t = &kDefaultTriangleTransform;
	RecItem &r       = new_item(c, ITEM_TRIS, (uint32_t)c->target, (uint32_t)n);
	r.item.texId     = (texId >= 0 && c->texIsWhite[texId]) ? -1 : texId;
	r.opaque         = r.item.texId < 0 || c->texIsOpaque[r.item.texId];
	r.item.lightMode = DTR_B200_SHADE_FULLBRIGHT; // NullRenderLightInternal (:1352-1356)
	Basis2 b         = make_basis(t->rotation, t->scale[0], t->scale[1]);
	r.item.xAxis[0] = b.xAxis[0]; r.item.xAxis[1] = b.xAxis[1];
	r.item.yAxis[0] = b.yAxis[0]; r.item.yAxis[1] = b.yAxis[1];
	r.item.anchor[0] = t->anchor[0];
	r.item.anchor[1] = t->anchor[1];
	c->triangles += (uint64_t)n;
	return r;
}

int record_tris(dtr_b200_ctx *c, int n, const float *p, const float *color, const float *uv, int texId,
                const dtr_b200_transform *t)
{
	size_t offP, offC, offUV = 0;
	int    rc;
	if ((rc = payload_push(c, p, sizeof(float) * 9 * (size_t)n, &offP))) return rc;
	if ((rc = payload_push(c, color, sizeof(float) * 4 * (size_t)n, &offC))) return rc;
	if (uv && (rc = payload_push(c, uv, sizeof(float) * 6 * (size_t)n, &offUV))) return rc;
	RecItem &r    = new_tris_item(c, n, texId, t);
	r.payload[0]  = offP;
	r.relocate[0] = true;
	r.payload[1]  = offC;
	r.relocate[1] = true;
	r.payload[2]  = offUV;
	r.relocate[2] = (uv != nullptr);
	for (int i = 0; i < n && r.opaque; i++) r.opaque = color[4 * (size_t)i + 3] == 1.0f;
	return 0;
}

// Reserves `bytes` of the flush's device snapshot for the device array src (16-byte aligned); returns the offset.
// Nothing is read here: the flush gathers every such array with one kernel.
size_t snap_push(dtr_b200_ctx *c, const void *src, size_t bytes, bool color)
{
	const size_t at = (c->snapUsed + 15) & ~(size_t)15;
	c->devArrays.push_back({src, at, bytes, color});
	c->snapUsed = at + bytes;
	return at;
}

// p / color / uv of dtr_b200_triangles_device are device memory of the context's device (device or managed)
bool on_ctx_device(const dtr_b200_ctx *c, const void *p)
{
	cudaPointerAttributes a{};
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess)
	{
		cudaGetLastError(); // (not sticky: clear it)
		return false;
	}
	return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == c->device;
}

constexpr int EVENTS_PER_RUN = 7; // pre start, after setup, after scan, after bin | raster start, after the stage's first kernel, raster end

int mark(dtr_b200_ctx *c, cudaStream_t stream)
{
	if (!c->profiling || c->events.size() >= (size_t)EVENTS_PER_RUN * 8192) return 0;
	cudaEvent_t e;
	if (!c->eventPool.empty())
	{
		e = c->eventPool.back();
		c->eventPool.pop_back();
	}
	else CU(cudaEventCreate(&e));
	CU(cudaEventRecord(e, stream));
	c->events.push_back(e);
	return 0;
}

int run_pipeline(dtr_b200_ctx *c, uint32_t numActive, uint32_t numItems, uint32_t numPrims, uint32_t maxFramePrims,
                 bool replay)
{
	Geometry g   = c->geom;
	g.numFrames  = (int32_t)numActive;
	g.segs       = (int32_t)std::max<uint32_t>(1u, (maxFramePrims + BIN_SEG - 1) / BIN_SEG);
	g.pad[0] = g.pad[1] = g.pad[2] = 0;
	const uint32_t numTiles = numActive * (uint32_t)g.bandTiles;
	const size_t   numSeg   = (size_t)numTiles * (size_t)g.segs; // (tile, segment) counters
	if (numSeg >= (1ull << 31)) return fail(c, DTR_B200_ERR_OVERFLOW, "more than 2^31 (tile, segment) counters in one flush");
	const FrameState *dFrames = (const FrameState *)c->dCmd.p;
	const DrawItem   *dItems  = (const DrawItem *)((const uint8_t *)c->dCmd.p + sizeof(FrameState) * numActive);
	const uint32_t   *dBlockItem = (const uint32_t *)(dItems + numItems);

	// A flush runs everything on the main stream with buffer set 0 (it has to wait for the list
	// total on the host anyway).  A replay takes the other set in turn and runs setup / scan / bin on
	// preStream: they only touch the set's buffers, so they may overlap the previous raster kernel,
	// whose tail leaves SMs idle; the raster kernels themselves stay ordered on the main stream.
	const bool             overlap = replay && c->replayOverlap;
	dtr_b200_ctx::PipeSet &S   = c->sets[overlap ? c->nextReplaySet : 0];
	const cudaStream_t     pre = overlap ? c->preStream : c->stream;
	if (overlap) c->nextReplaySet = (c->nextReplaySet + 1) % dtr_b200_ctx::PIPE_SETS;
	else if (replay) CU(cudaStreamSynchronize(c->preStream)); // set 0 may be in use by an overlapped replay
	if (S.rasterPending && pre != c->stream) CU(cudaStreamWaitEvent(pre, S.rasterDone, 0));

	int rc;
	// one buffer, one memset: (tile, segment) counts | per-tile counts (segs > 1 only) | look-back words
	const size_t tileWords   = g.segs > 1 ? (size_t)numTiles : 0;
	const size_t countWords  = (numSeg + tileWords + 1) & ~(size_t)1; // keep the 64-bit words aligned
	const size_t statusWords = scan_status_words(numTiles);
	{
		const void *before = S.tileCount.p;
		if ((rc = ensure_dev(c, S.tileCount, sizeof(uint32_t) * countWords + sizeof(unsigned long long) * statusWords))) return rc;
		if (S.tileCount.p != before) S.cleanBytes = 0; // a new allocation has not been cleared by anyone
	}
	if ((rc = ensure_dev(c, S.order, 32 * std::max<size_t>(numTiles, 1)))) return rc;
	if ((rc = ensure_dev(c, S.tileOffset, sizeof(uint32_t) * ((size_t)numTiles + 1)))) return rc;
	if ((rc = ensure_dev(c, S.segRel, sizeof(uint32_t) * std::max<size_t>(g.segs > 1 ? numSeg : 1, 1)))) return rc;
	if ((rc = ensure_dev(c, S.prims, sizeof(PrimRecord) * (size_t)std::max(numPrims, 1u)))) return rc;
	if ((rc = ensure_dev(c, S.bounds, sizeof(PrimBounds) * (size_t)std::max(numPrims, 1u)))) return rc;
	if ((rc = ensure_dev(c, S.primZ, sizeof(int32_t) * (size_t)std::max(numPrims, 1u)))) return rc;
	if (c->dIds && (rc = ensure_dev(c, S.primId, sizeof(uint32_t) * (size_t)std::max(numPrims, 1u)))) return rc;
	uint32_t *dSegCount  = (uint32_t *)S.tileCount.p;
	uint32_t *dTileCount = g.segs > 1 ? dSegCount + numSeg : dSegCount; // with one segment they are the same thing

	unsigned long long *dScanStatus = (unsigned long long *)(dSegCount + countWords);
	if ((rc = mark(c, pre))) return rc;
	const size_t zeroBytes = sizeof(uint32_t) * countWords + sizeof(unsigned long long) * statusWords;
	// a replay finds the counters already cleared by the previous raster kernel of this set
	if (!(replay && S.cleanBytes >= zeroBytes)) CU(cudaMemsetAsync(dSegCount, 0, zeroBytes, pre));
	S.cleanBytes = 0;
	if (numPrims)
	{
		SetupParams SP;
		SP.items       = dItems;
		SP.blockItem   = dBlockItem;
		SP.numItems    = (int)numItems;
		SP.numPrims    = numPrims;
		SP.prims       = (PrimRecord *)S.prims.p;
		SP.bounds      = (PrimBounds *)S.bounds.p;
		SP.primZ       = (int32_t *)S.primZ.p;
		SP.segCount    = dSegCount;
		SP.frames      = dFrames;
		SP.textures    = (const TexDesc *)c->dTextures.p;
		SP.g           = g;
		SP.primId      = c->dIds ? (uint32_t *)S.primId.p : nullptr;
		launch_setup(SP, pre);
		c->launches++;
	}
	if ((rc = mark(c, pre))) return rc;
	if (g.segs > 1)
	{
		TileSumParams TS;
		TS.segCount  = dSegCount;
		TS.segRel    = (uint32_t *)S.segRel.p;
		TS.tileCount = dTileCount;
		TS.numTiles  = numTiles;
		TS.segs      = (uint32_t)g.segs;
		launch_tile_sum(TS, pre);
		c->launches++;
	}
	ScanParams SC;
	SC.counts      = dTileCount;
	SC.offsets     = (uint32_t *)S.tileOffset.p;
	SC.n           = numTiles;
	SC.order       = (uint4 *)S.order.p;
	SC.frames      = dFrames;
	SC.bandTiles   = (uint32_t)g.bandTiles;
	SC.tilesX      = (uint32_t)g.tilesX;
	SC.bandTileY0  = (uint32_t)g.bandTileY0;
	SC.status      = dScanStatus;
	SC.totals      = S.counters + 1;
	SC.workCounter = (uint32_t *)(S.counters + 3);
	SC.numBusy     = (uint32_t *)(S.counters + 4);
	launch_scan(SC, pre);
	c->launches++;
	if ((rc = mark(c, pre))) return rc;

	uint64_t total = c->last.listTotal;
	if (!replay)
	{
		// with device arrays, the gather kernel's translucent flag (counters[2]) comes back with the list total
		unsigned long long t[2] = {0, 0};
		const bool gathered = !c->devArrays.empty();
		CU(cudaMemcpyAsync(t, S.counters + 1, sizeof(t[0]) * (gathered ? 2 : 1), cudaMemcpyDeviceToHost, pre));
		CU(cudaStreamSynchronize(pre));
		total = t[0];
		if (total >= (1ull << 31)) return fail(c, DTR_B200_ERR_OVERFLOW, "more than 2^31 (primitive, tile) pairs in one flush");
		if (t[1]) c->last.deferred = c->last.oneKernel = false; // some device colour has alpha != 1: the pass can blend
	}
	if ((rc = ensure_dev(c, S.lists, sizeof(uint32_t) * (size_t)std::max<uint64_t>(total, 1)))) return rc;
	if ((rc = ensure_dev(c, S.listBounds, 2 * sizeof(uint32_t) * (size_t)std::max<uint64_t>(total, 1)))) return rc;
	if ((rc = ensure_dev(c, S.listZ, sizeof(int32_t) * (size_t)std::max<uint64_t>(total, 1)))) return rc;

	if (numPrims && total)
	{
		BinParams B;
		B.bounds       = (const PrimBounds *)S.bounds.p;
		B.frames       = dFrames;
		B.segCount     = dSegCount;
		B.segRel       = (const uint32_t *)S.segRel.p;
		B.tileOffset   = (const uint32_t *)S.tileOffset.p;
		B.lists        = (uint32_t *)S.lists.p;
		B.listBounds   = (uint2 *)S.listBounds.p;
		B.primZ        = (const int32_t *)S.primZ.p;
		B.listZ        = (int32_t *)S.listZ.p;
		B.listCapacity = (uint32_t)std::min({S.lists.cap / sizeof(uint32_t), S.listBounds.cap / (2 * sizeof(uint32_t)), S.listZ.cap / sizeof(int32_t)});
		B.groupRows    = 0;
		B.g            = g;
		launch_bin(B, c->limits, pre);
		c->launches++;
	}
	if ((rc = mark(c, pre))) return rc;
	if (pre != c->stream)
	{
		CU(cudaEventRecord(S.preDone, pre));
		CU(cudaStreamWaitEvent(c->stream, S.preDone, 0));
	}

	RasterParams R;
	R.color      = c->outColor;
	R.depth      = c->outDepth;
	R.tagColor   = c->dColor;
	R.frames     = dFrames;
	R.prims      = (const PrimRecord *)S.prims.p;
	R.bounds     = (const PrimBounds *)S.bounds.p;
	R.tileCount  = dTileCount;
	R.tileOffset = (const uint32_t *)S.tileOffset.p;
	R.order      = (const uint4 *)S.order.p;
	R.lists      = (const uint32_t *)S.lists.p;
	R.listBounds = (const uint2 *)S.listBounds.p;
	R.listZ      = (const int32_t *)S.listZ.p;
	R.textures   = (const TexDesc *)c->dTextures.p;
	R.setPixels  = c->dSetPixels;
	R.workCounter    = (uint32_t *)(S.counters + 3);
	R.numBusy        = (const uint32_t *)(S.counters + 4);
	R.listTotal      = S.counters + 1;
	R.zeroBase       = dSegCount;
	R.zeroWords      = zeroBytes / sizeof(uint32_t);
	R.anyTextured    = c->last.anyTextured ? 1u : 0u;
	R.numTiles       = 0;
	R.smallTilesMin  = 0;
	R.g          = g;
	R.ids        = c->dIds; // the IDS variants of the stage's kernels, or (null) the ones without id logic
	R.primId     = c->dIds ? (const uint32_t *)S.primId.p : nullptr;
	if ((rc = mark(c, c->stream))) return rc;
	if (c->last.deferred)
	{
		// (profiling: the event between the visibility and the resolve kernel)
		launch_raster_deferred(R, c->limits, c->stream, c->last.oneKernel, [](void *ctx, cudaStream_t s2) { mark(static_cast<dtr_b200_ctx *>(ctx), s2); }, c);
		c->launches += c->last.oneKernel ? 1 : 2;
	}
	else
	{
		launch_raster(R, c->limits, c->stream);
		c->launches++;
		if ((rc = mark(c, c->stream))) return rc; // (a single kernel: the stage's first kernel is all of it)
	}
	if ((rc = mark(c, c->stream))) return rc;
	CU(cudaEventRecord(S.rasterDone, c->stream));
	S.rasterPending = true;
	S.cleanBytes    = zeroBytes;
	CU(cudaGetLastError());

	c->last.valid     = true;
	c->last.numActive = numActive;
	c->last.numItems  = numItems;
	c->last.numPrims  = numPrims;
	c->last.listTotal = total;
	c->last.maxFramePrims = maxFramePrims;
	c->last.g         = g;
	return 0;
}

int do_flush(dtr_b200_ctx *c)
{
	// active frames: anything with recorded items or a pending on-chip init
	std::vector<int32_t> slotOf(c->numFrames, -1);
	std::vector<uint32_t> active;
	for (int f = 0; f < c->numFrames; f++)
		if (c->frames[f].recorded || c->frames[f].pendingInit)
		{
			slotOf[f] = (int32_t)active.size();
			active.push_back((uint32_t)f);
		}
	if (active.empty()) return 0;
	// replays may still be running their pre-raster stages on preStream; a flush rewrites the
	// command block they read
	CU(cudaStreamSynchronize(c->preStream));
	CU(cudaStreamSynchronize(c->stream));
	if (c->readHi > c->readLo)
	{
		// a frame that is still being read back must not be overwritten
		bool overlap = false;
		for (uint32_t f : active) overlap = overlap || ((int)f >= c->readLo && (int)f < c->readHi);
		if (overlap) CU(cudaStreamWaitEvent(c->stream, c->copyDone, 0));
	}

	// frames are independent, so grouping items by frame (stable) preserves every frame's order
	std::stable_sort(c->rec.begin(), c->rec.end(),
	                 [](const RecItem &a, const RecItem &b) { return a.frame < b.frame; });

	uint32_t numActive = (uint32_t)active.size(), numItems = (uint32_t)c->rec.size();
	// command block: FrameState[numActive] | DrawItem[numItems] | item of every setup CTA's first primitive
	uint64_t totalPrims = 0;
	for (const RecItem &r : c->rec) totalPrims += r.item.count;
	if (totalPrims >= (1ull << 31)) return fail(c, DTR_B200_ERR_OVERFLOW, "more than 2^31 primitives in one flush");
	const size_t numBlocks = (size_t)((totalPrims + SETUP_THREADS - 1) / SETUP_THREADS);
	size_t   cmdBytes  = sizeof(FrameState) * numActive + sizeof(DrawItem) * numItems + sizeof(uint32_t) * numBlocks;
	// ... | the gather kernel's segment table, one per device array (only when there are any)
	const size_t numSegs  = c->devArrays.size();
	const size_t segsAt   = (cmdBytes + 15) & ~(size_t)15;
	if (numSegs) cmdBytes = segsAt + sizeof(GatherSegment) * numSegs;
	int      rc;
	if ((rc = ensure_pinned(c, c->staging, c->stagingCap, 0, cmdBytes))) return rc;
	if ((rc = ensure_dev(c, c->dCmd, cmdBytes))) return rc;
	if ((rc = ensure_dev(c, c->dPayload, std::max<size_t>(c->payloadUsed, 16)))) return rc;
	if (numSegs && (rc = ensure_dev(c, c->dSnap, c->snapUsed))) return rc;

	FrameState *fs = (FrameState *)c->staging;
	DrawItem   *it = (DrawItem *)(c->staging + sizeof(FrameState) * numActive);
	for (uint32_t s = 0; s < numActive; s++)
	{
		FrameHost &fh     = c->frames[active[s]];
		fs[s].init        = fh.pendingInit;
		fs[s].clearPacked = fh.clearPacked;
		fs[s].primBegin = fs[s].primEnd = 0;
		fs[s].frameIndex = active[s];
		fs[s].pad[0] = fs[s].pad[1] = fs[s].pad[2] = 0;
	}
	uint64_t prim = 0;
	int32_t  cur  = -1;
	for (uint32_t i = 0; i < numItems; i++)
	{
		RecItem &r    = c->rec[i];
		int32_t  slot = slotOf[r.frame];
		if (slot != cur)
		{
			if (cur >= 0) fs[cur].primEnd = (uint32_t)prim;
			fs[slot].primBegin = (uint32_t)prim;
			cur                = slot;
		}
		r.item.frame    = (uint32_t)slot;
		r.item.primBase = (uint32_t)prim;
		for (int j = 0; j < 3; j++)
		{
			if (r.relocate[j]) r.item.ptr[j] = (uint64_t)((uint8_t *)c->dPayload.p + r.payload[j]);
			if (r.fromSnap[j]) r.item.ptr[j] = (uint64_t)((uint8_t *)c->dSnap.p + r.snap[j]);
		}
		it[i] = r.item;
		prim += r.item.count;
		if (prim >= (1ull << 31)) return fail(c, DTR_B200_ERR_OVERFLOW, "more than 2^31 primitives in one flush");
	}
	if (cur >= 0) fs[cur].primEnd = (uint32_t)prim;
	{
		uint32_t *blockItem = (uint32_t *)(it + numItems);
		uint32_t  cursor    = 0;
		for (size_t b = 0; b < numBlocks; b++)
		{
			const uint64_t first = (uint64_t)b * SETUP_THREADS;
			while (cursor + 1 < numItems && it[cursor + 1].primBase <= first) cursor++;
			blockItem[b] = cursor;
		}
	}
	// slots with no items keep primBegin == primEnd
	for (uint32_t s = 0; s < numActive; s++)
		if (c->frames[active[s]].recorded == 0) fs[s].primBegin = fs[s].primEnd = 0;

	GatherParams gather{};
	if (numSegs)
	{
		GatherSegment *seg   = (GatherSegment *)(c->staging + segsAt);
		uint64_t       chunk = 0;
		for (size_t s = 0; s < numSegs; s++)
		{
			const dtr_b200_ctx::DeviceArray &a = c->devArrays[s];
			seg[s] = GatherSegment{(uint64_t)(uintptr_t)a.src, (uint64_t)((uint8_t *)c->dSnap.p + a.at), (uint64_t)a.bytes, (uint32_t)chunk, a.color ? 1u : 0u};
			chunk += gather_chunks(a.bytes);
		}
		if (chunk >= (1ull << 32)) return fail(c, DTR_B200_ERR_OVERFLOW, "more than 2^32 gather chunks of device arrays in one flush");
		gather.segs        = (const GatherSegment *)((uint8_t *)c->dCmd.p + segsAt);
		gather.numSegs     = (uint32_t)numSegs;
		gather.numChunks   = (uint32_t)chunk;
		gather.translucent = c->sets[0].counters + 2; // read back with the list total (run_pipeline)
	}
	c->uploadBytes = cmdBytes + c->payloadUsed;
	CU(cudaMemcpyAsync(c->dCmd.p, c->staging, cmdBytes, cudaMemcpyHostToDevice, c->stream));
	if (c->payloadUsed)
		CU(cudaMemcpyAsync(c->dPayload.p, c->payload, c->payloadUsed, cudaMemcpyHostToDevice, c->stream));
	if (numSegs)
	{
		// the snapshot the pipeline (and every replay of this flush) reads instead of the callers' arrays; like the
		// readback resolve kernels it is not counted in kernelLaunches
		CU(cudaMemsetAsync(gather.translucent, 0, sizeof(unsigned long long), c->stream));
		launch_gather_device_inputs(gather, c->limits, c->stream);
		CU(cudaGetLastError());
	}

	c->last.anyTextured = false;
	for (uint32_t i = 0; i < numItems; i++) c->last.anyTextured = c->last.anyTextured || (it[i].type != ITEM_RAW && it[i].texId >= 0);
	// Deferred pass (dtr_deferred.cuh): only when nothing can ever be blended -- every primitive an opaque
	// triangle, every frame starting from an on-chip clear.  (With foreign output planes -- a band written
	// into another GPU's frame -- the one-kernel form stores finished regions straight to the output; in
	// the two-kernel form the visibility kernel leaves its tags in this context's own colour planes and
	// the resolve kernel stores every pixel of the busy tiles to the output.  Nothing is ever read back
	// over NVLink.)  A clear colour with bit 31 set would read as a pending tag at the pixels no triangle
	// covers (VIS_PENDING): such a pass takes the single kernel, which gives the same frames.
	{
		bool deferred = c->opaqueStage != DTR_B200_OPAQUE_SINGLE_KERNEL && numItems > 0;
		for (uint32_t s2 = 0; s2 < numActive && deferred; s2++)
			deferred = (fs[s2].init & FI_COLOR_CLEAR) != 0 && (fs[s2].clearPacked & VIS_PENDING) == 0;
		for (uint32_t i = 0; i < numItems && deferred; i++) deferred = c->rec[i].item.type != ITEM_RAW && c->rec[i].opaque;
		c->last.deferred  = deferred;
		c->last.oneKernel = deferred && c->opaqueStage == DTR_B200_OPAQUE_ONE_KERNEL;
	}
	uint32_t maxFramePrims = 0;
	for (uint32_t s2 = 0; s2 < numActive; s2++) maxFramePrims = std::max(maxFramePrims, fs[s2].primEnd - fs[s2].primBegin);
	rc = run_pipeline(c, numActive, numItems, (uint32_t)prim, maxFramePrims, false);
	// the host copies were consumed (run_pipeline synchronises before binning)
	for (uint32_t s = 0; s < numActive; s++)
	{
		FrameHost &fh  = c->frames[active[s]];
		fh.pendingInit = 0;
		fh.recorded    = 0;
	}
	c->rec.clear();
	c->payloadUsed = 0;
	c->devArrays.clear();
	c->snapUsed = 0;
	return rc;
}

bool valid_frame(const dtr_b200_ctx *c, int f) { return f >= 0 && f < c->numFrames; }

} // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char *dtr_b200_version(void) { return "dtr_b200 0.1 (sm_100a)"; }

const char *dtr_b200_last_error(const dtr_b200_ctx *ctx) { return ctx ? ctx->err.c_str() : g_createError.c_str(); }

int dtr_b200_create(int device, int width, int height, int numFrames, dtr_b200_ctx **out)
{
	dtr_b200_ctx *c = nullptr; // for CU(): errors land in g_createError
	if (!out) return fail(nullptr, DTR_B200_ERR_ARG, "out is NULL");
	*out = nullptr;
	if (width <= 0 || height <= 0 || width > 16384 || height > 16384 || numFrames <= 0)
		return fail(nullptr, DTR_B200_ERR_ARG, "width/height must be in [1,16384] and numFrames >= 1");
	int count = 0;
	CU(cudaGetDeviceCount(&count));
	if (device < 0 || device >= count) return fail(nullptr, DTR_B200_ERR_CUDA, "no such CUDA device (this back end has no CPU fallback)");
	CU(cudaSetDevice(device));
	dtr_b200_ctx *n = new (std::nothrow) dtr_b200_ctx();
	if (!n) return fail(nullptr, DTR_B200_ERR_NOMEM, "out of host memory");
	n->device    = device;
	n->width     = width;
	n->height    = height;
	n->numFrames = numFrames;
	n->frames.resize(numFrames);
	size_t plane = (size_t)width * height;
	cudaError_t e;
	if ((e = cudaStreamCreateWithFlags(&n->ownStream, cudaStreamNonBlocking)) != cudaSuccess ||
	    (e = cudaStreamCreateWithFlags(&n->copyStream, cudaStreamNonBlocking)) != cudaSuccess ||
	    (e = cudaEventCreateWithFlags(&n->renderDone, cudaEventDisableTiming)) != cudaSuccess ||
	    (e = cudaEventCreateWithFlags(&n->copyDone, cudaEventDisableTiming)) != cudaSuccess ||
	    (e = cudaMalloc((void **)&n->dColor, plane * numFrames * sizeof(uint32_t))) != cudaSuccess ||
	    (e = cudaMalloc((void **)&n->dDepth, plane * numFrames * sizeof(float))) != cudaSuccess ||
	    (e = cudaStreamCreateWithFlags(&n->preStream, cudaStreamNonBlocking)) != cudaSuccess ||
	    (e = cudaMalloc((void **)&n->dSetPixels, 8 * sizeof(unsigned long long))) != cudaSuccess ||
	    (e = cudaMemset(n->dColor, 0, plane * numFrames * sizeof(uint32_t))) != cudaSuccess ||
	    (e = cudaMemset(n->dSetPixels, 0, 8 * sizeof(unsigned long long))) != cudaSuccess)
	{
		fail(nullptr, DTR_B200_ERR_CUDA, "allocating frame targets", e);
		dtr_b200_destroy(n);
		return DTR_B200_ERR_CUDA;
	}
	for (auto &ps : n->sets)
	{
		if ((e = cudaMalloc((void **)&ps.counters, 8 * sizeof(unsigned long long))) != cudaSuccess ||
		    (e = cudaMemset(ps.counters, 0, 8 * sizeof(unsigned long long))) != cudaSuccess ||
		    (e = cudaEventCreateWithFlags(&ps.preDone, cudaEventDisableTiming)) != cudaSuccess ||
		    (e = cudaEventCreateWithFlags(&ps.rasterDone, cudaEventDisableTiming)) != cudaSuccess)
		{
			fail(nullptr, DTR_B200_ERR_CUDA, "allocating pipeline state", e);
			dtr_b200_destroy(n);
			return DTR_B200_ERR_CUDA;
		}
	}
	n->limits = query_launch_limits(device);
	// process-wide defaults from the environment (A/B runs): DTR_B200_DEFER=0 -> always the single raster kernel,
	// DTR_B200_FUSED=0 -> opaque passes as visibility + resolve (two kernels)
	if (const char *e = getenv("DTR_B200_FUSED"))
		if (e[0] == '0') n->opaqueStage = DTR_B200_OPAQUE_TWO_KERNELS;
	if (const char *e = getenv("DTR_B200_DEFER"))
		if (e[0] == '0') n->opaqueStage = DTR_B200_OPAQUE_SINGLE_KERNEL;
	launch_init_tables(n->ownStream);
	n->stream = n->ownStream;
	n->outColor = n->dColor;
	n->outDepth = n->dDepth;
	set_geometry(n, 0, height);
	// a frame that was never begun starts like the reference's first frame: depth reset
	for (auto &f : n->frames) f.pendingInit = FI_Z_RESET;
	*out = n;
	return DTR_B200_OK;
}

void dtr_b200_destroy(dtr_b200_ctx *c)
{
	if (!c) return;
	cudaSetDevice(c->device);
	if (c->stream) cudaStreamSynchronize(c->stream);
	for (auto &m : c->meshes)
	{
		cudaFree(m.vertexes);
		cudaFree(m.texUV);
		cudaFree(m.normals);
		cudaFree(m.faces);
	}
	for (auto &t : c->textures) cudaFree((void *)t.texels);
	for (auto &f : c->fonts) cudaFree(f.dAtlas);
	if (c->preStream) cudaStreamSynchronize(c->preStream);
	std::vector<DevBuf *> bufs = {&c->dTextures, &c->dTexIds, &c->dCmd, &c->dPayload, &c->dSnap};
	for (auto &ps : c->sets)
	{
		for (DevBuf *b : {&ps.prims, &ps.bounds, &ps.primZ, &ps.tileCount, &ps.tileOffset, &ps.order, &ps.lists, &ps.listBounds, &ps.listZ, &ps.segRel, &ps.primId}) bufs.push_back(b);
		cudaFree(ps.counters);
		if (ps.preDone) cudaEventDestroy(ps.preDone);
		if (ps.rasterDone) cudaEventDestroy(ps.rasterDone);
	}
	for (DevBuf *b : bufs) cudaFree(b->p);
	if (c->comm && c->ownComm && nccl_api().ok) nccl_api().CommDestroy(c->comm);
	cudaFree(c->dToken);
	if (c->ipcColor) cudaIpcCloseMemHandle(c->ipcColor);
	if (c->ipcDepth) cudaIpcCloseMemHandle(c->ipcDepth);
	cudaFree(c->dColor);
	cudaFree(c->dDepth);
	cudaFree(c->dIds);
	cudaFree(c->dSetPixels);
	if (c->payload) cudaFreeHost(c->payload);
	if (c->staging) cudaFreeHost(c->staging);
	for (cudaEvent_t e : c->events) cudaEventDestroy(e);
	for (cudaEvent_t e : c->eventPool) cudaEventDestroy(e);
	if (c->copyStream)
	{
		cudaStreamSynchronize(c->copyStream);
		cudaStreamDestroy(c->copyStream);
	}
	if (c->renderDone) cudaEventDestroy(c->renderDone);
	if (c->copyDone) cudaEventDestroy(c->copyDone);
	for (int k = 0; k < 2; k++)
	{
		cudaFree(c->packStage[k].p);
		if (c->packFree[k]) cudaEventDestroy(c->packFree[k]);
	}
	if (c->preStream) cudaStreamDestroy(c->preStream);
	if (c->ownStream) cudaStreamDestroy(c->ownStream);
	delete c;
}

int dtr_b200_set_stream(dtr_b200_ctx *c, void *cudaStream)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	CU(cudaStreamSynchronize(c->stream));
	c->stream = cudaStream ? (cudaStream_t)cudaStream : c->ownStream;
	return DTR_B200_OK;
}

int dtr_b200_set_band(dtr_b200_ctx *c, int y0, int y1)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (y0 < 0 || y1 > c->height || y0 >= y1 || (y0 % TILE_H) != 0 || ((y1 % TILE_H) != 0 && y1 != c->height))
	{
		char msg[128];
		snprintf(msg, sizeof(msg), "band must be tile aligned (multiples of %d rows, or end at height)", TILE_H);
		return fail(c, DTR_B200_ERR_ARG, msg);
	}
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	set_geometry(c, y0, y1);
	c->last.valid = false;
	return DTR_B200_OK;
}

namespace
{
// The nearest-texel fetch clamps u, v to [0, 1] and indexes (int)(v*h) * w + (int)(u*w) like the reference
// (DTRendererRender.cpp:1196-1203): v == 1 lands on row h, u == 1 in the last row one texel past it.  The
// reference reads whatever follows its bitmap there; every texture allocation carries one spare row plus one
// texel so that the same read stays inside it (in-range results are unaffected).  After a texture with any alpha
// below 255 the spare texels are zeros (transparent).  After an opaque one they are opaque white: a pass of
// opaque triangles takes the deferred raster stage, which shades a visible fragment with alpha 1 and never
// blends it, so every texel the fetch can read must be opaque for that pass to equal the single kernel; white
// is also what an all-white texture implies, whose fetch is skipped.
int write_texture_padding(dtr_b200_ctx *c, const TexDesc &td, bool opaque)
{
	const size_t               padBytes = ((size_t)td.w + 1) * 4;
	const std::vector<uint8_t> pad(padBytes, opaque ? 0xFF : 0x00);
	CU(cudaMemcpy(const_cast<uint32_t *>(td.texels) + (size_t)td.w * td.h, pad.data(), padBytes, cudaMemcpyHostToDevice));
	return 0;
}

// Copies the texture table, with the texture just appended, to the device; *texId: the new texture's id
int publish_new_texture(dtr_b200_ctx *c, int *texId)
{
	CU(cudaStreamSynchronize(c->stream)); // the old table may be in use
	int rc = ensure_dev(c, c->dTextures, sizeof(TexDesc) * std::max<size_t>(c->textures.capacity(), 16));
	if (rc) return rc;
	CU(cudaMemcpy(c->dTextures.p, c->textures.data(), sizeof(TexDesc) * c->textures.size(), cudaMemcpyHostToDevice));
	*texId = (int)c->textures.size() - 1;
	return DTR_B200_OK;
}
} // namespace

int dtr_b200_upload_texture(dtr_b200_ctx *c, const uint8_t *texels, int width, int height, int bytesPerPixel, int *texId)
{
	if (!c || !texId) return DTR_B200_ERR_ARG;
	if (!texels || width <= 0 || height <= 0 || width > 32767 || height > 32767 || bytesPerPixel != 4)
		return fail(c, DTR_B200_ERR_ARG, "texture must be non-NULL RGBA8 with dimensions in [1,32767]");
	CU(cudaSetDevice(c->device));
	uint32_t *d     = nullptr;
	size_t    bytes = (size_t)width * height * 4;
	const size_t padBytes = ((size_t)width + 1) * 4; // the spare texels: see write_texture_padding
	CU(cudaMalloc((void **)&d, bytes + padBytes));
	CU(cudaMemcpy(d, texels, bytes, cudaMemcpyHostToDevice));
	c->textures.push_back(TexDesc{d, width, height});
	{
		// 255 * (1/255.0f) == 1.0f and 1.0f^2 == 1.0f in fp32, so an all-white opaque texture leaves
		// every channel bit-identical: triangles using it skip the fetch (DTRRender_Mesh always
		// samples mesh->tex, so "untextured" meshes carry exactly such a 1x1 texture)
		bool           white = true;
		const uint32_t *t32  = reinterpret_cast<const uint32_t *>(texels);
		if (((uintptr_t)texels & 3) == 0)
		{
			for (size_t i = 0; i < (size_t)width * height && white; i++) white = (t32[i] == 0xFFFFFFFFu);
		}
		else
		{
			for (size_t i = 0; i < bytes && white; i++) white = (texels[i] == 0xFF);
		}
		c->texIsWhite.push_back(white ? 1 : 0);
		bool opaque = true;
		for (size_t i = 3; i < bytes && opaque; i += 4) opaque = (texels[i] == 0xFF);
		c->texIsOpaque.push_back(opaque ? 1 : 0);
		int rc = write_texture_padding(c, c->textures.back(), opaque);
		if (rc) return rc;
	}
	return publish_new_texture(c, texId);
}

int dtr_b200_create_texture(dtr_b200_ctx *c, int width, int height, int *texId)
{
	if (!c || !texId) return DTR_B200_ERR_ARG;
	if (width <= 0 || height <= 0 || width > 32767 || height > 32767) return fail(c, DTR_B200_ERR_ARG, "texture dimensions must be in [1,32767]");
	CU(cudaSetDevice(c->device));
	uint32_t    *d     = nullptr;
	const size_t bytes = ((size_t)width * height + width + 1) * 4; // texels and the spare texels (write_texture_padding)
	CU(cudaMalloc((void **)&d, bytes));
	// all-zero texels: what dtr_b200_upload_texture makes of them (neither white nor opaque, zero spare texels)
	CU(cudaMemsetAsync(d, 0, bytes, c->stream));
	c->textures.push_back(TexDesc{d, width, height});
	c->texIsWhite.push_back(0);
	c->texIsOpaque.push_back(0);
	return publish_new_texture(c, texId);
}

int dtr_b200_update_texture(dtr_b200_ctx *c, int texId, const uint8_t *texels)
{
	if (!c || !texels) return DTR_B200_ERR_ARG;
	if (texId < 0 || texId >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c); // draw calls recorded so far sample the old contents
	if (rc) return rc;
	CU(cudaStreamSynchronize(c->preStream));
	CU(cudaStreamSynchronize(c->stream));
	const TexDesc &td    = c->textures[texId];
	const size_t   count = (size_t)td.w * td.h;
	CU(cudaMemcpy(const_cast<uint32_t *>(td.texels), texels, count * 4, cudaMemcpyHostToDevice));
	bool white = true;
	for (size_t i = 0; i < count * 4 && white; i++) white = (texels[i] == 0xFF);
	c->texIsWhite[texId] = white ? 1 : 0;
	bool opaque = true;
	for (size_t i = 3; i < count * 4 && opaque; i += 4) opaque = (texels[i] == 0xFF);
	c->texIsOpaque[texId] = opaque ? 1 : 0;
	c->last.valid        = false; // a replay would keep the old "textured" decision
	if ((rc = write_texture_padding(c, td, opaque))) return rc;
	return DTR_B200_OK;
}

int dtr_b200_upload_bitmap_straight(dtr_b200_ctx *c, const uint8_t *rgba, int width, int height, int *texId)
{
	// upload the straight-alpha texels, then run DTRAsset_LoadBitmap's premultiply pass on the device
	int rc = dtr_b200_upload_texture(c, rgba, width, height, 4, texId);
	if (rc) return rc;
	launch_premultiply(const_cast<uint32_t *>(c->textures[*texId].texels), (size_t)width * height, c->stream);
	CU(cudaGetLastError());
	CU(cudaStreamSynchronize(c->stream));
	return DTR_B200_OK;
}

int dtr_b200_read_texture(dtr_b200_ctx *c, int texId, uint8_t *rgba)
{
	if (!c || !rgba) return DTR_B200_ERR_ARG;
	if (texId < 0 || texId >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream)); // dtr_b200_frames_to_textures writes texels in stream order
	const TexDesc &td = c->textures[texId];
	CU(cudaMemcpy(rgba, td.texels, (size_t)td.w * td.h * 4, cudaMemcpyDeviceToHost));
	return DTR_B200_OK;
}

int dtr_b200_frames_to_textures(dtr_b200_ctx *c, int first, int n, const int *texIds)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!texIds || n < 1 || !valid_frame(c, first) || !valid_frame(c, first + n - 1)) return fail(c, DTR_B200_ERR_ARG, "frame range out of bounds");
	if (c->outColor != c->dColor)
		return fail(c, DTR_B200_ERR_ARG, "foreign output planes are set: this context's colour planes do not hold the frames");
	const int            ow = c->width / c->resolve, oh = c->height / c->resolve;
	std::vector<uint8_t> taken(c->textures.size(), 0);
	for (int i = 0; i < n; i++)
	{
		const int t = texIds[i];
		if (t < 0 || t >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
		if (c->textures[t].w != ow || c->textures[t].h != oh)
			return fail(c, DTR_B200_ERR_ARG, "texture size is not the frame size over the readback resolve factor");
		if (taken[t]++) return fail(c, DTR_B200_ERR_ARG, "the same texId twice in one call");
	}
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c); // draw calls recorded so far are converted, and sample the old texels
	if (rc) return rc;
	if ((rc = ensure_dev(c, c->dTexIds, sizeof(int32_t) * n))) return rc;
	CU(cudaMemcpyAsync(c->dTexIds.p, texIds, sizeof(int32_t) * n, cudaMemcpyHostToDevice, c->stream));
	FrameTextureParams P{};
	P.color    = c->dColor + (size_t)c->width * c->height * first;
	P.texIds   = (const int32_t *)c->dTexIds.p;
	P.textures = (const TexDesc *)c->dTextures.p;
	P.width    = c->width;
	P.height   = c->height;
	P.frames   = n;
	launch_frames_to_textures(P, c->resolve, c->stream);
	CU(cudaGetLastError());
	// the decisions draw calls take when they are recorded
	for (int i = 0; i < n; i++)
	{
		c->texIsWhite[texIds[i]]  = 0;
		c->texIsOpaque[texIds[i]] = 1;
	}
	c->last.valid = false; // a replay would keep the old decisions
	return DTR_B200_OK;
}

namespace
{
// vertexes / texUV / normals of a DTRMesh, as they are (DTRendererAsset.h:27-41)
int upload_mesh_arrays(dtr_b200_ctx *c, MeshAsset &a, const float *vertexes, uint32_t nV, const float *texUV, uint32_t nT,
                       const float *normals, uint32_t nN)
{
	CU(cudaMalloc((void **)&a.vertexes, sizeof(float) * 4 * nV));
	CU(cudaMalloc((void **)&a.texUV, sizeof(float) * 3 * nT));
	CU(cudaMalloc((void **)&a.normals, sizeof(float) * 3 * nN));
	CU(cudaMemcpy(a.vertexes, vertexes, sizeof(float) * 4 * nV, cudaMemcpyHostToDevice));
	CU(cudaMemcpy(a.texUV, texUV, sizeof(float) * 3 * nT, cudaMemcpyHostToDevice));
	CU(cudaMemcpy(a.normals, normals, sizeof(float) * 3 * nN, cudaMemcpyHostToDevice));
	return 0;
}
void free_mesh(MeshAsset &a)
{
	cudaFree(a.vertexes);
	cudaFree(a.texUV);
	cudaFree(a.normals);
	cudaFree(a.faces);
	a = MeshAsset();
}
} // namespace

int dtr_b200_upload_mesh(dtr_b200_ctx *c, const dtr_b200_mesh_desc *m, int texId, int *meshId)
{
	if (!c || !meshId) return DTR_B200_ERR_ARG;
	if (!m || !m->vertexes || !m->texUV || !m->normals || !m->faces || !m->numFaces)
		return fail(c, DTR_B200_ERR_ARG, "mesh needs vertexes, texUV, normals and faces");
	if (texId >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
	// the reference asserts on out-of-range indices (DTRendererRender.cpp:1450-1502)
	for (size_t i = 0; i < (size_t)m->numFaces * 9; i++)
	{
		int32_t  idx = m->faces[i];
		uint32_t lim = (i % 9 < 3) ? m->numVertexes : ((i % 9 < 6) ? m->numTexUV : m->numNormals);
		if (idx < 0 || (uint32_t)idx >= lim) return fail(c, DTR_B200_ERR_ARG, "face index out of range");
	}
	CU(cudaSetDevice(c->device));
	MeshAsset a;
	a.numFaces    = m->numFaces;
	a.numVertexes = m->numVertexes;
	a.numNormals  = m->numNormals;
	a.texId       = texId;
	int rc = upload_mesh_arrays(c, a, m->vertexes, m->numVertexes, m->texUV, m->numTexUV, m->normals, m->numNormals);
	if (rc)
	{
		free_mesh(a);
		return rc;
	}
	CU(cudaMalloc((void **)&a.faces, sizeof(int32_t) * 9 * m->numFaces));
	CU(cudaMemcpy(a.faces, m->faces, sizeof(int32_t) * 9 * m->numFaces, cudaMemcpyHostToDevice));
	c->meshes.push_back(a);
	*meshId = (int)c->meshes.size() - 1;
	return DTR_B200_OK;
}

int dtr_b200_upload_mesh_faces(dtr_b200_ctx *c, const dtr_b200_mesh_faces_desc *m, int texId, int *meshId)
{
	static_assert(sizeof(dtr_b200_mesh_face) == 48, "dtr_b200_mesh_face must mirror DTRMeshFace");
	if (!c || !meshId) return DTR_B200_ERR_ARG;
	if (!m || !m->vertexes || !m->texUV || !m->normals || !m->faces || !m->numFaces || !m->arena || !m->arenaBytes)
		return fail(c, DTR_B200_ERR_ARG, "mesh needs vertexes, texUV, normals, faces and the arena block of the index arrays");
	if (texId >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
	CU(cudaSetDevice(c->device));
	MeshAsset a;
	a.numFaces    = m->numFaces;
	a.numVertexes = m->numVertexes;
	a.numNormals  = m->numNormals;
	a.texId       = texId;
	int rc = upload_mesh_arrays(c, a, m->vertexes, m->numVertexes, m->texUV, m->numTexUV, m->normals, m->numNormals);
	uint8_t  *dFaces = nullptr, *dArena = nullptr;
	uint32_t *dErr = nullptr, err = 0;
	cudaError_t e = cudaSuccess;
	if (!rc && ((e = cudaMalloc((void **)&a.faces, sizeof(int32_t) * 9 * m->numFaces)) != cudaSuccess ||
	            (e = cudaMalloc((void **)&dFaces, sizeof(dtr_b200_mesh_face) * (size_t)m->numFaces)) != cudaSuccess ||
	            (e = cudaMalloc((void **)&dArena, m->arenaBytes)) != cudaSuccess ||
	            (e = cudaMalloc((void **)&dErr, sizeof(uint32_t))) != cudaSuccess ||
	            (e = cudaMemsetAsync(dErr, 0, sizeof(uint32_t), c->stream)) != cudaSuccess ||
	            // one copy each: the DTRMeshFace array and the block its pointers lead into
	            (e = cudaMemcpyAsync(dFaces, m->faces, sizeof(dtr_b200_mesh_face) * (size_t)m->numFaces, cudaMemcpyHostToDevice, c->stream)) != cudaSuccess ||
	            (e = cudaMemcpyAsync(dArena, m->arena, m->arenaBytes, cudaMemcpyHostToDevice, c->stream)) != cudaSuccess))
		rc = fail(c, DTR_B200_ERR_CUDA, "uploading the mesh's face arrays", e);
	if (!rc)
	{
		FlattenParams F;
		F.faces       = dFaces;
		F.arena       = dArena;
		F.hostArena   = (uint64_t)(uintptr_t)m->arena;
		F.arenaBytes  = (uint64_t)m->arenaBytes;
		F.numFaces    = m->numFaces;
		F.numVertexes = m->numVertexes;
		F.numTexUV    = m->numTexUV;
		F.numNormals  = m->numNormals;
		F.out         = a.faces;
		F.error       = dErr;
		launch_flatten_faces(F, c->stream);
		c->launches++;
		if ((e = cudaGetLastError()) != cudaSuccess ||
		    (e = cudaMemcpyAsync(&err, dErr, sizeof(err), cudaMemcpyDeviceToHost, c->stream)) != cudaSuccess ||
		    (e = cudaStreamSynchronize(c->stream)) != cudaSuccess)
			rc = fail(c, DTR_B200_ERR_CUDA, "flattening the mesh's face arrays", e);
		else if (err)
			rc = fail(c, DTR_B200_ERR_ARG, "malformed face: index arrays outside the arena, counts not 3 / >=3 / 3, or an index out of range");
	}
	cudaFree(dFaces);
	cudaFree(dArena);
	cudaFree(dErr);
	if (rc)
	{
		free_mesh(a);
		return rc;
	}
	c->meshes.push_back(a);
	*meshId = (int)c->meshes.size() - 1;
	return DTR_B200_OK;
}

int dtr_b200_set_target(dtr_b200_ctx *c, int frame)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!valid_frame(c, frame)) return fail(c, DTR_B200_ERR_ARG, "frame out of range");
	c->target = frame;
	return DTR_B200_OK;
}

int dtr_b200_begin_frame(dtr_b200_ctx *c, int frame, const uint32_t *hostColor, const float *hostZ)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!valid_frame(c, frame)) return fail(c, DTR_B200_ERR_ARG, "frame out of range");
	CU(cudaSetDevice(c->device));
	if (c->frames[frame].recorded)
	{
		int rc = do_flush(c);
		if (rc) return rc;
	}
	size_t     plane = (size_t)c->width * c->height;
	FrameHost &fh    = c->frames[frame];
	// a dtr_b200_clear recorded as the frame's on-chip colour init stays pending (the reference's
	// Clear writes the colour buffer, the frame start only resets depth) unless colour is uploaded now
	fh.pendingInit &= FI_COLOR_CLEAR;
	fh.triangles = 0;
	// an asynchronous readback of this frame may still be in flight on the copy stream
	if ((hostZ || hostColor) && frame >= c->readLo && frame < c->readHi) CU(cudaStreamWaitEvent(c->stream, c->copyDone, 0));
	if (hostZ)
	{
		CU(cudaMemcpyAsync(c->outDepth + plane * frame, hostZ, plane * sizeof(float), cudaMemcpyHostToDevice, c->stream));
		// uploaded depth was written by no triangle of this frame (a reset depth zeroes the ids on chip, with FI_Z_RESET)
		if (c->dIds) CU(cudaMemsetAsync(c->dIds + plane * frame, 0, plane * sizeof(uint32_t), c->stream));
	}
	else fh.pendingInit |= FI_Z_RESET;
	if (hostColor)
	{
		fh.pendingInit &= ~(uint32_t)FI_COLOR_CLEAR;
		CU(cudaMemcpyAsync(c->outColor + plane * frame, hostColor, plane * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
	}
	c->target = frame;
	return DTR_B200_OK;
}

int dtr_b200_flush(dtr_b200_ctx *c)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	return do_flush(c);
}

int dtr_b200_replay(dtr_b200_ctx *c)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!c->last.valid) return fail(c, DTR_B200_ERR_ARG, "nothing to replay");
	if (!c->rec.empty()) return fail(c, DTR_B200_ERR_ARG, "replay with unflushed draw calls pending");
	CU(cudaSetDevice(c->device));
	return run_pipeline(c, c->last.numActive, c->last.numItems, c->last.numPrims, c->last.maxFramePrims, true);
}

int dtr_b200_set_replay_overlap(dtr_b200_ctx *c, int enable)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->preStream));
	CU(cudaStreamSynchronize(c->stream));
	c->replayOverlap = enable != 0;
	return DTR_B200_OK;
}

int dtr_b200_sync(dtr_b200_ctx *c)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	return DTR_B200_OK;
}

namespace
{
// The next of the two staging buffers, grown to `bytes`; the context's stream waits until the previous
// transfer out of it has finished.  *turn: its index, for packFree.
int acquire_stage(dtr_b200_ctx *c, size_t bytes, int *turn)
{
	const int k = c->packTurn;
	c->packTurn ^= 1;
	if (!c->packFree[k]) CU(cudaEventCreateWithFlags(&c->packFree[k], cudaEventDisableTiming));
	else CU(cudaStreamWaitEvent(c->stream, c->packFree[k], 0)); // the previous transfer out of this buffer
	if (bytes > c->packStage[k].cap)
	{
		CU(cudaStreamSynchronize(c->copyStream)); // ensure_dev frees the old buffer
		int rc = ensure_dev(c, c->packStage[k], bytes);
		if (rc) return rc;
	}
	*turn = k;
	return DTR_B200_OK;
}

// Resolves frames [first, first + n) at the context's factor into device memory (each output may be null),
// in stream order.  It reads the planes the unresolved readbacks copy.
int resolve_into(dtr_b200_ctx *c, int first, int n, uint32_t *color, float *z, uint32_t *ids)
{
	const size_t       plane = (size_t)c->width * c->height;
	FrameResolveParams P{};
	P.color    = c->outColor + plane * first;
	P.depth    = c->outDepth + plane * first;
	P.ids      = c->dIds ? c->dIds + plane * first : nullptr;
	P.outColor = color;
	P.outDepth = z;
	P.outIds   = ids;
	P.width    = c->width;
	P.height   = c->height;
	P.frames   = n;
	launch_resolve_frames(P, c->resolve, c->stream);
	CU(cudaGetLastError());
	return DTR_B200_OK;
}

// The synchronous readbacks at k > 1 (after the flush): resolve into a staging buffer, copy out, wait
int read_resolved(dtr_b200_ctx *c, int first, int n, uint32_t *hostColor, float *hostZ, uint32_t *hostIds)
{
	const size_t bytes = (size_t)(c->width / c->resolve) * (c->height / c->resolve) * n * sizeof(uint32_t);
	void *const  host[3] = {hostColor, hostZ, hostIds};
	const int    planes  = (hostColor != nullptr) + (hostZ != nullptr) + (hostIds != nullptr);
	if (planes)
	{
		int turn = 0, rc = acquire_stage(c, bytes * planes, &turn);
		if (rc) return rc;
		uint8_t *dev[3] = {nullptr, nullptr, nullptr}, *next = static_cast<uint8_t *>(c->packStage[turn].p);
		for (int i = 0; i < 3; i++)
			if (host[i])
			{
				dev[i] = next;
				next += bytes;
			}
		rc = resolve_into(c, first, n, (uint32_t *)dev[0], (float *)dev[1], (uint32_t *)dev[2]);
		if (rc) return rc;
		for (int i = 0; i < 3; i++)
			if (host[i]) CU(cudaMemcpyAsync(host[i], dev[i], bytes, cudaMemcpyDeviceToHost, c->stream));
	}
	CU(cudaStreamSynchronize(c->stream));
	return DTR_B200_OK;
}
} // namespace

int dtr_b200_set_readback_resolve(dtr_b200_ctx *c, int k)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (k < 1 || k > 4 || c->width % k || c->height % k)
		return fail(c, DTR_B200_ERR_ARG, "resolve factor must be in 1..4 and divide the frame's width and height");
	c->resolve = k;
	return DTR_B200_OK;
}

int dtr_b200_resolve_frames(dtr_b200_ctx *c, int first, int n, void *color, void *z, void *ids)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (ids && !c->dIds) return fail(c, DTR_B200_ERR_ARG, "triangle id output is off (dtr_b200_set_id_output)");
	if (n <= 0 || !valid_frame(c, first) || !valid_frame(c, first + n - 1)) return fail(c, DTR_B200_ERR_ARG, "frame range out of bounds");
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	if (c->resolve > 1) return resolve_into(c, first, n, (uint32_t *)color, (float *)z, (uint32_t *)ids);
	const size_t bytes = (size_t)c->width * c->height * n * sizeof(uint32_t), off = (size_t)c->width * c->height * first;
	if (color) CU(cudaMemcpyAsync(color, c->outColor + off, bytes, cudaMemcpyDeviceToDevice, c->stream));
	if (z) CU(cudaMemcpyAsync(z, c->outDepth + off, bytes, cudaMemcpyDeviceToDevice, c->stream));
	if (ids) CU(cudaMemcpyAsync(ids, c->dIds + off, bytes, cudaMemcpyDeviceToDevice, c->stream));
	return DTR_B200_OK;
}

int dtr_b200_end_frame(dtr_b200_ctx *c, int frame, uint32_t *hostColor, float *hostZ)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!valid_frame(c, frame)) return fail(c, DTR_B200_ERR_ARG, "frame out of range");
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	if (c->resolve > 1) return read_resolved(c, frame, 1, hostColor, hostZ, nullptr);
	size_t plane = (size_t)c->width * c->height;
	if (hostColor)
		CU(cudaMemcpyAsync(hostColor, c->outColor + plane * frame, plane * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	if (hostZ) CU(cudaMemcpyAsync(hostZ, c->outDepth + plane * frame, plane * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return DTR_B200_OK;
}

int dtr_b200_read_frames(dtr_b200_ctx *c, int first, int n, uint32_t *hostColor, float *hostZ)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (n <= 0 || !valid_frame(c, first) || !valid_frame(c, first + n - 1)) return fail(c, DTR_B200_ERR_ARG, "frame range out of bounds");
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	if (c->resolve > 1) return read_resolved(c, first, n, hostColor, hostZ, nullptr);
	size_t plane = (size_t)c->width * c->height;
	if (hostColor)
		CU(cudaMemcpyAsync(hostColor, c->outColor + plane * first, plane * n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	if (hostZ)
		CU(cudaMemcpyAsync(hostZ, c->outDepth + plane * first, plane * n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return DTR_B200_OK;
}

int dtr_b200_read_frames_async(dtr_b200_ctx *c, int first, int n, uint32_t *hostColor, float *hostZ)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (n <= 0 || !valid_frame(c, first) || !valid_frame(c, first + n - 1)) return fail(c, DTR_B200_ERR_ARG, "frame range out of bounds");
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	if (c->resolve > 1)
	{
		// resolve into a staging buffer, copy from there: the frames are free once the resolve kernel has run
		const size_t bytes  = (size_t)(c->width / c->resolve) * (c->height / c->resolve) * n * sizeof(uint32_t);
		const int    planes = (hostColor != nullptr) + (hostZ != nullptr);
		if (!planes) return DTR_B200_OK;
		int turn = 0;
		if ((rc = acquire_stage(c, bytes * planes, &turn))) return rc;
		uint8_t *dev = static_cast<uint8_t *>(c->packStage[turn].p), *devZ = hostColor ? dev + bytes : dev;
		if ((rc = resolve_into(c, first, n, hostColor ? (uint32_t *)dev : nullptr, hostZ ? (float *)devZ : nullptr, nullptr))) return rc;
		CU(cudaEventRecord(c->renderDone, c->stream));
		CU(cudaStreamWaitEvent(c->copyStream, c->renderDone, 0));
		if (hostColor) CU(cudaMemcpyAsync(hostColor, dev, bytes, cudaMemcpyDeviceToHost, c->copyStream));
		if (hostZ) CU(cudaMemcpyAsync(hostZ, devZ, bytes, cudaMemcpyDeviceToHost, c->copyStream));
		CU(cudaEventRecord(c->packFree[turn], c->copyStream));
		return DTR_B200_OK;
	}
	size_t plane = (size_t)c->width * c->height;
	CU(cudaEventRecord(c->renderDone, c->stream));
	CU(cudaStreamWaitEvent(c->copyStream, c->renderDone, 0));
	if (hostColor)
		CU(cudaMemcpyAsync(hostColor, c->outColor + plane * first, plane * n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->copyStream));
	if (hostZ)
		CU(cudaMemcpyAsync(hostZ, c->outDepth + plane * first, plane * n * sizeof(float), cudaMemcpyDeviceToHost, c->copyStream));
	CU(cudaEventRecord(c->copyDone, c->copyStream));
	// conservative: one range covering every read in flight
	if (c->readHi > c->readLo)
	{
		c->readLo = std::min(c->readLo, first);
		c->readHi = std::max(c->readHi, first + n);
	}
	else
	{
		c->readLo = first;
		c->readHi = first + n;
	}
	return DTR_B200_OK;
}

int dtr_b200_read_frames_bgr24_async(dtr_b200_ctx *c, int first, int n, uint8_t *hostBgr)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (n <= 0 || !hostBgr || !valid_frame(c, first) || !valid_frame(c, first + n - 1))
		return fail(c, DTR_B200_ERR_ARG, "frame range out of bounds or NULL destination");
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	const int    ow = c->width / c->resolve;
	const size_t pitch = ((size_t)ow * 3 + 3) & ~(size_t)3, rows = (size_t)n * (c->height / c->resolve), bytes = pitch * rows;
	int          k = 0;
	if ((rc = acquire_stage(c, bytes, &k))) return rc;
	// the frames are free again as soon as the pack kernel has run (same stream as the rendering)
	const uint32_t *frames = c->outColor + (size_t)c->width * c->height * first;
	if (c->resolve > 1)
		launch_resolve_pack_bgr24(frames, static_cast<uint32_t *>(c->packStage[k].p), c->width, c->resolve, rows, (int)(pitch / 4), c->stream);
	else launch_pack_bgr24(frames, static_cast<uint32_t *>(c->packStage[k].p), c->width, rows, (int)(pitch / 4), c->stream);
	CU(cudaGetLastError());
	CU(cudaEventRecord(c->renderDone, c->stream));
	CU(cudaStreamWaitEvent(c->copyStream, c->renderDone, 0));
	CU(cudaMemcpyAsync(hostBgr, c->packStage[k].p, bytes, cudaMemcpyDeviceToHost, c->copyStream));
	CU(cudaEventRecord(c->packFree[k], c->copyStream));
	return DTR_B200_OK;
}

int dtr_b200_wait_reads(dtr_b200_ctx *c)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->copyStream));
	c->readLo = c->readHi = 0;
	return DTR_B200_OK;
}

// ---- rendering into a peer GPU's frames (sort-first bands without a gather step) -----------------
static_assert(sizeof(cudaIpcMemHandle_t) == DTR_B200_IPC_HANDLE_BYTES, "IPC handle size");

int dtr_b200_export_frames(dtr_b200_ctx *c, uint8_t *colorHandle, uint8_t *depthHandle)
{
	if (!c || !colorHandle || !depthHandle) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	cudaIpcMemHandle_t hc, hz;
	CU(cudaIpcGetMemHandle(&hc, c->dColor));
	CU(cudaIpcGetMemHandle(&hz, c->dDepth));
	memcpy(colorHandle, &hc, sizeof(hc));
	memcpy(depthHandle, &hz, sizeof(hz));
	return DTR_B200_OK;
}

int dtr_b200_set_output_planes(dtr_b200_ctx *c, void *color, void *depth)
{
	if (!c || ((color == nullptr) != (depth == nullptr))) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c); // what was recorded so far belongs to the previous target
	if (rc) return rc;
	CU(cudaStreamSynchronize(c->stream));
	c->outColor = color ? (uint32_t *)color : c->dColor;
	c->outDepth = depth ? (float *)depth : c->dDepth;
	c->last.valid = false; // a replay must not silently switch targets
	return DTR_B200_OK;
}

int dtr_b200_open_peer_frames(dtr_b200_ctx *c, const uint8_t *colorHandle, const uint8_t *depthHandle)
{
	if (!c || !colorHandle || !depthHandle) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	if (c->ipcColor || c->ipcDepth) return fail(c, DTR_B200_ERR_ARG, "peer frames already open");
	cudaIpcMemHandle_t hc, hz;
	memcpy(&hc, colorHandle, sizeof(hc));
	memcpy(&hz, depthHandle, sizeof(hz));
	CU(cudaIpcOpenMemHandle(&c->ipcColor, hc, cudaIpcMemLazyEnablePeerAccess));
	CU(cudaIpcOpenMemHandle(&c->ipcDepth, hz, cudaIpcMemLazyEnablePeerAccess));
	return dtr_b200_set_output_planes(c, c->ipcColor, c->ipcDepth);
}

int dtr_b200_enable_peer_access(dtr_b200_ctx *c, int peerDevice)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	int can = 0;
	CU(cudaDeviceCanAccessPeer(&can, c->device, peerDevice));
	if (!can) return fail(c, DTR_B200_ERR_CUDA, "devices cannot access each other's memory");
	cudaError_t e = cudaDeviceEnablePeerAccess(peerDevice, 0);
	if (e == cudaErrorPeerAccessAlreadyEnabled)
	{
		cudaGetLastError();
		return DTR_B200_OK;
	}
	CU(e);
	return DTR_B200_OK;
}

// ---- sort-first bands behind the C ABI: partition, exchange (NCCL) and barrier -------------------
int dtr_b200_tile_height(void) { return TILE_H; }

int dtr_b200_band_rows(int height, int nranks, int rank, int *y0, int *y1)
{
	if (height <= 0 || nranks <= 0 || rank < 0 || rank >= nranks || !y0 || !y1) return DTR_B200_ERR_ARG;
	const int tiles = (height + TILE_H - 1) / TILE_H, base = tiles / nranks, rem = tiles % nranks;
	const int t0 = rank * base + std::min(rank, rem), t1 = t0 + base + (rank < rem ? 1 : 0);
	*y0 = std::min(t0 * TILE_H, height);
	*y1 = std::min(t1 * TILE_H, height);
	return DTR_B200_OK;
}

#define NC(call)                                                                                          \
	do                                                                                                    \
	{                                                                                                     \
		int r_ = (call);                                                                                  \
		if (r_ != 0)                                                                                      \
		{                                                                                                 \
			std::string m_ = std::string(#call ": ") + (N.GetErrorString ? N.GetErrorString(r_) : "NCCL error"); \
			return fail(c, DTR_B200_ERR_CUDA, m_.c_str());                                                \
		}                                                                                                 \
	} while (0)

int dtr_b200_band_comm_unique_id(uint8_t id[DTR_B200_NCCL_ID_BYTES])
{
	static_assert(sizeof(NcclUniqueId) == DTR_B200_NCCL_ID_BYTES, "ncclUniqueId size");
	dtr_b200_ctx  *c = nullptr;
	const NcclApi &N = nccl_api();
	if (!id) return DTR_B200_ERR_ARG;
	if (!N.ok) return fail(c, DTR_B200_ERR_CUDA, N.err.c_str());
	NcclUniqueId u;
	NC(N.GetUniqueId(&u));
	memcpy(id, &u, sizeof(u));
	return DTR_B200_OK;
}

namespace
{
int adopt_comm(dtr_b200_ctx *c, NcclComm comm, bool own, int nranks, int rank)
{
	if (c->comm && c->ownComm) nccl_api().CommDestroy(c->comm);
	c->comm      = comm;
	c->ownComm   = own;
	c->commRanks = nranks;
	c->commRank  = rank;
	if (!c->dToken)
	{
		CU(cudaMalloc((void **)&c->dToken, sizeof(float)));
		CU(cudaMemset(c->dToken, 0, sizeof(float)));
	}
	return DTR_B200_OK;
}
} // namespace

int dtr_b200_band_comm_init(dtr_b200_ctx *c, const uint8_t id[DTR_B200_NCCL_ID_BYTES], int nranks, int rank)
{
	if (!c || !id || nranks <= 0 || rank < 0 || rank >= nranks) return DTR_B200_ERR_ARG;
	const NcclApi &N = nccl_api();
	if (!N.ok) return fail(c, DTR_B200_ERR_CUDA, N.err.c_str());
	CU(cudaSetDevice(c->device));
	NcclUniqueId u;
	memcpy(&u, id, sizeof(u));
	NcclComm comm = nullptr;
	NC(N.CommInitRank(&comm, nranks, u, rank));
	return adopt_comm(c, comm, true, nranks, rank);
}

int dtr_b200_band_comm_attach(dtr_b200_ctx *c, void *ncclComm, int nranks, int rank)
{
	if (!c || !ncclComm || nranks <= 0 || rank < 0 || rank >= nranks) return DTR_B200_ERR_ARG;
	const NcclApi &N = nccl_api();
	if (!N.ok) return fail(c, DTR_B200_ERR_CUDA, N.err.c_str());
	CU(cudaSetDevice(c->device));
	return adopt_comm(c, (NcclComm)ncclComm, false, nranks, rank);
}

int dtr_b200_gather_bands(dtr_b200_ctx *c, int frame, int dstRank)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!c->comm) return fail(c, DTR_B200_ERR_ARG, "no band communicator (dtr_b200_band_comm_init / _attach)");
	if (!valid_frame(c, frame) || dstRank < 0 || dstRank >= c->commRanks) return fail(c, DTR_B200_ERR_ARG, "frame or dstRank out of range");
	const NcclApi &N = nccl_api();
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	const size_t plane = (size_t)c->width * c->height;
	uint32_t    *col   = c->outColor + plane * frame;
	float       *dep   = c->outDepth + plane * frame;
	if (c->commRank != dstRank)
	{
		// the rows this context rasterises must be its rank's band of THE partition
		int y0 = 0, y1 = 0;
		dtr_b200_band_rows(c->height, c->commRanks, c->commRank, &y0, &y1);
		if (y1 > y0 && (c->geom.bandTileY0 * TILE_H != y0 || std::min(c->geom.bandTileY1 * TILE_H, c->height) != y1))
			return fail(c, DTR_B200_ERR_ARG, "this context's band is not dtr_b200_band_rows(height, nranks, rank)");
	}
	NC(N.GroupStart());
	for (int r = 0; r < c->commRanks; r++)
	{
		int y0 = 0, y1 = 0;
		dtr_b200_band_rows(c->height, c->commRanks, r, &y0, &y1);
		if (r == dstRank || y1 <= y0) continue;
		const size_t off = (size_t)y0 * c->width, n = (size_t)(y1 - y0) * c->width; // rows are contiguous: one message per plane
		if (c->commRank == dstRank)
		{
			NC(N.Recv(col + off, n, NCCL_UINT32, r, c->comm, c->stream));
			NC(N.Recv(dep + off, n, NCCL_FLOAT32, r, c->comm, c->stream));
		}
		else if (c->commRank == r)
		{
			NC(N.Send(col + off, n, NCCL_UINT32, dstRank, c->comm, c->stream));
			NC(N.Send(dep + off, n, NCCL_FLOAT32, dstRank, c->comm, c->stream));
		}
	}
	NC(N.GroupEnd());
	return DTR_B200_OK;
}

int dtr_b200_band_barrier(dtr_b200_ctx *c)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!c->comm) return fail(c, DTR_B200_ERR_ARG, "no band communicator (dtr_b200_band_comm_init / _attach)");
	const NcclApi &N = nccl_api();
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	NC(N.AllReduce(c->dToken, c->dToken, 1, NCCL_FLOAT32, NCCL_SUM, c->comm, c->stream));
	return DTR_B200_OK;
}
#undef NC

int dtr_b200_frame_device_ptrs(dtr_b200_ctx *c, int frame, void **color, void **z)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!valid_frame(c, frame)) return fail(c, DTR_B200_ERR_ARG, "frame out of range");
	size_t plane = (size_t)c->width * c->height;
	if (color) *color = c->outColor + plane * frame;
	if (z) *z = c->outDepth + plane * frame;
	return DTR_B200_OK;
}

int dtr_b200_set_id_output(dtr_b200_ctx *c, int enable)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	if ((enable != 0) == (c->dIds != nullptr)) return DTR_B200_OK;
	// (enqueued passes may still use the buffers; draw calls recorded but not yet flushed run with the new setting)
	CU(cudaStreamSynchronize(c->preStream));
	CU(cudaStreamSynchronize(c->stream));
	if (!enable)
	{
		CU(cudaFree(c->dIds));
		c->dIds = nullptr;
		for (auto &ps : c->sets)
		{
			CU(cudaFree(ps.primId.p));
			ps.primId = DevBuf();
		}
		return DTR_B200_OK;
	}
	const size_t bytes = (size_t)c->width * c->height * c->numFrames * sizeof(uint32_t);
	uint32_t    *d     = nullptr;
	const cudaError_t e = cudaMalloc((void **)&d, bytes);
	if (e == cudaErrorMemoryAllocation)
	{
		cudaGetLastError(); // (not sticky: clear it)
		return fail(c, DTR_B200_ERR_NOMEM, "allocating the triangle id planes", e);
	}
	if (e != cudaSuccess) return fail(c, DTR_B200_ERR_CUDA, "allocating the triangle id planes", e);
	c->dIds = d;
	CU(cudaMemsetAsync(c->dIds, 0, bytes, c->stream));
	return DTR_B200_OK;
}

int dtr_b200_read_ids(dtr_b200_ctx *c, int first, int n, uint32_t *hostIds)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!c->dIds) return fail(c, DTR_B200_ERR_ARG, "triangle id output is off (dtr_b200_set_id_output)");
	if (!hostIds || n <= 0 || !valid_frame(c, first) || !valid_frame(c, first + n - 1)) return fail(c, DTR_B200_ERR_ARG, "frame range out of bounds");
	CU(cudaSetDevice(c->device));
	int rc = do_flush(c);
	if (rc) return rc;
	if (c->resolve > 1) return read_resolved(c, first, n, nullptr, nullptr, hostIds);
	const size_t plane = (size_t)c->width * c->height;
	CU(cudaMemcpyAsync(hostIds, c->dIds + plane * first, plane * n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return DTR_B200_OK;
}

int dtr_b200_frame_id_ptr(dtr_b200_ctx *c, int frame, void **ids)
{
	if (!c || !ids) return DTR_B200_ERR_ARG;
	if (!c->dIds) return fail(c, DTR_B200_ERR_ARG, "triangle id output is off (dtr_b200_set_id_output)");
	if (!valid_frame(c, frame)) return fail(c, DTR_B200_ERR_ARG, "frame out of range");
	*ids = c->dIds + (size_t)c->width * c->height * frame;
	return DTR_B200_OK;
}

int dtr_b200_get_stats(dtr_b200_ctx *c, dtr_b200_stats *out)
{
	if (!c || !out) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	unsigned long long sp = 0;
	CU(cudaMemcpy(&sp, c->dSetPixels, sizeof(sp), cudaMemcpyDeviceToHost));
	out->setPixels      = sp;
	out->triangles      = c->triangles;
	out->primitives     = c->last.numPrims;
	out->listEntries    = c->last.listTotal;
	out->kernelLaunches = c->launches;
	out->uploadBytes    = c->uploadBytes;
	return DTR_B200_OK;
}

int dtr_b200_last_pass_deferred(const dtr_b200_ctx *c) { return (c && c->last.valid && c->last.deferred) ? (c->last.oneKernel ? 2 : 1) : 0; }

int dtr_b200_set_opaque_stage(dtr_b200_ctx *c, int mode)
{
	if (!c || mode < DTR_B200_OPAQUE_SINGLE_KERNEL || mode > DTR_B200_OPAQUE_ONE_KERNEL) return DTR_B200_ERR_ARG;
	c->opaqueStage = mode;
	return DTR_B200_OK;
}

int dtr_b200_selftest(dtr_b200_ctx *c, uint64_t *mismatches)
{
	if (!c || !mismatches) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	unsigned long long *d = nullptr, h = 0;
	CU(cudaMalloc((void **)&d, sizeof(h)));
	CU(cudaMemsetAsync(d, 0, sizeof(h), c->stream));
	launch_selftest_sqrt(d, c->stream);
	CU(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	CU(cudaFree(d));
	*mismatches = h;
	return DTR_B200_OK;
}

int dtr_b200_set_profiling(dtr_b200_ctx *c, int enable)
{
	if (!c) return DTR_B200_ERR_ARG;
	c->profiling = enable != 0;
	return DTR_B200_OK;
}

int dtr_b200_reset_stage_ms(dtr_b200_ctx *c)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	for (cudaEvent_t e : c->events) c->eventPool.push_back(e);
	c->events.clear();
	return DTR_B200_OK;
}

int dtr_b200_get_stage_ms(dtr_b200_ctx *c, float ms[4], int *runs)
{
	if (!c || !ms || !runs) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	ms[0] = ms[1] = ms[2] = ms[3] = 0.0f;
	CU(cudaStreamSynchronize(c->preStream));
	*runs = (int)(c->events.size() / EVENTS_PER_RUN);
	for (int r = 0; r < *runs; r++)
	{
		// setup, scan, bin: consecutive events on the stream that ran them; raster: its own pair of
		// events on the main stream (with pipelined replays the raster kernel may start long after bin)
		const cudaEvent_t *ev = &c->events[(size_t)EVENTS_PER_RUN * r];
		for (int s2 = 0; s2 < 3; s2++)
		{
			float t = 0.0f;
			CU(cudaEventElapsedTime(&t, ev[s2], ev[s2 + 1]));
			ms[s2] += t;
		}
		float t = 0.0f;
		CU(cudaEventElapsedTime(&t, ev[4], ev[6]));
		ms[3] += t;
	}
	return DTR_B200_OK;
}

int dtr_b200_get_raster_split_ms(dtr_b200_ctx *c, float ms[2], int *runs)
{
	if (!c || !ms || !runs) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	ms[0] = ms[1] = 0.0f;
	*runs = (int)(c->events.size() / EVENTS_PER_RUN);
	for (int r = 0; r < *runs; r++)
	{
		const cudaEvent_t *ev = &c->events[(size_t)EVENTS_PER_RUN * r];
		float a = 0.0f, b = 0.0f;
		CU(cudaEventElapsedTime(&a, ev[4], ev[5]));
		CU(cudaEventElapsedTime(&b, ev[5], ev[6]));
		ms[0] += a;
		ms[1] += b;
	}
	return DTR_B200_OK;
}

int dtr_b200_reset_stats(dtr_b200_ctx *c)
{
	if (!c) return DTR_B200_ERR_ARG;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	CU(cudaMemset(c->dSetPixels, 0, sizeof(unsigned long long)));
	c->triangles = 0;
	c->launches  = 0;
	return DTR_B200_OK;
}

// ---- draw calls ---------------------------------------------------------------------------------

int dtr_b200_clear(dtr_b200_ctx *c, const float rgb[3])
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!rgb) return DTR_B200_OK;
	uint32_t   packed = pack_clear(rgb);
	FrameHost &fh     = c->frames[c->target];
	if (fh.recorded == 0)
	{
		// first command of the batch for this frame: the tile kernel generates the colour on chip
		fh.pendingInit |= FI_COLOR_CLEAR;
		fh.clearPacked = packed;
		return DTR_B200_OK;
	}
	PrimRecord r;
	memset(&r, 0, sizeof(r));
	r.w[QW_FLAGS]  = PRIM_CLEAR;
	r.w[QW_MIN]    = 0;
	r.w[QW_MAX]    = (uint32_t)c->width | ((uint32_t)c->height << 16);
	r.w[QW_PACKED] = packed;
	return record_raw(c, r);
}

int dtr_b200_triangle(dtr_b200_ctx *c, const float p1[3], const float p2[3], const float p3[3],
                      const float color[4], const dtr_b200_transform *t)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!p1 || !p2 || !p3 || !color) return DTR_B200_OK;
	float p[9] = {p1[0], p1[1], p1[2], p2[0], p2[1], p2[2], p3[0], p3[1], p3[2]};
	return record_tris(c, 1, p, color, nullptr, -1, t);
}

int dtr_b200_triangles(dtr_b200_ctx *c, int n, const float *p, const float *color, const dtr_b200_transform *t)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (n <= 0 || !p || !color) return DTR_B200_OK;
	return record_tris(c, n, p, color, nullptr, -1, t);
}

int dtr_b200_textured_triangle(dtr_b200_ctx *c, const float p1[3], const float p2[3], const float p3[3],
                               const float uv1[2], const float uv2[2], const float uv3[2], int texId,
                               const float color[4], const dtr_b200_transform *t)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!p1 || !p2 || !p3 || !uv1 || !uv2 || !uv3 || !color) return DTR_B200_OK;
	if (texId >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
	float p[9]  = {p1[0], p1[1], p1[2], p2[0], p2[1], p2[2], p3[0], p3[1], p3[2]};
	float uv[6] = {uv1[0], uv1[1], uv2[0], uv2[1], uv3[0], uv3[1]};
	return record_tris(c, 1, p, color, uv, texId < 0 ? -1 : texId, t);
}

int dtr_b200_mesh_views(dtr_b200_ctx *c, int meshId, const dtr_b200_light *light, int nViews, const float *pos,
                        const dtr_b200_transform *transforms, int firstFrame)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!light || !pos || !transforms || nViews <= 0) return DTR_B200_OK;
	if (meshId < 0 || meshId >= (int)c->meshes.size()) return fail(c, DTR_B200_ERR_ARG, "meshId out of range");
	if (!valid_frame(c, firstFrame) || !valid_frame(c, firstFrame + nViews - 1))
		return fail(c, DTR_B200_ERR_ARG, "views do not fit the context's frames");
	const MeshAsset &m = c->meshes[meshId];
	Basis2           b = make_basis(0.0f, 1.0f, 1.0f); // DTRRender_DefaultTriangleTransform()
	for (int v = 0; v < nViews; v++)
	{
		const dtr_b200_transform &t = transforms[v];
		Mat4     M = mesh_matrix(c->width, c->height, pos + 3 * v, t.rotation, t.anchor, t.scale);
		RecItem &r = new_item(c, ITEM_MESH, (uint32_t)(firstFrame + v), m.numFaces);
		// DTRRender_Mesh always samples mesh->tex (:1563-1564); an all-white one is a no-op
		r.item.texId     = (m.texId >= 0 && c->texIsWhite[m.texId]) ? -1 : m.texId;
		r.opaque         = light->color[3] == 1.0f && (r.item.texId < 0 || c->texIsOpaque[r.item.texId]);
		r.item.lightMode = (uint32_t)light->mode;
		r.item.ptr[0]    = (uint64_t)m.vertexes;
		r.item.ptr[1]    = (uint64_t)m.texUV;
		r.item.ptr[2]    = (uint64_t)m.normals;
		r.item.ptr[3]    = (uint64_t)m.faces;
		r.item.xAxis[0] = b.xAxis[0]; r.item.xAxis[1] = b.xAxis[1];
		r.item.yAxis[0] = b.yAxis[0]; r.item.yAxis[1] = b.yAxis[1];
		r.item.anchor[0] = 0.33f;
		r.item.anchor[1] = 0.33f;
		memcpy(r.item.m, M.e, sizeof(float) * 16);
		r.item.lightVec[0] = light->vector[0];
		r.item.lightVec[1] = light->vector[1];
		r.item.lightVec[2] = light->vector[2];
		memcpy(r.item.color, light->color, sizeof(float) * 4);
		c->triangles += m.numFaces;
	}
	return DTR_B200_OK;
}

int dtr_b200_triangles_device(dtr_b200_ctx *c, int n, const float *p, const float *color, const float *uv, int texId,
                              const dtr_b200_transform *t)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (n <= 0 || !p || !color) return DTR_B200_OK;
	if (texId >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
	if (!on_ctx_device(c, p) || !on_ctx_device(c, color) || (uv && !on_ctx_device(c, uv)))
		return fail(c, DTR_B200_ERR_ARG, "p / color / uv must be device memory of the context's device");
	RecItem &r    = new_tris_item(c, n, (uv && texId >= 0) ? texId : -1, t);
	r.snap[0]     = snap_push(c, p, sizeof(float) * 9 * (size_t)n, false);
	r.fromSnap[0] = true;
	r.snap[1]     = snap_push(c, color, sizeof(float) * 4 * (size_t)n, true);
	r.fromSnap[1] = true;
	if (uv)
	{
		r.snap[2]     = snap_push(c, uv, sizeof(float) * 6 * (size_t)n, false);
		r.fromSnap[2] = true;
	}
	return DTR_B200_OK;
}

int dtr_b200_mesh_views_device(dtr_b200_ctx *c, int meshId, const dtr_b200_light *light, int nViews, const float *pos,
                               const dtr_b200_transform *transforms, int firstFrame, const float *vertexes, const float *normals)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!light || !pos || !transforms || nViews <= 0 || !vertexes) return DTR_B200_OK;
	if (meshId < 0 || meshId >= (int)c->meshes.size()) return fail(c, DTR_B200_ERR_ARG, "meshId out of range");
	if (!valid_frame(c, firstFrame) || !valid_frame(c, firstFrame + nViews - 1))
		return fail(c, DTR_B200_ERR_ARG, "views do not fit the context's frames");
	if (!on_ctx_device(c, vertexes) || (normals && !on_ctx_device(c, normals)))
		return fail(c, DTR_B200_ERR_ARG, "vertexes / normals must be device memory of the context's device");
	const size_t first = c->rec.size();
	int          rc    = dtr_b200_mesh_views(c, meshId, light, nViews, pos, transforms, firstFrame);
	if (rc) return rc;
	// view v: vertex set v (and normal set v) instead of the mesh's own arrays
	const MeshAsset &m  = c->meshes[meshId];
	const size_t     vB = sizeof(float) * 4 * (size_t)m.numVertexes, nB = sizeof(float) * 3 * (size_t)m.numNormals;
	const size_t     vAt = snap_push(c, vertexes, vB * nViews, false);
	const size_t     nAt = normals ? snap_push(c, normals, nB * nViews, false) : 0;
	for (int v = 0; v < nViews; v++)
	{
		RecItem &r    = c->rec[first + v];
		r.snap[0]     = vAt + vB * v; // vB is a multiple of 16: every set stays float4 aligned
		r.fromSnap[0] = true;
		if (normals)
		{
			r.snap[2]     = nAt + nB * v;
			r.fromSnap[2] = true;
		}
	}
	return DTR_B200_OK;
}

int dtr_b200_mesh(dtr_b200_ctx *c, int meshId, const dtr_b200_light *light, const float pos[3],
                  const dtr_b200_transform *t)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!t) t = &kDefaultTransform;
	return dtr_b200_mesh_views(c, meshId, light, 1, pos, t, c->target);
}

namespace
{
// DTRRender_Line (:294-356) as one PRIM_LINE record
int emit_line(dtr_b200_ctx *c, const int32_t a[2], const int32_t b[2], const float color[4])
{
	// DTRRender_Line (:294-356): x-major integer DDA after the optional axis swap
	int ax = a[0], ay = a[1], bx = b[0], by = b[1];
	int steep = std::abs(ax - bx) < std::abs(ay - by);
	if (steep) { std::swap(ax, ay); std::swap(bx, by); }
	if (bx < ax) { std::swap(ax, bx); std::swap(ay, by); }
	int run = bx - ax, rise = by - ay;
	if (run <= 0) return DTR_B200_OK;
	int delta = (by > ay) ? 1 : -1;
	// pixel bbox in screen orientation, clipped (SetPixel rejects the rest, :129-130)
	int majLo = ax, majHi = ax + run; // [lo, hi)
	int minLo = std::min(ay, by), minHi = std::max(ay, by) + 1;
	int x0 = steep ? minLo : majLo, x1 = steep ? minHi : majHi, y0 = steep ? majLo : minLo, y1 = steep ? majHi : minHi;
	x0 = clampi(x0, 0, c->width); x1 = clampi(x1, 0, c->width);
	y0 = clampi(y0, 0, c->height); y1 = clampi(y1, 0, c->height);
	if (x1 <= x0 || y1 <= y0) return DTR_B200_OK;
	float col[4];
	to_linear_premul(color, col);
	PrimRecord r;
	memset(&r, 0, sizeof(r));
	r.w[QW_FLAGS] = PRIM_LINE;
	r.w[QW_MIN]   = (uint32_t)x0 | ((uint32_t)y0 << 16);
	r.w[QW_MAX]   = (uint32_t)x1 | ((uint32_t)y1 << 16);
	for (int i = 0; i < 4; i++) r.w[QW_COLOR + i] = f2u(col[i]);
	r.w[QW_LINE + 0] = (uint32_t)ax;
	r.w[QW_LINE + 1] = (uint32_t)ay;
	r.w[QW_LINE + 2] = (uint32_t)run;
	r.w[QW_LINE + 3] = (uint32_t)(std::abs(rise) * 2);
	r.w[QW_LINE + 4] = (uint32_t)delta;
	r.w[QW_LINE + 5] = (uint32_t)steep;
	return record_raw(c, r);
}

int emit_line4(dtr_b200_ctx *c, int x0, int y0, int x1, int y1, const float color[4])
{
	const int32_t a[2] = {x0, y0}, b[2] = {x1, y1};
	return emit_line(c, a, b, color);
}

int emit_rectangle(dtr_b200_ctx *c, const float mn[2], const float mx[2], const float color[4], const dtr_b200_transform *t);

// The four bounding-box lines the reference's debug build draws (:492-501, :732-741); the corners
// are truncated to integers like DqnV2i_2f does.
int emit_bbox_lines(dtr_b200_ctx *c, const float bounds[4], const float color[4])
{
	const int x0 = (int)bounds[0], y0 = (int)bounds[1], x1 = (int)bounds[2], y1 = (int)bounds[3];
	int rc;
	if ((rc = emit_line4(c, x0, y0, x0, y1, color))) return rc;
	if ((rc = emit_line4(c, x0, y1, x1, y1, color))) return rc;
	if ((rc = emit_line4(c, x1, y1, x1, y0, color))) return rc;
	return emit_line4(c, x1, y0, x0, y0, color);
}

// DTRRender_Rectangle (:415-513) including, when enabled, its DTR_DEBUG_RENDER block: bounding-box
// lines in the rectangle's colour AFTER the linear/premultiply conversion (the reference reuses the
// converted variable, and DTRRender_Line converts it again), and a green outline when rotation > 0.
int emit_rectangle(dtr_b200_ctx *c, const float mn[2], const float mx[2], const float color[4], const dtr_b200_transform *t)
{
	PrimRecord r;
	float      pts[4][2], bounds[4];
	int        rc = 0;
	if (setup_quad(c->width, c->height, mn, mx, t->rotation, t->anchor, t->scale, color, false, -1, 0, 0, &r, pts, bounds))
		rc = record_raw(c, r);
	if (rc || !c->debugMarkers) return rc;
	float lin[4];
	to_linear_premul(color, lin);
	if ((rc = emit_bbox_lines(c, bounds, lin))) return rc;
	if (t->rotation > 0)
	{
		const float green[4] = {0, 1, 0, 1};
		for (int i = 0; i < 4 && !rc; i++)
			rc = emit_line4(c, (int)pts[i][0], (int)pts[i][1], (int)pts[(i + 1) & 3][0], (int)pts[(i + 1) & 3][1], green);
	}
	return rc;
}
} // namespace

int dtr_b200_line(dtr_b200_ctx *c, const int32_t a[2], const int32_t b[2], const float color[4])
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!a || !b || !color) return DTR_B200_OK;
	return emit_line(c, a, b, color);
}

int dtr_b200_upload_font(dtr_b200_ctx *c, const uint8_t *atlas, int atlasWidth, int atlasHeight,
                         const dtr_b200_packedchar *chars, int codepointMin, int codepointMax, int *fontId)
{
	if (!c || !fontId) return DTR_B200_ERR_ARG;
	if (!atlas || !chars || atlasWidth <= 0 || atlasHeight <= 0 || codepointMax <= codepointMin)
		return fail(c, DTR_B200_ERR_ARG, "bad font");
	CU(cudaSetDevice(c->device));
	dtr_b200_ctx::FontHost f;
	f.w = atlasWidth; f.h = atlasHeight; f.cpMin = codepointMin; f.cpMax = codepointMax;
	f.chars.assign(chars, chars + (codepointMax - codepointMin));
	const size_t bytes = (size_t)atlasWidth * atlasHeight;
	CU(cudaMalloc((void **)&f.dAtlas, bytes));
	CU(cudaMemcpy(f.dAtlas, atlas, bytes, cudaMemcpyHostToDevice));
	c->fonts.push_back(std::move(f));
	*fontId = (int)c->fonts.size() - 1;
	return DTR_B200_OK;
}

int dtr_b200_text(dtr_b200_ctx *c, int fontId, const float pos[2], const char *text, const float color[4], int len)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!text || !pos || !color) return DTR_B200_OK; // the reference returns silently (:197-200)
	if (fontId < 0 || fontId >= (int)c->fonts.size()) return fail(c, DTR_B200_ERR_ARG, "fontId out of range");
	const dtr_b200_ctx::FontHost &f = c->fonts[fontId];
	if (len == -1) len = (int)strlen(text);
	float col[4];
	to_linear_premul(color, col);
	float       posx = pos[0], posy = pos[1];
	const float ipw = 1.0f / (float)f.w, iph = 1.0f / (float)f.h; // stbtt_GetPackedQuad (stb_truetype.h:3739-3763)
	for (int index = 0; index < len; index++)
	{
		const int charIndex = (int)text[index] - f.cpMin;
		if (charIndex < 0 || charIndex >= f.cpMax - f.cpMin) return fail(c, DTR_B200_ERR_ARG, "character outside the font's codepoint range");
		const dtr_b200_packedchar &b = f.chars[charIndex];
		const float qx0 = (float)(int)std::floor((double)((posx + b.xoff) + 0.5f));
		const float qy0 = (float)(int)std::floor((double)((posy + b.yoff) + 0.5f));
		const float s0 = (float)b.x0 * ipw, t0 = (float)b.y0 * iph, s1 = (float)b.x1 * ipw, t1 = (float)b.y1 * iph;
		posx += b.xadvance;
		const float    fminx = s0 * (float)f.w, fminy = t1 * (float)f.h; // fontRect.min (:226-227)
		const float    fmaxx = s1 * (float)f.w, fmaxy = t0 * (float)f.h; // fontRect.max
		const uint32_t pitch = (uint32_t)f.w;
		const uint32_t fontOffset = (uint32_t)(fminx + (fmaxy * (float)pitch)); // (:236)
		const float    fho = b.yoff2 + b.yoff;                                   // (:246)
		const int      fw = std::abs((int)(fminx - fmaxx)), fh = std::abs((int)(fminy - fmaxy));
		if (fw <= 0 || fh <= 0) continue;
		// pixels touched: actualX / actualY are monotone in x / y (:264-265)
		int x0 = (int)(qx0 + 0.0f), x1 = (int)(qx0 + (float)(fw - 1)) + 1;
		int y0 = (int)((qy0 + 0.0f) - fho), y1 = (int)((qy0 + (float)(fh - 1)) - fho) + 1;
		x0 = clampi(x0, 0, c->width); x1 = clampi(x1, 0, c->width);
		y0 = clampi(y0, 0, c->height); y1 = clampi(y1, 0, c->height);
		if (x1 <= x0 || y1 <= y0) continue;
		PrimRecord r;
		memset(&r, 0, sizeof(r));
		r.w[QW_FLAGS] = PRIM_GLYPH;
		r.w[QW_MIN]   = (uint32_t)x0 | ((uint32_t)y0 << 16);
		r.w[QW_MAX]   = (uint32_t)x1 | ((uint32_t)y1 << 16);
		for (int i = 0; i < 4; i++) r.w[QW_COLOR + i] = f2u(col[i]);
		const unsigned long long ap = (unsigned long long)(uintptr_t)f.dAtlas;
		r.w[QW_GLYPH + 0] = (uint32_t)ap;
		r.w[QW_GLYPH + 1] = (uint32_t)(ap >> 32);
		r.w[QW_GLYPH + 2] = fontOffset;
		r.w[QW_GLYPH + 3] = pitch;
		r.w[QW_GLYPH + 4] = (uint32_t)fw;
		r.w[QW_GLYPH + 5] = (uint32_t)fh;
		r.w[QW_GLYPH + 6] = f2u(qx0);
		r.w[QW_GLYPH + 7] = f2u(qy0);
		r.w[QW_GLYPH + 8] = f2u(fho);
		r.w[QW_GLYPH + 9] = (uint32_t)((size_t)f.w * f.h);
		int rc = record_raw(c, r);
		if (rc) return rc;
	}
	return DTR_B200_OK;
}

int dtr_b200_set_debug_markers(dtr_b200_ctx *c, int enable)
{
	if (!c) return DTR_B200_ERR_ARG;
	c->debugMarkers = enable != 0;
	return DTR_B200_OK;
}

int dtr_b200_rectangle(dtr_b200_ctx *c, const float mn[2], const float mx[2], const float color[4],
                       const dtr_b200_transform *t)
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!mn || !mx || !color) return DTR_B200_OK;
	if (!t) t = &kDefaultTransform;
	return emit_rectangle(c, mn, mx, color, t);
}
int dtr_b200_bitmap(dtr_b200_ctx *c, int texId, const float pos[2], const dtr_b200_transform *t, const float color[4])
{
	if (!c) return DTR_B200_ERR_ARG;
	if (!pos) return DTR_B200_OK;
	if (texId < 0 || texId >= (int)c->textures.size()) return fail(c, DTR_B200_ERR_ARG, "texId out of range");
	if (!t) t = &kDefaultTransform;
	const float white[4] = {1, 1, 1, 1};
	if (!color) color = white;
	const TexDesc &td    = c->textures[texId];
	float          mn[2] = {pos[0], pos[1]};
	float          mx[2] = {pos[0] + (float)td.w, pos[1] + (float)td.h}; // min + dim (:1607-1608)
	PrimRecord     r;
	float          pts[4][2], bounds[4];
	int            rc = 0;
	if (setup_quad(c->width, c->height, mn, mx, t->rotation, t->anchor, t->scale, color, true, texId, td.w, td.h, &r, pts, bounds))
		rc = record_raw(c, r);
	if (rc || !c->debugMarkers) return rc;
	// DebugRenderMarkers(pList, 4, transform, bbox, basis, vertex markers) (:719-771, :1783-1790):
	// red bounding box; the basis is only drawn for 3-point lists; a 10x10 rectangle per corner in
	// green, blue, purple, red -- each of which draws its own debug bounding box in turn
	const float red[4] = {1, 0, 0, 1};
	if ((rc = emit_bbox_lines(c, bounds, red))) return rc;
	const float markerColor[4][4] = {{0, 1, 0, 1}, {0, 0, 1, 1}, {1, 0, 1, 1}, {1, 0, 0, 1}};
	for (int i = 0; i < 4 && !rc; i++)
	{
		const float a[2] = {pts[i][0] - 5.0f, pts[i][1] - 5.0f}, b[2] = {pts[i][0] + 5.0f, pts[i][1] + 5.0f};
		rc = emit_rectangle(c, a, b, markerColor[i], &kDefaultTransform);
	}
	return rc;
}

} // extern "C"
