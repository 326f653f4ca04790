// Stand-in for the original DTRenderer's DTRendererRender.h (with the asset types it pulls in) -- TEST
// INFRASTRUCTURE ONLY, see dqn.h here.  Only the members the harness and the mirror use are declared.
// DTRMeshFace and stbtt_packedchar are handed to the C ABI as they are, so they must have the original's
// layout; DTRRenderB200.h checks both against dtr_b200_mesh_face and dtr_b200_packedchar.
#ifndef DTRO_STANDIN_DTRENDERER_RENDER_H
#define DTRO_STANDIN_DTRENDERER_RENDER_H

#include "dqn.h"

struct DTRRenderBuffer;
struct PlatformAPI;
struct PlatformJobQueue;

struct stbtt_packedchar { u16 x0, y0, x1, y1; f32 xoff, yoff, xadvance, xoff2, yoff2; };

struct DTRBitmap { u8 *memory; DqnV2i dim; i32 bytesPerPixel; };

struct DTRFont { u8 *bitmap; DqnV2i bitmapDim; DqnV2i codepointRange; stbtt_packedchar *atlas; };

struct DTRMeshFace
{
	i32 *vertexIndex; u32 numVertexIndex;
	i32 *texIndex;    u32 numTexIndex;
	i32 *normalIndex; u32 numNormalIndex;
};

struct DTRMesh
{
	DqnV4 *vertexes; DqnV3 *texUV; DqnV3 *normals; DTRMeshFace *faces;
	u32 numVertexes, numTexUV, numNormals, numFaces;
	DTRBitmap tex;
};

struct DTRRenderTransform { f32 rotation; DqnV3 anchor; DqnV3 scale; };

inline DTRRenderTransform DTRRender_DefaultTransform()
{
	DTRRenderTransform r = {0.0f, DqnV3_3f(0.5f, 0.5f, 0.5f), DqnV3_3f(1, 1, 1)};
	return r;
}

inline DTRRenderTransform DTRRender_DefaultTriangleTransform()
{
	DTRRenderTransform r = {0.0f, DqnV3_3f(0.33f, 0.33f, 0.33f), DqnV3_3f(1, 1, 1)};
	return r;
}

enum DTRRenderShadingMode { DTRRenderShadingMode_FullBright, DTRRenderShadingMode_Flat, DTRRenderShadingMode_Gouraud };

struct DTRRenderLight { enum DTRRenderShadingMode mode; DqnV3 vector; DqnV4 color; };

struct DTRRenderContext
{
	DTRRenderBuffer  *renderBuffer;
	DqnMemStack      *tempStack;
	PlatformAPI      *api;
	PlatformJobQueue *jobQueue;
	bool              multithread;
};

#endif
