// Stand-in for the original DTRenderer's DTRenderer.h (and the platform types it pulls in) -- TEST
// INFRASTRUCTURE ONLY, see dqn.h here.
#ifndef DTRO_STANDIN_DTRENDERER_H
#define DTRO_STANDIN_DTRENDERER_H

#include "DTRendererRender.h"

struct PlatformLock;
struct PlatformFlags { bool canUseSSE2, canUseRdtsc; };
struct PlatformAPI { void *unused; };

struct DTRRenderBuffer
{
	i32 width, height, bytesPerPixel;
	PlatformLock *renderLock;
	volatile u8 *memory;
	volatile f32 *zBuffer;
	volatile bool *pixelLockTable;
};

#endif
