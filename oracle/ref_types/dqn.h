// Stand-in for the original DTRenderer's dqn.h -- TEST INFRASTRUCTURE ONLY (see oracle/Makefile, target ref).
// Declares just the Dqn types and helpers that ref_b200_harness.cpp and dtrenderer_b200/host/DTRRenderB200.h use,
// with the original's member names, so the drop-in mirror can be built and checked where the original's sources
// are not present.  Where they are, the harness is built against the real headers instead.
#ifndef DTRO_STANDIN_DQN_H
#define DTRO_STANDIN_DQN_H

#include <float.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

typedef uint8_t  u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t  i32;
typedef float    f32;

#define DQN_MEGABYTE(x) ((size_t)(x) * 1024 * 1024)
#define DQN_F32_MIN -FLT_MAX

union DqnV2  { struct { f32 x, y; }; struct { f32 w, h; }; f32 e[2]; };
union DqnV2i { struct { i32 x, y; }; struct { i32 w, h; }; struct { i32 min, max; }; i32 e[2]; };
union DqnV3  { struct { f32 x, y, z; }; struct { f32 r, g, b; }; f32 e[3]; };
union DqnV4  { struct { f32 x, y, z, w; }; struct { f32 r, g, b, a; }; f32 e[4]; };

inline DqnV2  DqnV2_2f(f32 x, f32 y) { DqnV2 r; r.x = x; r.y = y; return r; }
inline DqnV2i DqnV2i_2i(i32 x, i32 y) { DqnV2i r; r.x = x; r.y = y; return r; }
inline DqnV3  DqnV3_3f(f32 x, f32 y, f32 z) { DqnV3 r; r.x = x; r.y = y; r.z = z; return r; }
inline DqnV4  DqnV4_4f(f32 x, f32 y, f32 z, f32 w) { DqnV4 r; r.x = x; r.y = y; r.z = z; r.w = w; return r; }

struct DqnMemStack { u8 *memory; size_t size; };
inline bool DqnMemStack_Init(DqnMemStack *s, size_t size, bool zero)
{
	s->memory = (u8 *)(zero ? calloc(1, size) : malloc(size));
	s->size   = s->memory ? size : 0;
	return s->memory != NULL;
}
inline void DqnMemStack_Free(DqnMemStack *s) { free(s->memory); s->memory = NULL; s->size = 0; }

#endif
