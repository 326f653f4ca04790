// dtr_deferred.cuh -- the deferred variant of the raster stage, included by dtr_kernels.cu.
//
// When EVERY primitive of a pass is an opaque triangle (colour alpha 1, no texture or a texture whose
// texels all have alpha 255) and every frame of the pass starts from an on-chip clear, the colour a
// pixel ends up with is the shading of the LAST fragment that passed the depth test there -- nothing is
// ever blended.  The pass then runs visibility first and shades every visible pixel ONCE (instead of once
// per depth-test pass: 1.5 x fewer on the sphere), in one of two forms (dtr_b200_set_opaque_stage):
//
//   raster_opaque_kernel<true>   (default) the same region walk as raster_kernel (list walk, depth culls,
//                       lane-parallel setup, sub-block classification, fp32 table coverage step, strict->
//                       depth test), but a passing fragment only leaves its primitive's index in the
//                       colour tile (0x80000000 | index; finished colours have a zero top byte).  No
//                       fragment queue, no shading slots: 9.3 KB of shared memory per warp and 80
//                       registers, i.e. SIX resident CTAs per SM instead of five, and a coverage step
//                       without the queue write.  When a region's walk is over, the warp that owns it
//                       shades the pixels that still carry an index -- from shared memory, two sub-blocks
//                       per step as two interleaved instruction streams (the walk's registers are free by
//                       then) -- and writes the region back once, finished.  The int32 edge functions are
//                       re-evaluated at the pixel from the record (exact, so the same bits as in the
//                       coverage step), then the reference's arithmetic (SlowTriangle :1177-1222) in the
//                       reference's order.  SetPixel calls are counted in the walk (every fragment that
//                       passes the depth test is one, whether or not it survives).
//   raster_opaque_kernel<false> + resolve_kernel   the walk alone (the region is written back with its
//                       pending indices), then one thread per pixel of the tiles that have primitives
//                       shades the pixels that still carry an index: full occupancy, coalesced, but a
//                       second pass over the busy tiles and a second kernel.  (The first form of the
//                       stage; kept selectable: it is the measured baseline of the one-kernel form.)
//
// Triangle id planes (RasterParams::ids): the IDS instantiations keep an id tile per warp beside the tag tile
// and write it back with the region; the ids are final then, so resolve_kernel needs no id logic.
//
// Inexact triangles (sequential fp32 accumulation, see raster_tri_replay) cannot be re-evaluated per
// pixel without their accumulation order; their fragments are shaded at once in the walk (a
// __noinline__ call on a path that ~2 % of mesh triangles take) and stored as finished colours.
#pragma once

struct VisSmem
{
	uint32_t c[REGION_WORDS];   // finished colour (top byte 0) or 0x80000000 | primitive index
	float    z[REGION_WORDS];
	int      zk[32];            // depth bound (key) of the 32 list entries of the current chunk
	uint4    geo[GROUP * 5];    // {E1o,E2o,E3o,bbox} {dx1,dx2,dx3,flags} {dy1,dy2,dy3,rel | index} {Emax1,Emax2,Emax3,zkey} {1/area,z1,dz2,dz3}
	uint4    sub[32];           // current triangle, per sub-block: {E1,E2,E3 at its origin as fp32 (exact), in-bbox pixel mask}
};
constexpr int      VIS_CTAS_PER_SM = 6;
constexpr int      VIS_IDS_CTAS_PER_SM = 4; // the id-plane variants: what their shared memory (VisSmem + IdSmem per warp) allows
constexpr uint32_t VIS_EMPTY_SHIFT = 0; // (2: no gain) log2 of the untouched tiles per work item of a large launch
constexpr uint32_t VIS_OUTSIDE     = 0x40000000u; // resolve_kernel: a pixel of the tile that lies outside the frame (no colour has this bit)

// The reference's per-fragment arithmetic after the depth test for an OPAQUE fragment (SlowTriangle
// :1177-1222, SetPixel :124-191 with a == 1): barycentrics, Gouraud, nearest texel, modulate, gamma-2
// store.  `rec` is the triangle's 160-byte record (any address space), e1..e3 its edge functions at
// the pixel.  Returns the packed 0x00RRGGBB pixel.
__device__ __forceinline__ uint32_t shade_opaque_from_record(const uint4 *rec, const float e1, const float e2, const float e3)
{
	const float4   a4  = u2f4(rec[4]); // 1/area, z1, dz2, dz3
	const float4   c   = u2f4(rec[5]); // linear premultiplied colour
	const uint4    a6  = rec[6];       // red light products, flags | texId << 8
	const uint32_t ft  = a6.w;
	const float    inv = a4.x;
	const float    bA = e1 * inv, bB = e2 * inv, bC = e3 * inv;
	const bool     grey = (ft & PF_GREY) != 0;
	float          fr = c.x, fg = c.y, fb = c.z;
	if (!(ft & PF_IGNORE_LIGHT))
	{
		const float lr = ((__uint_as_float(a6.x) * bA) + (__uint_as_float(a6.y) * bB)) + (__uint_as_float(a6.z) * bC);
		fr = fr * lr;
		if (grey)
		{
			fg = fr; fb = fr; // same operands, same bits
		}
		else
		{
			const float4 a7 = u2f4(rec[7]);
			const float4 a8 = u2f4(rec[8]);
			const float  lg = ((a7.x * bA) + (a7.y * bB)) + (a7.z * bC);
			const float  lb = ((a7.w * bA) + (a8.x * bB)) + (a8.y * bC);
			fg = fg * lg; fb = fb * lb;
		}
	}
	const bool textured = (ft & PF_TEXTURED) != 0;
	if (textured)
	{
		const uint4  t0 = rec[3]; // dy3, texels lo, texels hi, w | h << 16
		const float4 a8 = u2f4(rec[8]), a9 = u2f4(rec[9]);
		float u = (a8.z + (a9.x * bB)) + (a9.z * bC);
		float v = (a8.w + (a9.y * bB)) + (a9.w * bC);
		u = __saturatef(u); // DqnMath_Clampf(v, 0, 1): see texel_issue
		v = __saturatef(v);
		const uint32_t *texels = reinterpret_cast<const uint32_t *>(((unsigned long long)t0.z << 32) | t0.y);
		const uint32_t  texW = t0.w & 0xFFFFu, texH = t0.w >> 16;
		const uint32_t  tx = (uint32_t)(int)(u * (float)texW), ty = (uint32_t)(int)(v * (float)texH); // NEAREST
		const Texel     t = texel_linear(__ldg(texels + (ty * texW + tx)));
		fr = fr * t.r; fg = fg * t.g; fb = fb * t.b; // (alpha: 1 * 1, the fragment is opaque by construction)
	}
	if (grey && !textured) return out_byte(fr) * 0x010101u;
	return (out_byte(fr) << 16) | (out_byte(fg) << 8) | out_byte(fb);
}

// the rare path of the visibility kernel: a fragment of an INEXACT triangle, shaded at once
__device__ __noinline__ uint32_t shade_opaque_now(const PrimRecord *rec, float e1, float e2, float e3)
{
	return shade_opaque_from_record(reinterpret_cast<const uint4 *>(rec), e1, e2, e3);
}

// N pixels at once, for instruction-level parallelism: the same operations in the same order per pixel
// as shade_opaque_from_record, written side by side so that the N dependency chains (and the N texel
// fetches) overlap.  The pixels' triangles must agree in the flags that select the code path; if they
// do not (two kinds of triangle meet in one lane's group), the pixels are shaded one after the other.
template <int N>
__device__ __forceinline__ void shade_opaque_wide(const uint4 *const (&rec)[N], const float (&e1)[N], const float (&e2)[N],
                                                  const float (&e3)[N], uint32_t (&out)[N])
{
	float4 a4[N], c[N];
	uint4  a6[N];
#pragma unroll
	for (int k = 0; k < N; k++)
	{
		a4[k] = ldg4f(rec[k] + 4);
		c[k]  = ldg4f(rec[k] + 5);
		a6[k] = __ldg(rec[k] + 6);
	}
	const uint32_t ft = a6[0].w;
	uint32_t       differ = 0u;
#pragma unroll
	for (int k = 1; k < N; k++) differ |= ft ^ a6[k].w;
	if (differ & (PF_GREY | PF_IGNORE_LIGHT | PF_TEXTURED))
	{
#pragma unroll
		for (int k = 0; k < N; k++) out[k] = shade_opaque_now(reinterpret_cast<const PrimRecord *>(rec[k]), e1[k], e2[k], e3[k]); // (a call: rare)
		return;
	}
	float bA[N], bB[N], bC[N], fr[N], fg[N], fb[N];
#pragma unroll
	for (int k = 0; k < N; k++)
	{
		const float inv = a4[k].x;
		bA[k] = e1[k] * inv; bB[k] = e2[k] * inv; bC[k] = e3[k] * inv;
		fr[k] = c[k].x; fg[k] = c[k].y; fb[k] = c[k].z;
	}
	const bool grey = (ft & PF_GREY) != 0;
	if (!(ft & PF_IGNORE_LIGHT))
	{
#pragma unroll
		for (int k = 0; k < N; k++)
		{
			const float lr = ((__uint_as_float(a6[k].x) * bA[k]) + (__uint_as_float(a6[k].y) * bB[k])) + (__uint_as_float(a6[k].z) * bC[k]);
			fr[k] = fr[k] * lr;
		}
		if (grey)
		{
#pragma unroll
			for (int k = 0; k < N; k++) { fg[k] = fr[k]; fb[k] = fr[k]; } // same operands, same bits
		}
		else
		{
#pragma unroll
			for (int k = 0; k < N; k++)
			{
				const float4 q7 = ldg4f(rec[k] + 7);
				const float4 q8 = ldg4f(rec[k] + 8);
				const float  lg = ((q7.x * bA[k]) + (q7.y * bB[k])) + (q7.z * bC[k]);
				const float  lb = ((q7.w * bA[k]) + (q8.x * bB[k])) + (q8.y * bC[k]);
				fg[k] = fg[k] * lg; fb[k] = fb[k] * lb;
			}
		}
	}
	const bool textured = (ft & PF_TEXTURED) != 0;
	if (textured)
	{
		uint32_t tw[N];
#pragma unroll
		for (int k = 0; k < N; k++)
		{
			const uint4  t  = __ldg(rec[k] + 3); // dy3, texels lo, texels hi, w | h << 16
			const float4 q8 = ldg4f(rec[k] + 8), q9 = ldg4f(rec[k] + 9);
			float u = (q8.z + (q9.x * bB[k])) + (q9.z * bC[k]);
			float v = (q8.w + (q9.y * bB[k])) + (q9.w * bC[k]);
			u = __saturatef(u); // DqnMath_Clampf(v, 0, 1): see texel_issue
			v = __saturatef(v);
			const uint32_t *texels = reinterpret_cast<const uint32_t *>(((unsigned long long)t.z << 32) | t.y);
			const uint32_t  texW = t.w & 0xFFFFu, texH = t.w >> 16;
			const uint32_t  tx = (uint32_t)(int)(u * (float)texW), ty = (uint32_t)(int)(v * (float)texH); // NEAREST
			tw[k] = __ldg(texels + (ty * texW + tx));
		}
#pragma unroll
		for (int k = 0; k < N; k++)
		{
			const Texel tl = texel_linear(tw[k]);
			fr[k] = fr[k] * tl.r; fg[k] = fg[k] * tl.g; fb[k] = fb[k] * tl.b; // (alpha: 1 * 1, the fragment is opaque by construction)
		}
	}
	if (grey && !textured)
	{
#pragma unroll
		for (int k = 0; k < N; k++) out[k] = out_byte(fr[k]) * 0x010101u;
	}
	else
	{
#pragma unroll
		for (int k = 0; k < N; k++) out[k] = (out_byte(fr[k]) << 16) | (out_byte(fg[k]) << 8) | out_byte(fb[k]);
	}
}


// One region of the visibility pass (see process_region for the walk; only the differences are commented).
// FUSED: the pending pixels of the finished region are shaded HERE, from shared memory, before the region
// is written back (see raster_visres_kernel); the region then leaves the SM with finished colours only.
// IDS: the triangle ids as well, in I->t, set where a fragment sets its depth (and its tag, or its colour).
template <bool FUSED, bool IDS = false>
__device__ __forceinline__ void process_region_vis(const RasterParams &P, VisSmem &W, IdSmem *I, const int lane, const RegionJob &J,
                                                   uint32_t &shaded, uint32_t &nextItem)
{
	const uint32_t FULL = 0xffffffffu, ltMask = (1u << lane) - 1u;
	const int      gx = J.gx, gy = J.gy, width = P.g.width, height = P.g.height;
	const int      rx1 = min(gx + REGION_W, width), ry1 = min(gy + J.rows, height);
	const int      subsY = J.rows / SUB_H, regionWords = REGION_W * J.rows;
	const bool     vec = (width & 3) == 0;
	const float    zInit = -FLT_MAX;
	const int      vr = (lane >> 1) & 3, vx = (lane >> 3) * SUB_W + (lane & 1) * 4;
	const int      vsi = lane * 4;
	uint32_t *const gI = IDS ? P.ids + (J.gZ - P.depth) : nullptr; // the region's frame in the id planes

	if (J.count == 0)
	{
		if (lane == 0) nextItem = atomicAdd(P.workCounter, 1u);
		if (vec)
		{
			const uint4  c4 = make_uint4(J.clearPacked, J.clearPacked, J.clearPacked, J.clearPacked);
			const float4 z4 = make_float4(zInit, zInit, zInit, zInit);
#pragma unroll 4
			for (int i = 0; i < subsY; i++)
			{
				const int y = gy + 4 * i + vr, x = gx + vx;
				if (y < height && x < width)
				{
					const size_t gi = (size_t)y * width + x;
					if (J.genC) frame_store(reinterpret_cast<uint4 *>(J.gC + gi), c4);
					if (J.genZ) frame_store(reinterpret_cast<float4 *>(J.gZ + gi), z4);
					if (IDS && J.genZ) frame_store(reinterpret_cast<uint4 *>(gI + gi), make_uint4(0u, 0u, 0u, 0u));
				}
			}
		}
		else
		{
			for (int i = lane; i < regionWords; i += 32)
			{
				const int x = gx + (i & (REGION_W - 1)), y = gy + i / REGION_W;
				if (x < width && y < height)
				{
					const size_t gi = (size_t)y * width + x;
					if (J.genC) J.gC[gi] = J.clearPacked;
					if (J.genZ) J.gZ[gi] = zInit;
					if (IDS && J.genZ) gI[gi] = 0u;
				}
			}
		}
		return;
	}

	// ---- load / generate the region (a deferred pass always generates the colour: genC) ------------
	const size_t vOff  = (size_t)(gy + vr) * width + (gx + vx);
	const int    vRows = (gx + vx < width) ? (height - (gy + vr) + 3) >> 2 : 0;
	if (vec)
	{
		const float4 *pz = reinterpret_cast<const float4 *>(J.gZ + vOff);
		uint32_t     *sc = W.c + vsi;
		float        *sz = W.z + vsi;
#pragma unroll 4
		for (int i = 0; i < subsY; i++)
		{
			const bool in = i < vRows;
			float4     z4 = make_float4(zInit, zInit, zInit, zInit);
			if (!J.genZ && in) z4 = *pz;
			*reinterpret_cast<uint4 *>(sc)  = make_uint4(J.clearPacked, J.clearPacked, J.clearPacked, J.clearPacked);
			*reinterpret_cast<float4 *>(sz) = z4;
			pz += width;
			sc += SUBS_X * 32;
			sz += SUBS_X * 32;
		}
		if (IDS)
		{
			const uint4 *pi = reinterpret_cast<const uint4 *>(gI + vOff);
			uint32_t    *si = I->t + vsi;
#pragma unroll 4
			for (int i = 0; i < subsY; i++)
			{
				uint4 i4 = make_uint4(0u, 0u, 0u, 0u);
				if (!J.genZ && i < vRows) i4 = *pi;
				*reinterpret_cast<uint4 *>(si) = i4;
				pi += width;
				si += SUBS_X * 32;
			}
		}
	}
	else
	{
		for (int i = lane; i < regionWords; i += 32)
		{
			const int    rx = i & (REGION_W - 1), ry = i / REGION_W, x = gx + rx, y = gy + ry;
			const bool   in = (x < width && y < height);
			const size_t gi = (size_t)y * width + x;
			const int    si = pix_index((ry >> 2) * SUBS_X + (rx >> 3), ((ry & 3) << 3) + (rx & 7));
			W.c[si] = J.clearPacked;
			W.z[si] = (J.genZ || !in) ? zInit : J.gZ[gi];
			if (IDS) I->t[si] = (J.genZ || !in) ? 0u : gI[gi];
		}
	}
	__syncwarp();

	int zsub = depth_key(-FLT_MAX);
	uint32_t       passes  = 0; // this LANE's fragments that passed the depth test = SetPixel calls (summed once per warp at the end of the kernel: no vote in the coverage step)
	const uint32_t laneBit = 1u << lane;
	const uint32_t zAddrLane = (uint32_t)__cvta_generic_to_shared(W.z + lane);
	const uint32_t cAddrLane = (uint32_t)__cvta_generic_to_shared(W.c + lane);
	const uint32_t iAddrLane = IDS ? (uint32_t)__cvta_generic_to_shared(I->t + lane) : 0u;
	const int      lx = lane & 7, ly = lane >> 3;
	const int      sxo = (lane & 3) * SUB_W, syo = (lane >> 2) * SUB_H;

	// exact triangle: classification and table as in raster_tri; a passing fragment writes its depth
	// and its primitive's tag, nothing else
	auto raster_tri = [&](const uint4 g0, const uint4 g1, const uint4 g2, const uint4 g3, const uint4 g4, const uint32_t id) {
		const int      x0 = g0.w & 0xFF, y0 = (g0.w >> 8) & 0xFF, x1 = (g0.w >> 16) & 0xFF, y1 = g0.w >> 24;
		const float4   zp  = u2f4(g4); // 1/area, z1, z2-z1, z3-z1
		const uint32_t tag = VIS_PENDING | g2.w;
		uint32_t       cand;
		float          V1, V2, V3;
		{
			const int dx1 = (int)g1.x, dx2 = (int)g1.y, dx3 = (int)g1.z;
			const int dy1 = (int)g2.x, dy2 = (int)g2.y, dy3 = (int)g2.z;
			const int B1 = sxo * dx1 + syo * dy1, B2 = sxo * dx2 + syo * dy2, B3 = sxo * dx3 + syo * dy3;
			bool keep = (sxo < x1) && (sxo + SUB_W > x0) && (syo < y1) && (syo + SUB_H > y0);
			keep = keep && ((((int)g3.x + B1) | ((int)g3.y + B2) | ((int)g3.z + B3)) >= 0);
			keep = keep && ((int)g3.w > zsub);
			const int      nx = min(max(x1 - sxo, 0), SUB_W), ny = min(max(y1 - syo, 0), SUB_H);
			const uint32_t inMask = (((1u << nx) - 1u) * 0x01010101u) & (ny >= SUB_H ? 0xffffffffu : ((1u << (8 * ny)) - 1u));
			__syncwarp();
			W.sub[lane] = make_uint4(__float_as_uint((float)((int)g0.x + B1)), __float_as_uint((float)((int)g0.y + B2)),
			                         __float_as_uint((float)((int)g0.z + B3)), inMask);
			V1 = (float)(lx * dx1 + ly * dy1);
			V2 = (float)(lx * dx2 + ly * dy2);
			V3 = (float)(lx * dx3 + ly * dy3);
			cand = __ballot_sync(FULL, keep);
		}
		__syncwarp();
		while (cand)
		{
			uint32_t s, sBit;
			asm("bfind.u32 %0, %1;" : "=r"(s) : "r"(cand));
			asm("bmsk.clamp.b32 %0, %1, 1;" : "=r"(sBit) : "r"(s));
			cand ^= sBit;
			const uint4    sb = W.sub[s];
			const uint32_t za = zAddrLane + (s << 7), ca = cAddrLane + (s << 7);
			float          zOld;
			asm volatile("ld.shared.f32 %0, [%1];" : "=f"(zOld) : "r"(za) : "memory");
			const float e1 = __uint_as_float(sb.x) + V1, e2 = __uint_as_float(sb.y) + V2, e3 = __uint_as_float(sb.z) + V3;
			const bool  covered = (sb.w & laneBit) && ((__float_as_int(e1) | __float_as_int(e2) | __float_as_int(e3)) >= 0);
			const float bB = e2 * zp.x, bC = e3 * zp.x;
			const float z  = (zp.y + (bB * zp.z)) + (bC * zp.w);
			const bool  pass = covered & (z > zOld);
			asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t@q st.shared.f32 [%1], %2;\n\t@q st.shared.u32 [%3], %4;\n\t}"
			             :
			             : "r"((uint32_t)pass), "r"(za), "f"(z), "r"(ca), "r"(tag)
			             : "memory");
			if (IDS) asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %0, 0;\n\t@q st.shared.u32 [%1], %2;\n\t}" : : "r"((uint32_t)pass), "r"(iAddrLane + (s << 7)), "r"(id) : "memory");
			passes += pass ? 1u : 0u;
		}
	};

	// inexact triangle: the row-shared replay of raster_tri_replay; fragments are shaded at once
	auto raster_tri_replay = [&](const uint32_t pidx, const uint4 g0, const uint4 g1, const uint4 g2, const uint4 g4, const uint32_t id) {
		const int    x0 = g0.w & 0xFF, y0 = (g0.w >> 8) & 0xFF, x1 = (g0.w >> 16) & 0xFF, y1 = g0.w >> 24;
		const float4 zp = u2f4(g4);
		const float  fdx1 = __uint_as_float(g1.x), fdx2 = __uint_as_float(g1.y), fdx3 = __uint_as_float(g1.z);
		const float  fdy1 = __uint_as_float(g2.x), fdy2 = __uint_as_float(g2.y), fdy3 = __uint_as_float(g2.z);
		const int    minx = (int)(g2.w & 0xFFFFu), miny = (int)(g2.w >> 16); // bbox origin (the tag word carries it for inexact triangles)
		const int    relx = gx - minx, rely = gy - miny;
		float        R1 = __uint_as_float(g0.x), R2 = __uint_as_float(g0.y), R3 = __uint_as_float(g0.z);
		{
			const int ny = lane + rely;
			for (int k = 0; k < ny; k++) { R1 = R1 + fdy1; R2 = R2 + fdy2; R3 = R3 + fdy3; }
			const int nx0 = max(relx, 0);
			for (int k = 0; k < nx0; k++) { R1 = R1 + fdx1; R2 = R2 + fdx2; R3 = R3 + fdx3; }
		}
		const int  colBias = min(relx, 0);
		const bool keep = (sxo < x1) && (sxo + SUB_W > x0) && (syo < y1) && (syo + SUB_H > y0);
		uint32_t   cand = __ballot_sync(FULL, keep);
		while (cand)
		{
			const int s = 31 - __clz(cand);
			cand &= ~(1u << s);
			const int  col = (s & 3) * SUB_W + lx, row = (s >> 2) * SUB_H + ly;
			float      e1 = __shfl_sync(FULL, R1, row), e2 = __shfl_sync(FULL, R2, row), e3 = __shfl_sync(FULL, R3, row);
			const bool inb = (col >= x0) && (col < x1) && (row >= y0) && (row < y1);
			const int  na = inb ? col + colBias : 0;
			for (int k = 0; k < na; k++) { e1 = e1 + fdx1; e2 = e2 + fdx2; e3 = e3 + fdx3; }
			const bool  covered = inb && e1 >= 0.0f && e2 >= 0.0f && e3 >= 0.0f;
			const int   si = (s << 5) | lane;
			const float bB = e2 * zp.x, bC = e3 * zp.x;
			const float z  = (zp.y + (bB * zp.z)) + (bC * zp.w);
			const bool  pass = covered && (z > W.z[si]);
			if (pass)
			{
				W.z[si] = z;
				W.c[si] = shade_opaque_now(P.prims + pidx, e1, e2, e3);
				if (IDS) I->t[si] = id;
				passes++;
			}
		}
		__syncwarp();
	};

	uint32_t zcState = J.genZ ? 1u : 0u;
	for (uint32_t base = 0; base < J.count; base += 32)
	{
		const uint32_t e    = base + lane;
		uint32_t       pidx = 0;
		bool           ov   = false;
		if (e < J.count)
		{
			const uint32_t le = J.listOff + e;
			pidx          = __ldg(P.lists + le);
			const uint2 b = __ldg(P.listBounds + le);
			W.zk[lane]    = __ldg(P.listZ + le);
			const int minx = b.x & 0xFFFF, miny = b.x >> 16, maxx = b.y & 0xFFFF, maxy = b.y >> 16;
			ov = (minx < rx1) && (maxx > gx) && (miny < ry1) && (maxy > gy);
		}
		uint32_t m = __ballot_sync(FULL, ov);
		while (m)
		{
			if ((zcState & 0xFFu) == 0u)
			{
				const float4 *z4 = reinterpret_cast<const float4 *>(W.z);
				int mySub = DEPTH_KEY_UNKNOWN;
				for (int k = 0; k < regionWords / 128; k++)
				{
					const float4 q = z4[lane + 32 * k];
					float        v = fminf(fminf(q.x, q.y), fminf(q.z, q.w));
					v = fminf(v, __shfl_xor_sync(FULL, v, 1));
					v = fminf(v, __shfl_xor_sync(FULL, v, 2));
					v = fminf(v, __shfl_xor_sync(FULL, v, 4));
					const float t = __shfl_sync(FULL, v, (lane & 3) * 8);
					if ((lane >> 2) == k) mySub = depth_key(t);
				}
				zsub = mySub;
				const int zminKey = __reduce_min_sync(FULL, mySub);
				const uint32_t hidden  = __ballot_sync(FULL, W.zk[lane] <= zminKey) & m;
				const uint32_t prev    = zcState >> 8;
				const uint32_t backoff = ((uint32_t)__popc(hidden) >= ZCULL_RESET) ? 0u : (hidden ? prev : min(2u * prev + 1u, ZCULL_MAX_BACKOFF));
				zcState = backoff | (backoff << 8);
				m &= ~hidden;
				if (!m) break;
			}
			else zcState--;
			const bool     ing = ((m >> lane) & 1u) && (__popc(m & ltMask) < GROUP);
			const uint32_t gm  = __ballot_sync(FULL, ing);
			m &= ~gm;
			if (((m >> lane) & 1u) && (__popc(m & ltMask) < GROUP))
				asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char *>(P.prims + pidx))); // (only the first 128 bytes are used here)
			// five quads per triangle instead of eleven: geometry and the depth plane, no shading data
			bool  live = ing;
			uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0, q2 = q0, q3 = q0, q4 = q0, g0 = q0;
			int   relx = 0, rely = 0;
			if (ing)
			{
				const uint4 *rec = reinterpret_cast<const uint4 *>(P.prims + pidx);
				q0 = __ldg(rec); q1 = __ldg(rec + 1); q2 = __ldg(rec + 2); q3 = __ldg(rec + 3); q4 = __ldg(rec + 4);
				const int minx = q0.z & 0xFFFF, miny = q0.z >> 16, maxx = q0.w & 0xFFFF, maxy = q0.w >> 16;
				const int x0 = max(minx, gx) - gx, y0 = max(miny, gy) - gy;
				const int x1 = min(maxx, rx1) - gx, y1 = min(maxy, ry1) - gy;
				relx = gx - minx; rely = gy - miny;
				g0   = make_uint4(q1.x, q1.y, q1.z, (uint32_t)x0 | ((uint32_t)y0 << 8) | ((uint32_t)x1 << 16) | ((uint32_t)y1 << 24));
				if ((q0.x & PF_TYPE_MASK) != PRIM_TRI) live = false; // (cannot happen: the host only defers passes made of triangles)
				else if (q0.x & PF_EXACT)
				{
					g0.x = (uint32_t)((int)q1.x + relx * (int)q1.w + rely * (int)q2.z);
					g0.y = (uint32_t)((int)q1.y + relx * (int)q2.x + rely * (int)q2.w);
					g0.z = (uint32_t)((int)q1.z + relx * (int)q2.y + rely * (int)q3.x);
					const int xa = x0, xb = x1 - 1, ya = y0, yb = y1 - 1;
					const int m1 = (int)g0.x + max(xa * (int)q1.w, xb * (int)q1.w) + max(ya * (int)q2.z, yb * (int)q2.z);
					const int m2 = (int)g0.y + max(xa * (int)q2.x, xb * (int)q2.x) + max(ya * (int)q2.w, yb * (int)q2.w);
					const int m3 = (int)g0.z + max(xa * (int)q2.y, xb * (int)q2.y) + max(ya * (int)q3.x, yb * (int)q3.x);
					live = (m1 | m2 | m3) >= 0;
				}
			}
			const uint32_t lm = __ballot_sync(FULL, live);
			const int      ng = __popc(lm);
			if (live)
			{
				const int  r     = __popc(lm & ltMask);
				const bool exact = (q0.x & PF_EXACT) != 0;
				W.geo[r * 5 + 0] = g0;
				W.geo[r * 5 + 1] = make_uint4(q1.w, q2.x, q2.y, q0.x & 0xFFFFu);
				// exact: the primitive's index (the tag a fragment leaves); inexact: the bbox origin, and the index travels in g3.w
				W.geo[r * 5 + 2] = make_uint4(q2.z, q2.w, q3.x, exact ? pidx : q0.z);
				W.geo[r * 5 + 3] = make_uint4(
				    g0.x + (uint32_t)((SUB_W - 1) * max((int)q1.w, 0) + (SUB_H - 1) * max((int)q2.z, 0)),
				    g0.y + (uint32_t)((SUB_W - 1) * max((int)q2.x, 0) + (SUB_H - 1) * max((int)q2.w, 0)),
				    g0.z + (uint32_t)((SUB_W - 1) * max((int)q2.y, 0) + (SUB_H - 1) * max((int)q3.x, 0)),
				    exact ? (uint32_t)W.zk[lane] : pidx);
				W.geo[r * 5 + 4] = q4;
				if (IDS) I->geo[r] = __ldg(P.primId + pidx);
			}
			__syncwarp();
			for (int r = 0; r < ng; r++)
			{
				const uint4    g0r = W.geo[r * 5], g1 = W.geo[r * 5 + 1], g2 = W.geo[r * 5 + 2], g3 = W.geo[r * 5 + 3], g4 = W.geo[r * 5 + 4];
				const uint32_t id = IDS ? I->geo[r] : 0u;
				if (g1.w & PF_EXACT) raster_tri(g0r, g1, g2, g3, g4, id);
				else raster_tri_replay(g3.w, g0r, g1, g2, g4, id);
			}
			__syncwarp();
		}
	}
	shaded += passes;

	if (FUSED)
	{
		// ---- resolve in place ------------------------------------------------------------------------
		// The same arithmetic as resolve_kernel (int32 edge functions re-evaluated at the pixel from the
		// record, then the reference's shading); lane = pixel of a sub-block.  The lanes of an 8x4 block
		// mostly carry one or two tags, so the record loads of a step are a few broadcast lines.
		const int nSub = subsY * SUBS_X;
		// NW horizontally adjacent sub-blocks per step (a region has SUBS_X = 4 per row), one pixel of each
		// per lane, shaded as interleaved instruction streams.  A lane with pending pixels in only some of
		// them shades one of those again in place of the others: every lane with work runs the same code.
		constexpr int NW = 2;
		static_assert(SUBS_X % NW == 0, "a step's sub-blocks lie in one row of sub-blocks");
		for (int s = 0; s < nSub; s += NW)
		{
			uint32_t v[NW];
			bool     p[NW];
			int      first = -1;
#pragma unroll
			for (int k = NW - 1; k >= 0; k--)
			{
				v[k] = W.c[((s + k) << 5) | lane];
				p[k] = (v[k] & VIS_PENDING) != 0;
				if (p[k]) first = k;
			}
			if (first >= 0)
			{
				uint32_t vf = v[0];
#pragma unroll
				for (int k = 1; k < NW; k++)
					if (first == k) vf = v[k];
				const int    y = gy + (s / SUBS_X) * SUB_H + ly; // (the step's sub-blocks lie in one row of sub-blocks)
				const uint4 *rec[NW];
				float        e1[NW], e2[NW], e3[NW];
#pragma unroll
				for (int k = 0; k < NW; k++)
				{
					const uint32_t t  = p[k] ? v[k] : vf;
					const int      sk = s + (p[k] ? k : first);
					rec[k] = reinterpret_cast<const uint4 *>(P.prims + (t & ~VIS_PENDING));
					const uint4 q0 = __ldg(rec[k]), q1 = __ldg(rec[k] + 1), q2 = __ldg(rec[k] + 2), q3 = __ldg(rec[k] + 3);
					const int   x  = gx + (sk & (SUBS_X - 1)) * SUB_W + lx;
					const int   rx = x - (int)(q0.z & 0xFFFF), ry = y - (int)(q0.z >> 16);
					e1[k] = (float)((int)q1.x + rx * (int)q1.w + ry * (int)q2.z);
					e2[k] = (float)((int)q1.y + rx * (int)q2.x + ry * (int)q2.w);
					e3[k] = (float)((int)q1.z + rx * (int)q2.y + ry * (int)q3.x);
				}
				uint32_t out[NW];
				shade_opaque_wide<NW>(rec, e1, e2, e3, out);
#pragma unroll
				for (int k = 0; k < NW; k++)
					if (p[k]) W.c[((s + k) << 5) | lane] = out[k];
			}
		}
		__syncwarp();
	}

	// ---- write the region back once (pending tags included: resolve_kernel finishes them) -----------
	if (lane == 0) nextItem = atomicAdd(P.workCounter, 1u); // (the round trip runs behind the stores)
	if (vec)
	{
		float4         *pz = reinterpret_cast<float4 *>(J.gZ + vOff);
		uint4          *pc = reinterpret_cast<uint4 *>(J.gC + vOff);
		const float    *sz = W.z + vsi;
		const uint32_t *sc = W.c + vsi;
		const int       n  = min(subsY, vRows);
#pragma unroll 4
		for (int i = 0; i < n; i++)
		{
			if (FUSED) frame_store(pc, *reinterpret_cast<const uint4 *>(sc)); // finished colours: evict first, like the depths
			else *pc = *reinterpret_cast<const uint4 *>(sc);                  // (plain stores: resolve_kernel reads these lines next)
			frame_store(pz, *reinterpret_cast<const float4 *>(sz));
			pc += width;
			pz += width;
			sc += SUBS_X * 32;
			sz += SUBS_X * 32;
		}
		if (IDS)
		{
			uint4          *pi = reinterpret_cast<uint4 *>(gI + vOff);
			const uint32_t *si = I->t + vsi;
			const int       n  = min(subsY, vRows);
#pragma unroll 4
			for (int i = 0; i < n; i++)
			{
				frame_store(pi, *reinterpret_cast<const uint4 *>(si));
				pi += width;
				si += SUBS_X * 32;
			}
		}
	}
	else
	{
		for (int i = lane; i < regionWords; i += 32)
		{
			const int rx = i & (REGION_W - 1), ry = i / REGION_W, x = gx + rx, y = gy + ry;
			if (x < width && y < height)
			{
				const size_t gi = (size_t)y * width + x;
				const int    si = pix_index((ry >> 2) * SUBS_X + (rx >> 3), ((ry & 3) << 3) + (rx & 7));
				J.gC[gi] = W.c[si];
				J.gZ[gi] = W.z[si];
				if (IDS) gI[gi] = I->t[si];
			}
		}
	}
	__syncwarp();
}

// the persistent item loop of raster_body, for the visibility pass
// (the kernels are instantiations of one __global__ template rather than wrappers around a device function: the
// two-kernel form keeps exactly the machine code it was measured with).  IDS: the variant that also keeps the
// triangle id planes (RasterParams::ids), with 16 KB more shared memory per CTA.
template <bool FUSED, bool IDS = false>
__global__ void __launch_bounds__(128, IDS ? VIS_IDS_CTAS_PER_SM : VIS_CTAS_PER_SM) raster_opaque_kernel(RasterParams P)
{
	__shared__ __align__(16) VisSmem sW[4];
	IdSmem *I = nullptr;
	if constexpr (IDS) I = id_smem();
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	for (size_t i = (size_t)blockIdx.x * 128 + tid; i < P.zeroWords; i += (size_t)gridDim.x * 128) P.zeroBase[i] = 0u;

	VisSmem     &W = sW[warp];
	uint32_t     shaded = 0;
	const size_t plane = (size_t)P.g.width * P.g.height;
	const uint32_t numTiles = P.numTiles;
	const uint32_t nBusy    = *P.numBusy;
	const uint32_t nEmpty   = numTiles - nBusy;
	const uint32_t nSmall   = min(nBusy, max((uint32_t)(((unsigned long long)nBusy * RASTER_SMALL_PERCENT) / 100), P.smallTilesMin));
	const uint32_t nBig     = nBusy - nSmall;
	const bool     fewPrims   = *P.listTotal <= 64ull * nBusy;
	const uint32_t smallShift = !fewPrims ? 2u : ((2 * nBusy < P.smallTilesMin) ? 4u : ((nBusy < P.smallTilesMin) ? 3u : 2u));
	// Untouched tiles can be handed out 1 << VIS_EMPTY_SHIFT per item when there are plenty: claiming an
	// item and loading its tile entry is a dependent ~1.3 us, streaming a tile's clear values takes less
	// (five tiles of six of the 1080p sphere views are untouched), so the entries of an item are loaded
	// together and the claim is paid once.  Four per item measured no gain over one, so the shift is 0.
	// The loops below keep their general form: written for one tile they compile to a different
	// instruction schedule than the one that was measured.  (Claiming items ahead instead -- a ring of up
	// to four claims per warp -- cost 12 %: the last busy regions then start late.)
	const uint32_t warpsTotal  = gridDim.x * 4u;
	const uint32_t emptyShift  = nEmpty >= 8u * warpsTotal ? VIS_EMPTY_SHIFT : 0u;
	const uint32_t emptyItems  = (nEmpty + (1u << emptyShift) - 1u) >> emptyShift;
	const uint32_t itemsBusy   = 2 * nBig + (nSmall << smallShift);
	const uint32_t itemsMixed  = itemsBusy + (uint32_t)(((unsigned long long)emptyItems * (100 - RASTER_TAIL_PERCENT)) / 100);
	const uint32_t itemsTotal  = itemsBusy + emptyItems;
	const unsigned long long ratio = itemsMixed ? ((((unsigned long long)itemsBusy << 32) + itemsMixed - 1) / itemsMixed) : 0ull;
	uint32_t next = 0;
	if (lane == 0) next = atomicAdd(P.workCounter, 1u);
	for (;;)
	{
		const uint32_t item = __shfl_sync(0xffffffffu, next, 0);
		if (item >= itemsTotal) break;
		bool     busy = false;
		uint32_t b0 = itemsBusy;
		if (item < itemsMixed)
		{
			b0   = (uint32_t)(((unsigned long long)item * ratio) >> 32);
			busy = (uint32_t)(((unsigned long long)(item + 1u) * ratio) >> 32) > b0;
		}
		if (!busy)
		{
			if (lane == 0) next = atomicAdd(P.workCounter, 1u);
			const uint32_t first = (item - b0) << emptyShift;
			const uint32_t n     = min(1u << emptyShift, nEmpty - first);
			uint32_t       fr[1 << VIS_EMPTY_SHIFT];
			uint4          e1[1 << VIS_EMPTY_SHIFT];
#pragma unroll
			for (uint32_t k = 0; k < (1u << VIS_EMPTY_SHIFT); k++)
				if (k < n)
				{
					const uint32_t slot = numTiles - 1 - (first + k);
					fr[k] = __ldg(&P.order[2 * slot].w);
					e1[k] = __ldg(P.order + 2 * slot + 1);
				}
#pragma unroll
			for (uint32_t k = 0; k < (1u << VIS_EMPTY_SHIFT); k++)
				if (k < n)
				{
					const bool genZ = (e1[k].y & FI_Z_RESET) != 0, genC = (e1[k].y & FI_COLOR_CLEAR) != 0;
					if (genZ || genC)
						stream_empty_tile<IDS>(P, (int)(e1[k].z & 0xFFFFu), (int)(e1[k].z >> 16), P.color + plane * fr[k], P.depth + plane * fr[k],
						                       IDS ? P.ids + plane * fr[k] : nullptr, genC, genZ, e1[k].x, lane);
				}
			continue;
		}
		uint32_t slot;
		int      rx, ry = 0, rows;
		if (b0 < 2 * nBig)
		{
			slot = b0 >> 1;
			rx   = (int)(b0 & 1) * REGION_W;
			rows = REGION_H;
		}
		else
		{
			const uint32_t k = b0 - 2 * nBig;
			slot = nBig + (k >> smallShift);
			rx   = (int)(k & 1) * REGION_W;
			rows = REGION_H >> (smallShift - 1);
			ry   = (int)((k >> 1) & ((1u << (smallShift - 1)) - 1u)) * rows;
		}
		const uint4 d0 = __ldg(P.order + 2 * slot), d1 = __ldg(P.order + 2 * slot + 1);
		const int   tx = (int)(d1.z & 0xFFFFu), ty = (int)(d1.z >> 16);
		const bool  genZ = (d1.y & FI_Z_RESET) != 0, genC = (d1.y & FI_COLOR_CLEAR) != 0;
		// a tile with primitives goes to the tag planes (the context's own; resolve_kernel finishes it into the output)
		uint32_t   *gC = ((d0.y && !FUSED) ? P.tagColor : P.color) + plane * d0.w;
		float      *gZ = P.depth + plane * d0.w;
		RegionJob J;
		J.gx   = tx * TILE_W + rx;
		J.gy   = ty * TILE_H + ry;
		J.rows = rows;
		if (J.gx >= P.g.width || J.gy >= P.g.height)
		{
			if (lane == 0) next = atomicAdd(P.workCounter, 1u);
			continue;
		}
		J.count       = d0.y;
		J.clearPacked = d1.x;
		J.gC          = gC;
		J.gZ          = gZ;
		J.genZ        = genZ;
		J.genC        = genC;
		J.listOff     = d0.z;
		process_region_vis<FUSED, IDS>(P, W, I, lane, J, shaded, next);
	}
	shaded = __reduce_add_sync(0xffffffffu, shaded);
	if (lane == 0 && shaded) atomicAdd(P.setPixels, (unsigned long long)shaded);
}

constexpr auto raster_vis_kernel = raster_opaque_kernel<false>; // visibility only: resolve_kernel follows
// Visibility and resolve in ONE kernel: a region's pending pixels are shaded from shared memory as soon as
// its walk is over, by the warp that owns it; no tag planes, no second pass over the busy tiles.
constexpr auto raster_visres_kernel = raster_opaque_kernel<true>;
constexpr auto raster_vis_ids_kernel    = raster_opaque_kernel<false, true>;
constexpr auto raster_visres_ids_kernel = raster_opaque_kernel<true, true>;

// Resolve: every pixel of the tiles that have primitives; a pixel that still carries a tag is shaded
// from its triangle's record.  One CTA per busy tile (grid-stride), thread t takes pixels t + 256 k of
// the tile, row-major: a warp reads and writes whole 128-byte row segments.
constexpr int RESOLVE_MIN_CTAS = 8; // 32 registers: all 64 warps of an SM resident
__global__ void __launch_bounds__(256, RESOLVE_MIN_CTAS) resolve_kernel(ResolveParams R)
{
	constexpr int  PER_THREAD = TILE_W * TILE_H / 256;
	const uint32_t nBusy = *R.numBusy;
	const size_t   plane = (size_t)R.g.width * R.g.height;
	const bool     split = R.tags != R.color; // foreign output planes: every pixel of a busy tile is stored
	const int      px0 = (int)threadIdx.x & (TILE_W - 1), py0 = (int)threadIdx.x / TILE_W; // pixel of the first of the thread's rows
	for (uint32_t slot = blockIdx.x; slot < nBusy; slot += gridDim.x)
	{
		const uint4 d0 = __ldg(R.order + 2 * slot), d1 = __ldg(R.order + 2 * slot + 1);
		const int   x = (int)(d1.z & 0xFFFFu) * TILE_W + px0, yTop = (int)(d1.z >> 16) * TILE_H + py0;
		const size_t    pix = plane * d0.w + (size_t)yTop * R.g.width + x;
		uint32_t       *col = R.color + pix;
		const uint32_t *tag = R.tags + pix;
		// all of the thread's tags first: eight independent loads in flight (the tags come from DRAM: the
		// visibility kernel wrote a gigabyte of frames since it stored them)
		uint32_t v[PER_THREAD];
#pragma unroll
		for (int k = 0; k < PER_THREAD; k++)
		{
			const int y = yTop + k * (256 / TILE_W);
			v[k] = (x < R.g.width && y < R.g.height) ? __ldcs(tag + (size_t)k * (256 / TILE_W) * R.g.width) : VIS_OUTSIDE;
		}
		// (unroll 2: -1 %; the tags then live in local memory)
#pragma unroll 8
		for (int k = 0; k < PER_THREAD; k++)
		{
			if (!(v[k] & VIS_PENDING))
			{
				// finished already (clear colour, or an inexact triangle's fragment): in place, unless the output is elsewhere
				if (split && v[k] != VIS_OUTSIDE) frame_store_u32(col + (size_t)k * (256 / TILE_W) * R.g.width, v[k]);
				continue;
			}
			const int    y   = yTop + k * (256 / TILE_W);
			const uint4 *rec = reinterpret_cast<const uint4 *>(R.prims + (v[k] & ~VIS_PENDING));
			const uint4  q0 = __ldg(rec), q1 = __ldg(rec + 1), q2 = __ldg(rec + 2), q3 = __ldg(rec + 3);
			// the int32 edge functions at this pixel: bbox-origin value + steps (exact, see setup_kernel)
			const int rx = x - (int)(q0.z & 0xFFFF), ry = y - (int)(q0.z >> 16);
			const int E1 = (int)q1.x + rx * (int)q1.w + ry * (int)q2.z;
			const int E2 = (int)q1.y + rx * (int)q2.x + ry * (int)q2.w;
			const int E3 = (int)q1.z + rx * (int)q2.y + ry * (int)q3.x;
			frame_store_u32(col + (size_t)k * (256 / TILE_W) * R.g.width, shade_opaque_from_record(rec, (float)E1, (float)E2, (float)E3));
		}
	}
}
