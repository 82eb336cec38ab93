// vrm_flat.cuh -- the traversal of vrm_core.cuh re-expressed as a per-ray STATE MACHINE whose states are code blocks
// that the lanes of a warp share.
//
// Why: the reference's control flow is four levels of nested data-dependent loops (scene walk > region march > voxel
// steps / cluster jumps, then the same again for the shadow ray).  Executed as written, a warp serialises lanes that are
// in different loops or have different trip counts: the first sm_100a capture showed 10.6 of 32 threads active per
// instruction for VCS + longest axis (profiles/r01a_ncu_render_vcs_longestaxis.json).  Here a ray is always in one of five
// states and each state's work is one block of straight-line code:
//     kStRegion  enter the region under the ray (table entry already read): leave / null region / load the region
//     kStHead    longest axis only: loop condition of Renderer.cuh:787 + the order of this iteration's voxel tests
//     kStMain    [one advance: next voxel edge | cluster edge | cluster jump | null-region edge] + ONE voxel test
//     kStHit     shade the hit (applyLighting) and turn the lane into the hit's shadow ray
//     kStDone    pixel resolved
// `step()` runs the blocks in program order (region -> head -> main), so a lane that enters a stored region does its
// prologue, its loop head and its first voxel test in one pass, and ALL advances -- voxel steps, cluster skips, cluster
// jumps and null-region skips, primary or shadow -- go through the one advance site and all voxel tests through the one
// test site: lanes of a warp in different phases execute the same instructions.
//
// The per-ray state is kept small (profiles/r01e: the first layout spent 6 % of its issue slots on local-memory traffic): the walk-space
// permutation is three storage shifts + three region-table strides, state and advance mode are ONE word, flags are bits of another,
// the tX/tY/tZ/tMin of the last advance are reduced to the three equality bits the normal needs, and the light's direction constants
// come precomputed from the host (LightWalk).  The fused render kernel is compiled for 56 registers (9 CTAs per SM): ptxas then spills
// ~0.5 KB per thread, 3 % of the executed instructions, all of it in the generic pass -- measured faster than 64 registers with a
// quarter of the spills (1.224 vs 1.244 ms, DESIGN.md 3.2).
//
// ARITHMETIC IS UNCHANGED: the same operations in the same order as vrm_core.cuh / the reference -- only the order in
// which different rays' operations are interleaved changes.  tests/hostsim runs this very code on the CPU against the
// oracle (bit-exact RGB, hit maps and event counters).
#pragma once

#include "vrm_core.cuh"

// 1: the state machine's VCS test site reads the cluster-exists flag from the header word it needs anyway (one load);
// 0: separate 64-byte-per-region cluster mask first (two dependent loads, but empty clusters never touch the headers)
// cold member functions of the state machine: out of line on the device (they copy the whole ray state)
#if defined(__CUDACC__)
#define VRM_FLAT_COLD __host__ __device__ __noinline__
#else
#define VRM_FLAT_COLD
#endif

#ifndef VRM_VCS_FUSED_EXIST
#define VRM_VCS_FUSED_EXIST 1
#endif

namespace vrm
{

// ONE state word per ray: values 0..4 are "kStMain" -- the value IS the AdvMode the next step starts with (so `is a cluster jump next`
// is one compare, and the word the warp votes on classifies a lane completely) -- then the other blocks.  st <= kStHead: marching.
enum FlatState : int
{
	kStMainLast = 4,  // st <= kStMainLast: kStMain, st = kAdvNone / kAdvNext / kAdvCluster / kAdvJump / kAdvRegion
	kStRegion = 5,
	kStHead = 6,
	kStHit = 7,
	kStDone = 8,
	kStPark = 9   // kPpDefer: the ray met the ping-pong pathology; its lane stops and the caller parks it for resume_kernel
};

// What the advance of a kStMain step moves to.  All are "t_i = (next_i - o_i) / dir_i, o += (min t [+ EPSILON]) * dir".
enum AdvMode : int
{
	kAdvNone = 0,     // no advance: a longest-axis voxel test on gridValues
	kAdvNext = 1,     // next voxel edge +-EPSILON                      (Renderer.cuh:269-280,320-331)
	kAdvCluster = 2,  // cluster edge of the voxel under the ray        (Renderer.cuh:293-304)
	kAdvJump = 3,     // one iteration of performVoxelSpaceJump's loop   (Renderer.cuh:707-721): cluster edge of gridValues, scaled direction
	kAdvRegion = 4    // null-region skip to the region edge, no +EPSILON (Renderer.cuh:384-410, guarded twin 185-211)
};

// flag bits of FlatRay::fl
constexpr uint32_t kFlShadow = 1u;       // this is the shadow ray of an already shaded hit
constexpr uint32_t kFlShadowLA = 2u;     // ... walked with the longest-axis routines (Renderer.cuh:633-694) rather than the original ones (174-235)
constexpr uint32_t kFlEq0 = 4u;          // t_i == tMin of the last kAdvNext / kAdvJump advance, walk slot i = bit 2 + i  (getNormalFromTValues)
constexpr uint32_t kFlEqMask = 28u;
constexpr int kFlPermShift = 8;
constexpr int kFlHzShift = 14;           // bits 14-31: the shadow ray's horizon threshold, a signed integer (past_horizon); kHzNever: none
constexpr int32_t kHzNever = 131071, kHzMin = -131072;
constexpr int32_t kRiPending = -3;       // FlatRay::ri: the ray has left its region, rebase + table read still to do          // bits 8-13: world axis of walk slot 0 / 1 / 2, two bits each

// What a ray does when it meets the region-face ping-pong pathology (FlatRay::pingpong_skip):
//   kPpOff     nothing: it crawls like the reference
//   kPpDefer   it parks its whole state in a device queue and its lane finishes; resume_kernel (vrm_render.cu) continues such
//              rays with kPpInline.  This keeps the fast-forward (which copies the ray state and calls out of line) away from
//              the hot kernels: compiled into them -- even as a never-taken branch -- it cost 30 % of their speed.
//   kPpInline  fast-forward in place (resume kernel, host harness)
constexpr int kPpOff = 0, kPpDefer = 1, kPpInline = 2;
#ifndef VRM_REGION_VOTE
#define VRM_REGION_VOTE 0  // > 0: march_scene_flat_warp runs the region-entry block only when at least this many lanes want it (or nothing else can run)
#endif
#ifndef VRM_HEAD_VOTE
#define VRM_HEAD_VOTE 0    // the same for the longest-axis loop head
#endif
#ifndef VRM_PP_DEFAULT
#define VRM_PP_DEFAULT 2
#endif
#ifndef VRM_FAST_LA
#define VRM_FAST_LA 7      // a third warp-uniform block: longest-axis stepping (FlatRay::fast_la); A/B bits: 2 = without the stored-region entry, 4 = without the inner loop
#endif
#ifndef VRM_CC_MUL
#define VRM_CC_MUL 1       // 1: FlatRay::sh holds 1 << shift and the storage codes are multiply-add chains instead of shifts + ORs (measured: 1.335 -> 1.315 ms)
#endif
#ifndef VRM_CLS_LUT
#define VRM_CLS_LUT 1      // 1: the class a lane votes with comes from a nibble table indexed by the state word (measured: 1.335 -> 1.307 ms)
#endif
#ifndef VRM_FAST_ENTER
#define VRM_FAST_ENTER 0   // 1: fast_jump / fast_nullskip run a stored region's entry block in the pass that changed region (A/B: 1.338 vs 1.332 ms, off)
#endif
#ifndef VRM_FAST_LOOPS
#define VRM_FAST_LOOPS 1   // the warp stays inside a fast block while every marching lane still qualifies
#endif
#ifndef VRM_HORIZON_AT
#define VRM_HORIZON_AT 1   // where a shadow ray tests its horizon threshold: 0 after every cluster skip / jump / null-region skip, 1 when it changes region
#endif
#ifndef VRM_FAST_PATHS
#define VRM_FAST_PATHS 1   // march_scene_flat_warp (VCS + longest axis): warp-uniform fast paths for all-jump / all-null-region passes (FlatRay::fast_jump)
#endif
constexpr int kPpDefault = VRM_PP_DEFAULT;  // single-ray callers (host harness; 0 there = crawl like the reference); the kernels name their policy

struct DeferHeader
{
	unsigned int count;     // rays queued (may exceed capacity: the excess was not queued)
	unsigned int capacity;
	unsigned int pad[2];
};

VRM_HD PermRuntime unpack_perm(uint32_t fl)
{
	PermRuntime p;
	p.a0 = (int)((fl >> kFlPermShift) & 3u); p.a1 = (int)((fl >> (kFlPermShift + 2)) & 3u); p.a2 = (int)((fl >> (kFlPermShift + 4)) & 3u);
	return p;
}
VRM_HD uint32_t pack_perm(const PermRuntime& p) { return ((uint32_t)p.a0 | ((uint32_t)p.a1 << 2) | ((uint32_t)p.a2 << 4)) << kFlPermShift; }

// The light's direction in the two walk spaces a shadow ray can use, with its exact-division constants: the same for every
// shadow ray of a frame, so it is computed once on the host (same IEEE operations: make_raydir / scaled_raydir).
VRM_HD LightWalk make_light_walk(const Lighting& L)
{
	LightWalk w;
	const RayDir ki = make_raydir(L.dir[0], L.dir[1], L.dir[2]);
	for (int i = 0; i < 3; i++) { w.idD[i] = ki.d[i]; w.idR[i] = ki.rd[i]; }
	w.idThr = ki.thr;
	const PermRuntime p = rank_axes(L.dir[0], L.dir[1], L.dir[2]);
	float dw[3];
	to_walk(p, L.dir, dw);
	const RayDir k = make_raydir(dw[0], dw[1], dw[2]);
	const RayDir ko = scaled_raydir(k);
	for (int i = 0; i < 3; i++) { w.laD[i] = k.d[i]; w.laR[i] = k.rd[i]; w.laSD[i] = ko.d[i]; w.laSR[i] = ko.rd[i]; }
	w.laThr = (k.thr == k.thr && ko.thr == ko.thr) ? k.thr : NAN;
	w.laPerm = pack_perm(p);
	return w;
}

// apply_lighting's directional branch with the three colour / 255.0f divisions done by the exact reciprocal + FMA residual
// form (div_by_const; checked equal to IEEE division for every integer numerator up to 2^24).  Same values, a third of the
// instructions.  The point-light branch is the shared apply_lighting.
VRM_HD uint32_t apply_lighting_flat(const Lighting& L, const float* translation, uint32_t voxelColor, int normalAxis, float normalSign,
                                    const float* hitLocal, const int* regW)
{
	if (L.usePoint) return apply_lighting(L, translation, voxelColor, normalAxis, normalSign, hitLocal, regW);
	const float r255 = 0.00392156886f;  // RN(1 / 255)
	const float cr = div_by_const((float)(voxelColor >> 16), 255.0f, r255);
	const float cg = div_by_const((float)((voxelColor >> 8) & 0xFF), 255.0f, r255);
	const float cb = div_by_const((float)(voxelColor & 0xFF), 255.0f, r255);
	const float n0 = normalAxis == 0 ? normalSign : 0.0f, n1 = normalAxis == 1 ? normalSign : 0.0f, n2 = normalAxis == 2 ? normalSign : 0.0f;
	const float diff = fmaxf(vadd(vadd(vmul(n0, L.dir[0]), vmul(n1, L.dir[1])), vmul(n2, L.dir[2])), 0.0f);  // Renderer.cuh:57-66
	return vec_to_rgb(vmul(cr, vmul(diff, L.color[0])), vmul(cg, vmul(diff, L.color[1])), vmul(cb, vmul(diff, L.color[2])));
}

// primary_ray with its five divisions (two by the image size, three by the ray length) in the exact reciprocal form.
// invW / invH = RN(1 / W), RN(1 / H) from the host.
VRM_HD void primary_ray_flat(const float* cam, uint32_t x, uint32_t y, uint32_t W, uint32_t H, float invW, float invH, float* o, float* d)
{
	const float u = div_by_const(vadd((float)x, 0.5f), (float)W, invW);  // numerators >= 0.5, 1 <= W,H < 2^32: inside div_by_const's preconditions
	const float v = div_by_const(vadd((float)(H - y), 0.5f), (float)H, invH);
	float rel[3];
	for (int i = 0; i < 3; i++)
	{
		o[i] = vadd(vadd(cam[3 + i], vmul(u, cam[6 + i])), vmul(v, cam[9 + i]));
		rel[i] = vsub(o[i], cam[i]);
	}
	const float len = vsqrt(vadd(vadd(vmul(rel[0], rel[0]), vmul(rel[1], rel[1])), vmul(rel[2], rel[2])));
	const float rl = vrcp(len);
	const float thr = dir_component_safe(len) ? 7.888609052210118e-31f : NAN;
	div3(rel[0], rel[1], rel[2], len, len, len, rl, rl, rl, thr, d[0], d[1], d[2]);
}

template <int ST, int ALGO, bool STATS>
struct FlatRay
{
	static constexpr bool kLA = ALGO != kAlgoOriginal;

	// current ray (primary or shadow), region-local, walk space
	float o[3];    // original algorithm: ray origin; longest axis: oldRay origin (the reference copies between the two only
	               // at points where they are equal, Renderer.cuh:726,768,912)
	float d[3], rd[3];    // direction and RN(1 / d): exact division by a per-ray constant (vrm_core.cuh)
	float sd[3], srd[3];  // the same for the longest-axis-scaled direction (Ray.cuh:69): per-ray constants, not per region
	float thr;            // fast-division threshold: 2^-100 when every component of d (and sd) qualifies, else NaN
	uint32_t ur[3];       // region coordinates minus minCoord (walk space); in the table <=> all < diameter
	int32_t ri;           // table entry of the region under the ray: dense region index, -1 null region, -2 outside the table
	RegionRef<ST> r;      // hash table: the region's descriptor (the VCS addresses everything from ri)
	uint32_t sh[3];       // walk slot -> place of its coordinate inside a storage code: 1 << shift (VRM_CC_MUL; else the shift), shift = 6/3/0 per world x/y/z (VCS) or 14/7/0 (hash key)
	uint32_t rs[3];       // walk slot -> stride of its coordinate in the region table (1, D, D*D per world x/y/z)
	int st;               // FlatState; 0..4 = kStMain with that AdvMode
	uint32_t fl;          // kFl* bits
	// longest-axis state (slot 0 = longest axis).  g is also "the voxel under the ray" of the other advances.
	float ro[3];          // ray origin (rayMarchVoxelGridLongestAxis' `ray`); a pending hit keeps its position here
	int g[3];
	int ad1, ad2;         // axisDiff of the middle / shortest slot (slot 0's is the sign of d[0])
	uint32_t seq;         // slots still to test this iteration, two bits each, first in the low bits; slot 0 is always the last.  A pending hit (kStHit) keeps its packed normal / shadow-routine bits here
	// `result` = voxel colour (kStHit) -> shaded colour waiting for its shadow ray -> final pixel colour (kStDone).
	uint32_t result;

	VRM_HD bool shadow() const { return (fl & kFlShadow) != 0; }
	VRM_HD bool shadowOriginal() const { return (fl & (kFlShadow | kFlShadowLA)) == kFlShadow; }  // zero-direction guards in the null-region skip (Renderer.cuh:191-193)

	VRM_HD void finish(uint32_t colour)
	{
		result = colour;
		st = kStDone;
	}

	VRM_HD void set_perm(const SceneView& sv, const PermRuntime& p)
	{
		fl = (fl & ~(63u << kFlPermShift)) | pack_perm(p);
		const uint32_t D = sv.diameter;
		const int a[3] = {p.a0, p.a1, p.a2};
		for (int i = 0; i < 3; i++)
		{
			sh[i] = ST == kStorageHash ? (uint32_t)(kHashKeyBits * (2 - a[i])) : (uint32_t)(6 - 3 * a[i]);
#if VRM_CC_MUL
			sh[i] = 1u << sh[i];  // kept as the multiplier: the three fields are disjoint, so the code is one multiply-add chain
#endif
			rs[i] = a[i] == 0 ? 1u : (a[i] == 1 ? D : D * D);
		}
	}

	// VoxelScene::isRayInScene + getRegionStorageStructure (Renderer.cuh:29-44)
	VRM_HD void read_region_entry(RayCtx<ST, STATS>& c)
	{
		const uint32_t D = c.sv.diameter;
		if (!(ur[0] < D && ur[1] < D && ur[2] < D)) { ri = -2; return; }
		if (STATS) c.st.nRegionReads++;
		ri = ldg(c.sv.regionTable + (ur[0] * rs[0] + ur[1] * rs[1] + ur[2] * rs[2]));
	}

	// rebase into the neighbouring region after the ray left the current one (Renderer.cuh:421-429) and read its entry
	VRM_HD void change_region(RayCtx<ST, STATS>& c)
	{
		for (int i = 0; i < 3; i++)
		{
			const int diff = (int)floorf(vmul(o[i], 0.015625f));  // o / 64 (exact scaling by a power of two)
			ur[i] += (uint32_t)diff;
			o[i] = vsub(o[i], (float)(diff * kRegion));  // convertRayToLocalSpace(.., scale 1), Ray.cuh:14-17: the product with 1.0f is the identity
		}
		st = kStRegion;
		if (VRM_HORIZON_AT == 1 && past_horizon()) { finish(result); return; }
		if (!position_sane(o)) { ri = -2; return; }  // see position_sane (vrm_core.cuh)
		read_region_entry(c);
	}

	// rayMarchVoxelScene / rayMarchVoxelSceneLongestAxis up to the first region (Renderer.cuh:338-378, 917-954)
	VRM_HD void start_primary(RayCtx<ST, STATS>& c, const float* originW, const float* dirW, float scale)
	{
		fl = (uint32_t)kHzNever << kFlHzShift; result = 0; ri = -2; seq = 0; ad1 = ad2 = 0;
		g[0] = g[1] = g[2] = 0; ro[0] = ro[1] = ro[2] = 0.0f;
		PermRuntime p;
		p.a0 = 0; p.a1 = 1; p.a2 = 2;
		if constexpr (kLA) p = rank_axes(dirW[0], dirW[1], dirW[2]);
		set_perm(c.sv, p);
		float sW[3] = {canonical_zero(vmul(scale, vsub(originW[0], c.translation[0]))), canonical_zero(vmul(scale, vsub(originW[1], c.translation[1]))),
		               canonical_zero(vmul(scale, vsub(originW[2], c.translation[2])))};
		float dw[3];
		to_walk(p, sW, o); to_walk(p, dirW, dw);
		const RayDir k = make_raydir(dw[0], dw[1], dw[2]);
		for (int i = 0; i < 3; i++) { d[i] = k.d[i]; rd[i] = k.rd[i]; }
		thr = k.thr;
		if constexpr (kLA)
		{
			const RayDir ko = scaled_raydir(k);
			for (int i = 0; i < 3; i++) { sd[i] = ko.d[i]; srd[i] = ko.rd[i]; }
			if (!(ko.thr == ko.thr)) thr = NAN;
		}
		int reg[3] = {(int)floorf(vmul(o[0], 0.015625f)), (int)floorf(vmul(o[1], 0.015625f)), (int)floorf(vmul(o[2], 0.015625f))};
		const int minC = c.sv.minCoord;
		const uint32_t D = c.sv.diameter;
		while (reg[0] - minC < 0 || reg[1] - minC < 0 || reg[2] - minC < 0 ||
		       (uint32_t)(reg[0] - minC) > D - 1 || (uint32_t)(reg[1] - minC) > D - 1 || (uint32_t)(reg[2] - minC) > D - 1)
		{
			// scene-entry loop, Renderer.cuh:349-373
			const int far = (int)(D + (uint32_t)minC);
			float a0, a1, a2;
			div3(vsub((float)((d[0] < 0.0f ? far : minC) * kRegion), o[0]), vsub((float)((d[1] < 0.0f ? far : minC) * kRegion), o[1]),
			     vsub((float)((d[2] < 0.0f ? far : minC) * kRegion), o[2]), d[0], d[1], d[2], rd[0], rd[1], rd[2], thr, a0, a1, a2);
			if (a0 <= 0.0f) a0 = INFINITY;
			if (a1 <= 0.0f) a1 = INFINITY;
			if (a2 <= 0.0f) a2 = INFINITY;
			const float m = min3(a0, a1, a2);
			if (m == INFINITY || m != m) { finish(0); return; }  // (a NaN tMin only arises from 0/0: treated as a miss)
			const float s = vadd(m, kEps);
			o[0] = along(o[0], s, d[0]); o[1] = along(o[1], s, d[1]); o[2] = along(o[2], s, d[2]);
			reg[0] = (int)floorf(vmul(o[0], 0.015625f)); reg[1] = (int)floorf(vmul(o[1], 0.015625f)); reg[2] = (int)floorf(vmul(o[2], 0.015625f));
		}
		for (int i = 0; i < 3; i++)
		{
			o[i] = vsub(o[i], (float)(reg[i] * kRegion));  // Renderer.cuh:376-378
			ur[i] = (uint32_t)(reg[i] - minC);
		}
		st = kStRegion;
		read_region_entry(c);
	}

	// ---- kStHit: applyLighting(...) * !isInShadow...(Ray(hit, LIGHT_DIRECTION), currentRegion)  (Renderer.cuh:314-315,821-822,...)
	// v0..v2: the voxel that was hit (region-local, walk space), for the hit map
	VRM_HD void record_hit(RayCtx<ST, STATS>& c, uint32_t col, float p0, float p1, float p2, int nAxisW, float nSign, bool laKind, int v0, int v1, int v2)
	{
		if (shadow()) { finish(0); return; }  // any voxel on the shadow ray: colour * !inShadow = 0
		if (c.hitOut)
		{
			const PermRuntime p = unpack_perm(fl);
			const int minC = c.sv.minCoord;
			const int reg[3] = {(int)ur[0] + minC, (int)ur[1] + minC, (int)ur[2] + minC};
			record_hit_voxel(c, p, reg, v0, v1, v2);
		}
		result = col;
		ro[0] = p0; ro[1] = p1; ro[2] = p2;
		seq = (uint32_t)(nAxisW | (nSign < 0.0f ? 4 : 0) | (laKind ? 8 : 0));
		st = kStHit;
	}

	// the pending hit's lighting: where its shadow ray starts (WORLD axes) and the colour that survives when the light is visible
	VRM_HD void shade_hit(RayCtx<ST, STATS>& c, ShadowStart& ss) const
	{
		const int nAxisW = (int)(seq & 3u);
		const float nSign = (seq & 4u) ? -1.0f : 1.0f;
		const PermRuntime p = unpack_perm(fl);
		const int minC = c.sv.minCoord;
		const int reg[3] = {(int)ur[0] + minC, (int)ur[1] + minC, (int)ur[2] + minC};
		to_world(p, ro, ss.hitW); to_world(p, reg, ss.regW);
		ss.lit = apply_lighting_flat(c.light, c.translation, result, nAxisW, nSign, ss.hitW, ss.regW);
		ss.la = (kLA && (seq & 8u) != 0) ? 1 : 0;
	}

	// isInShadowOriginalRayMarch / isInShadowRayMarchVoxelSceneLongestAxis up to their first region (Renderer.cuh:174-199, 633-657): the
	// ray becomes the shadow ray of `ss`; it ends with result = ss.lit (light visible) or 0 (any voxel on the way)
	VRM_HD void start_shadow(RayCtx<ST, STATS>& c, const ShadowStart& ss)
	{
		const bool laKind = kLA && ss.la != 0;
		result = ss.lit;
		fl = kFlShadow | (laKind ? kFlShadowLA : 0u);
		seq = 0; ad1 = ad2 = 0; ri = -2;
		g[0] = g[1] = g[2] = 0; ro[0] = ro[1] = ro[2] = 0.0f;  // (every one of these is rewritten before it is read; a fresh ray of the shadow kernel starts defined)
		PermRuntime p;
		p.a0 = 0; p.a1 = 1; p.a2 = 2;
		if (laKind) p = unpack_perm(c.lw.laPerm);
		set_perm(c.sv, p);
		to_walk(p, ss.hitW, o);
		{
			int regWalk[3];
			to_walk(p, ss.regW, regWalk);
			const int minC = c.sv.minCoord;
			for (int i = 0; i < 3; i++) ur[i] = (uint32_t)(regWalk[i] - minC);
		}
		if (laKind)
		{
			for (int i = 0; i < 3; i++) { d[i] = c.lw.laD[i]; rd[i] = c.lw.laR[i]; }
			if constexpr (kLA) { for (int i = 0; i < 3; i++) { sd[i] = c.lw.laSD[i]; srd[i] = c.lw.laSR[i]; } }
			thr = c.lw.laThr;
		}
		else
		{
			for (int i = 0; i < 3; i++) { d[i] = c.lw.idD[i]; rd[i] = c.lw.idR[i]; }
			thr = c.lw.idThr;
		}
		fl |= (uint32_t)(c.hv.cells ? horizon_threshold(c, ss) : kHzNever) << kFlHzShift;
		st = kStRegion;
		read_region_entry(c);
	}

	// The shadow ray's threshold from ONE lookup of the horizon map at its start point (every later point of its line projects to the
	// same place).  Stated in the signed world coordinate of the ray's walk slot 0 -- a = hv.axis (the largest |n_a|) for the longest-axis
	// routine, world x for the original one (none when n_x = 0): the depth along n grows by 1 / |n_a| per unit of that coordinate.
	// Rounded up to whole voxels and clamped to 18 bits, it travels in the flag word instead of a register of its own: coordinates
	// relative to the table origin stay below 64 * 1024 = 65536, so kHzNever is never passed and kHzMin ends the ray at once.
	VRM_HD int32_t horizon_threshold(const RayCtx<ST, STATS>& c, const ShadowStart& ss) const
	{
		const HorizonView& h = c.hv;
		const int minC = c.sv.minCoord;
		float pw[3];
		for (int i = 0; i < 3; i++) pw[i] = (float)((ss.regW[i] - minC) * kRegion) + ss.hitW[i];  // relative to the table origin
		int iu = (int)floorf((pw[0] * h.e1[0] + pw[1] * h.e1[1] + pw[2] * h.e1[2] - h.u0) * h.invCell);
		int iv = (int)floorf((pw[0] * h.e2[0] + pw[1] * h.e2[1] + pw[2] * h.e2[2] - h.v0) * h.invCell);
		iu = iu < 0 ? 0 : (iu >= (int)h.nu ? (int)h.nu - 1 : iu);  // (a start point off the grid has no cluster near its line at all)
		iv = iv < 0 ? 0 : (iv >= (int)h.nv ? (int)h.nv - 1 : iv);
		const int32_t top = ldg(h.cells + ((uint32_t)iv * h.nu + (uint32_t)iu));
		const float depth0 = pw[0] * h.n[0] + pw[1] * h.n[1] + pw[2] * h.n[2];
		const int a = (fl & kFlShadowLA) ? h.axis : 0;
		const float na = pick3(a, h.n[0], h.n[1], h.n[2]), pa = pick3(a, pw[0], pw[1], pw[2]);
		if (na == 0.0f) return kHzNever;
		const float t = ceilf((na < 0.0f ? -pa : pa) + ((float)top + kHorizonMargin - depth0) * fabsf(na));
		return t >= (float)kHzNever ? kHzNever : (t <= (float)kHzMin ? kHzMin : (int32_t)t);
	}

	// a shadow ray beyond its threshold: every voxel test it could still make lies past the deepest occupied cluster near its line
	VRM_HD bool past_horizon() const
	{
		if (!(fl & kFlShadow)) return false;  // (primary rays hold kHzNever; the test only saves them the arithmetic)
		const float w = (float)(ur[0] * (uint32_t)kRegion) + o[0];
		return (d[0] < 0.0f ? -w : w) > (float)((int32_t)fl >> kFlHzShift);
	}

	VRM_HD void do_hit(RayCtx<ST, STATS>& c)
	{
		ShadowStart ss;
		shade_hit(c, ss);
		if (!c.light.useShadows || (c.skipDead && ss.lit == 0u)) { finish(ss.lit); return; }
		start_shadow(c, ss);
	}

	// ---- kStRegion ---------------------------------------------------------------------------------------------
	VRM_HD void do_region(RayCtx<ST, STATS>& c)
	{
		if (ri == -2) { finish(shadow() ? result : 0u); return; }  // left the scene: background / not shadowed
		if (ri == -1) { st = kAdvRegion; return; }  // null region: skip to its edge through the advance site
		r = load_region<ST>(c.sv, ri);
		bool la = false;
		if constexpr (kLA) la = !shadowOriginal();
		if (la)
		{
			// rayMarchVoxelGridLongestAxis prologue, Renderer.cuh:763-784.  The reference divides by the scaled longest
			// component +-1.0f: x / 1 = x and x / -1 = -x exactly.
			g[0] = (int)o[0]; g[1] = (int)o[1]; g[2] = (int)o[2];
			const float t = d[0] < 0.0f ? -vsub(vsub((float)g[0], kEps), o[0]) : vsub(vadd(vadd((float)g[0], kEps), 1.0f), o[0]);
			ro[0] = along(o[0], t, sd[0]); ro[1] = along(o[1], t, sd[1]); ro[2] = along(o[2], t, sd[2]);
			ad1 = (int)ro[1] - g[1];
			ad2 = (int)ro[2] - g[2];
			st = kStHead;
		}
		else st = kAdvNext;  // the region march starts with one step before the first test (Renderer.cuh:269-280)
	}

	// ---- kStHead (longest axis): Renderer.cuh:787-805 ------------------------------------------------------------------
	VRM_HD void do_head()
	{
		const int ad0 = d[0] < 0.0f ? -1 : 1;
		if (!grid_in_region(g[0] + ad0, g[1] + ad1, g[2] + ad2))
		{
			// Renderer.cuh:911-914: finish the region with the original algorithm from oldRay's origin (o already is it)
			st = kAdvNext;
			return;
		}
		if (ad2 != 0 && ad1 != 0)
		{
			const float rounded = sd[1] < 0.0f ? floorf(o[1]) : ceilf(o[1]);  // Renderer.cuh:784
			const float tt = div1(vsub(rounded, o[1]), sd[1], srd[1], thr);
			const float shortestPosition = vadd(o[2], vmul(sd[2], tt));
			const int shorterDiff = (int)floorf(shortestPosition) - g[2];
			seq = shorterDiff != 0 ? (2u | (1u << 2)) : (1u | (2u << 2));
		}
		else if (ad1 != 0) seq = 1u;
		else if (ad2 != 0) seq = 2u;
		else seq = 0u;
		st = kAdvNone;
	}

	// ---- the voxel test: doesVoxelSpaceExist + lookupVoxel on region-local walk-space coordinates ---------------------------
	// Returns whether the voxel space exists; col = colour or kEmpty.
	VRM_HD bool voxel_test(RayCtx<ST, STATS>& c, int c0, int c1, int c2, uint32_t& col)
	{
		col = kEmpty;
		if constexpr (ST == kStorageHash)
		{
#if VRM_CC_MUL
			const uint32_t key = (uint32_t)c0 * sh[0] + (uint32_t)c1 * sh[1] + (uint32_t)c2 * sh[2];
#else
			const uint32_t key = ((uint32_t)c0 << sh[0]) | ((uint32_t)c1 << sh[1]) | ((uint32_t)c2 << sh[2]);
#endif
#if VRM_HASH_CLUSTER_FILTER
			if (hash_cluster_occupied(c.sv.clusterMask, r.ri, key))  // negative filter, see lookup_voxel (vrm_core.cuh)
#endif
			{
				// both probes are issued before either compare: a miss (the common case) costs one round trip, not two
				const unsigned long long e1 = ldg(c.sv.slots + (r.base1 + hash_slot1(key, r.seed1, r.n)));
				const unsigned long long e2 = ldg(c.sv.slots + (r.base2 + hash_slot2(key, r.seed2, r.n)));
				if ((uint32_t)(e1 >> 32) == key) col = (uint32_t)e1;
				else if ((uint32_t)(e2 >> 32) == key) col = (uint32_t)e2;
			}
			if (STATS) { c.st.nExist++; c.st.nLookup++; c.st.nProbe2++; if (col != kEmpty) c.st.nLookupHit++; }
			return true;
		}
		else
		{
			// One value carries both codes: cc = cluster id << 9 | in-cluster code.  A coordinate v in [0, 64) contributes
			// (v & 7) | (v >> 3) << 9 = (v * 65) & 0x1E07, shifted to its axis' place.  (Bit 12 of the mask only matters for v = 64, the
			// reference's undefined corner -- a ray rebased onto the far face of a region: it makes this form alias the coordinate
			// into the neighbouring cluster id exactly like the nested form and the C oracle do.)
#if VRM_CC_MUL
			const uint32_t cc = (((uint32_t)c0 * 65u) & 0x1E07u) * sh[0] + (((uint32_t)c1 * 65u) & 0x1E07u) * sh[1] + (((uint32_t)c2 * 65u) & 0x1E07u) * sh[2];
#else
			const uint32_t cc = ((((uint32_t)c0 * 65u) & 0x1E07u) << sh[0]) | ((((uint32_t)c1 * 65u) & 0x1E07u) << sh[1]) | ((((uint32_t)c2 * 65u) & 0x1E07u) << sh[2]);
#endif
			// header word index inside the region = cid * 16 + code / 32 = cc >> 5; bit = code % 32 = cc % 32
#if VRM_VCS_FUSED_EXIST
			// ONE 8-byte load answers both questions: the word's .y carries the cluster-exists flag (vrm_build.cu)
			const uint2 h = ldg(c.sv.headers + ((uint32_t)ri * 8192u + (cc >> 5)));
			const bool e = (h.y & kHeaderClusterExists) != 0;
			if (STATS) { c.st.nExist++; if (!e) c.st.nExistFalse++; }
			if (!e) return false;
#else
			const uint32_t cid = cc >> 9;
#if VRM_SMEM_MASK && defined(__CUDA_ARCH__)
			// the warp's staged copy when this lane is in the staged region, else the mask in global memory
			const uint32_t mw = (c.smMask && ri == c.smRi) ? c.smMask[cid >> 5] : ldg(c.sv.clusterMask + ((uint32_t)ri * 16u + (cid >> 5)));
			const bool e = (mw >> (cid & 31u)) & 1u;
#else
			const bool e = (ldg(c.sv.clusterMask + ((uint32_t)ri * 16u + (cid >> 5))) >> (cid & 31u)) & 1u;
#endif
			if (STATS) { c.st.nExist++; if (!e) c.st.nExistFalse++; }
			if (!e) return false;
			const uint2 h = ldg(c.sv.headers + ((uint32_t)ri * 8192u + (cc >> 5)));
#endif
			const uint32_t bit = cc & 31u;
			if ((h.x >> bit) & 1u)
			{
				col = ldg(c.sv.values + ((h.y & ~kHeaderClusterExists) + (uint32_t)popc32(h.x & ((1u << bit) - 1u))));
#if VRM_COORD64_EMPTY
				// Only the longest-axis walk can ask for a coordinate of exactly 64 (the first tests after entering a region on its far
				// face, see vrm_core.cuh "a coordinate of 64"); the reference's key for it matches no stored voxel.  Applied HERE, after
				// the (in-bounds: the aliased cluster is a real one) load behind the occupancy bit, so that only a lookup that found
				// something pays for it -- the walk through empty space does not.
				if constexpr (kLA) { if (((uint32_t)c0 | (uint32_t)c1 | (uint32_t)c2) & 64u) col = kEmpty; }
#endif
			}
			if (STATS) { c.st.nLookup++; if (col != kEmpty) c.st.nLookupHit++; }
			return true;
		}
	}

	// A voxel was found right after an advance (the voxel under the new position).  Original algorithm: Renderer.cuh:312-315; jump:
	// Renderer.cuh:733-738 (tMin carries +EPSILON there, so the comparison normally falls through to the Z normal).
	// getNormalFromTValues tests X, then Y, else Z.
	VRM_HD void hit_after_advance(RayCtx<ST, STATS>& c, uint32_t col, bool jump)
	{
		const PermRuntime p = unpack_perm(fl);
		int mW = 0;
		if (fl & kFlEq0) mW |= 1 << p.a0;
		if (fl & (kFlEq0 << 1)) mW |= 1 << p.a1;
		if (fl & (kFlEq0 << 2)) mW |= 1 << p.a2;
		const int nAxisW = (mW & 1) ? 0 : ((mW & 2) ? 1 : 2);
		const float dn = p.a0 == nAxisW ? d[0] : (p.a1 == nAxisW ? d[1] : d[2]);  // scaled direction = s * d, s > 0: same sign
		record_hit(c, col, o[0], o[1], o[2], nAxisW, copysignf(1.0f, -dn), jump, g[0], g[1], g[2]);
	}

	// the jump reached a cluster that exists but the voxel is empty: re-snap to the longest axis and `continue` the while loop
	// (Renderer.cuh:742-750)
	VRM_HD void resnap_after_jump()
	{
		const float tNext = div1(vsub(sd[0] > 0.0f ? ceilf(o[0]) : floorf(o[0]), o[0]), sd[0], srd[0], thr);
		const float tt = vadd(tNext, kEps);
		ro[0] = along(o[0], tt, sd[0]); ro[1] = along(o[1], tt, sd[1]); ro[2] = along(o[2], tt, sd[2]);
		ad1 = (int)ro[1] - g[1];
		ad2 = (int)ro[2] - g[2];
		st = kStHead;
	}

	// ---- WARP-UNIFORM FAST PATHS (VCS + longest axis) ----------------------------------------------------------------------
	// The generic kStMain block serves five advance modes with selects and branches; a lockstep simulation of the bench frame
	// (tools/warp_profile.py) shows that in 27 % of a warp's passes EVERY marching lane is in a cluster jump and in ~20 % every
	// marching lane stands at the entry of a null region.  For those passes the warp runs one of the two blocks below: do_main with
	// the mode constant-folded -- the same operations on the same values in the same order, nothing else.  A lane whose step needs
	// anything outside the common case (IEEE slow-path division: unsafe direction, denormal-range or ZERO numerator -- which is
	// also the only way into the crawl fast-forwards, since m == 0 needs a zero numerator) returns false WITHOUT having changed
	// anything; the caller then runs the generic pass for the warp.
	//
	// do_main with mode == kAdvJump: one iteration of performVoxelSpaceJump's loop (Renderer.cuh:707-750)
	VRM_HD bool fast_jump(RayCtx<ST, STATS>& c)
	{
		const float n0 = vadd((float)(int)((uint32_t)g[0] & ~7u), sd[0] > 0.0f ? 8.0f : 0.0f);
		const float n1 = vadd((float)(int)((uint32_t)g[1] & ~7u), sd[1] > 0.0f ? 8.0f : 0.0f);
		const float n2 = vadd((float)(int)((uint32_t)g[2] & ~7u), sd[2] > 0.0f ? 8.0f : 0.0f);
		const float x0 = vsub(n0, o[0]), x1 = vsub(n1, o[1]), x2 = vsub(n2, o[2]);
		if (!(fminf(fabsf(x0), fminf(fabsf(x1), fabsf(x2))) >= thr)) return false;  // div3's slow path (also every m == 0 case)
		const float a0 = div_by_const(x0, sd[0], srd[0]), a1 = div_by_const(x1, sd[1], srd[1]), a2 = div_by_const(x2, sd[2], srd[2]);
		const float s = vadd(min3(a0, a1, a2), kEps);  // the jump guards nothing (Renderer.cuh:457-459) and its tMin includes +EPSILON (713-716)
		o[0] = along(o[0], s, sd[0]); o[1] = along(o[1], s, sd[1]); o[2] = along(o[2], s, sd[2]);
		if (VRM_HORIZON_AT == 0 && past_horizon()) { finish(result); return true; }
		// The equality bits of this advance (which t equals tMin, for the normal) are only ever read by a hit of the voxel test that
		// follows in this very step: the next advance that can precede a hit -- another jump or the original algorithm's kAdvNext --
		// rewrites them, a kAdvCluster only ever follows a kAdvNext, and longest-axis test hits take their normal from the slot.  So
		// they are formed at the hit (0.3 times per ray) instead of at each of the ~9 jumps per ray.
		if (!ray_in_region(o)) { change_region(c); enter_stored_region(c); return true; }
		g[0] = (int)o[0]; g[1] = (int)o[1]; g[2] = (int)o[2];
		uint32_t col;
		const bool e = voxel_test(c, g[0], g[1], g[2], col);
		if (col != kEmpty)
		{
			fl = (fl & ~kFlEqMask) | (a0 == s ? kFlEq0 : 0u) | (a1 == s ? kFlEq0 << 1 : 0u) | (a2 == s ? kFlEq0 << 2 : 0u);
			hit_after_advance(c, col, true);
		}
		else if (e) resnap_after_jump();
		return true;
	}

	// A fast block that changed region runs the new region's entry block right away when the region is stored (prologue of the
	// longest-axis march): the lane is then at the loop head and its next pass can be a longest-axis-stepping pass instead of a
	// generic one (stored-region entries were part of 12 % of the passes, nearly all of them generic because of that one block).
	VRM_HD void enter_stored_region(RayCtx<ST, STATS>& c)
	{
#if VRM_FAST_ENTER
		if (st == kStRegion && ri >= 0) do_region(c);
#endif
	}

	// Longest-axis stepping: every marching lane of the warp is entering a stored region, at the loop head, or has voxel tests of its
	// iteration left (28 % of the passes of the bench frame).  The generic pass minus its advance half and its dispatch; a lane that
	// leaves the pattern (empty cluster -> jump, leaving the region -> original algorithm's tail) just waits for the next pass.
	VRM_HD void fast_la(RayCtx<ST, STATS>& c)
	{
		if ((VRM_FAST_LA & 2) == 0) { if (st == kStRegion) do_region(c); }  // (ri != -1: the caller keeps null regions for fast_nullskip)
		if (st == kStHead) do_head();
		if (st == kAdvNone) do_main<false, kPpOff, true>(c);
	}

	// do_region with ri == -1 followed by do_main with mode == kAdvRegion: skip to the null region's edge, no +EPSILON
	// (Renderer.cuh:384-410, guarded twin 185-211 -- with a finite thr no direction component is zero, so the guards are moot)
	VRM_HD bool fast_nullskip(RayCtx<ST, STATS>& c)
	{
		const float lo = vsub(0.0f, kEps), hi = vadd((float)kRegion, kEps);
		const float x0 = vsub(d[0] > 0.0f ? hi : lo, o[0]), x1 = vsub(d[1] > 0.0f ? hi : lo, o[1]), x2 = vsub(d[2] > 0.0f ? hi : lo, o[2]);  // 0.0f + lo = lo, 0.0f + hi = hi
		if (!(fminf(fabsf(x0), fminf(fabsf(x1), fabsf(x2))) >= thr)) return false;
		const float a0 = div_by_const(x0, d[0], rd[0]), a1 = div_by_const(x1, d[1], rd[1]), a2 = div_by_const(x2, d[2], rd[2]);
		const float s = min3(a0, a1, a2);
		o[0] = along(o[0], s, d[0]); o[1] = along(o[1], s, d[1]); o[2] = along(o[2], s, d[2]);
		if (VRM_HORIZON_AT == 0 && past_horizon()) { finish(result); return true; }
		change_region(c);
		enter_stored_region(c);
		return true;
	}

	// ---- kStMain: [one advance] + one voxel test ------------------------------------------------------------------------
	// NOSKIP: plain execution without the crawl / ping-pong fast-forwards (the fast-forwards use it to probe cycles)
	// TESTONLY: the caller guarantees mode == kAdvNone (fast_la): the advance half is compiled out
	template <bool NOSKIP = false, int PP = kPpDefault, bool TESTONLY = false>
	VRM_HD void do_main(RayCtx<ST, STATS>& c)
	{
		int slot = 0;
		const int mode = st;  // the AdvMode this step starts with (st <= kStMainLast here)
		const bool test = kLA && (TESTONLY || mode == kAdvNone);
		const bool jump = kLA && !TESTONLY && mode == kAdvJump;
		if (!test)
		{
			const bool skip = mode == kAdvRegion;
			float e0 = d[0], e1 = d[1], e2 = d[2], q0 = rd[0], q1 = rd[1], q2 = rd[2];
			if constexpr (kLA) { if (jump) { e0 = sd[0]; e1 = sd[1]; e2 = sd[2]; q0 = srd[0]; q1 = srd[1]; q2 = srd[2]; } }
			float n0, n1, n2;
			if (mode == kAdvNext)
			{
				n0 = next_edge(e0, o[0]); n1 = next_edge(e1, o[1]); n2 = next_edge(e2, o[2]);
			}
			else
			{
				// cluster edge of the voxel of the failed test ((int)o for the original algorithm, gridValues in a jump: g either
				// way), or the region's far face +EPSILON / near face -EPSILON
				const float lo = skip ? vsub(0.0f, kEps) : 0.0f, hi = skip ? vadd((float)kRegion, kEps) : 8.0f;
				const uint32_t keep = skip ? 0u : ~7u;
				n0 = vadd((float)(int)((uint32_t)g[0] & keep), e0 > 0.0f ? hi : lo);
				n1 = vadd((float)(int)((uint32_t)g[1] & keep), e1 > 0.0f ? hi : lo);
				n2 = vadd((float)(int)((uint32_t)g[2] & keep), e2 > 0.0f ? hi : lo);
			}
			float a0, a1, a2;
			div3(vsub(n0, o[0]), vsub(n1, o[1]), vsub(n2, o[2]), e0, e1, e2, q0, q1, q2, thr, a0, a1, a2);
			// zero-direction guards exist only in the shadow routines of the ORIGINAL algorithm: its null-region skip
			// (Renderer.cuh:191-193) and shadowRayMarchVoxelGrid (113-115,137-139,160-162), which also finishes a region for the
			// longest-axis shadow routine (630); the longest-axis jump and null-region skip guard nothing (457-459, 650-652)
			const bool gd = skip ? shadowOriginal() : (jump ? false : shadow());
			if (gd) { a0 = (e0 != 0.0f) ? a0 : INFINITY; a1 = (e1 != 0.0f) ? a1 : INFINITY; a2 = (e2 != 0.0f) ? a2 : INFINITY; }
			float m = min3(a0, a1, a2);
			if (!NOSKIP && m == 0.0f && (mode == kAdvCluster || jump))
			{
				// the ray sits on a cluster face it cannot leave: fast-forward the EPSILON crawl (crawl_skip, vrm_core.cuh)
				const CrawlResult cr = crawl_skip_cold(o[0], o[1], o[2], e0, e1, e2, thr, g[0], g[1], g[2]);
				const int skipped = cr.skipped;
				if constexpr (kLA && ST == kStorageVcs && PP != kPpOff)
				{
					// ... or it also sits exactly on a REGION face and hops between the two regions every iteration (pingpong_skip)
					if (skipped == 0 && jump && (o[1] == 0.0f || o[1] == (float)kRegion || o[2] == 0.0f || o[2] == (float)kRegion))
					{
						if constexpr (PP == kPpInline) { if (pingpong_skip(c)) return; }
						else { if (c.deferQueue) { st = kStPark; return; } }  // nothing has been changed yet: the resume kernel redoes this step
					}
				}
				if (skipped > 0)
				{
					o[0] = cr.o0; o[1] = cr.o1; o[2] = cr.o2;
					if (STATS) { c.st.nExist += skipped; c.st.nExistFalse += skipped; c.st.nCrawlSkipped += skipped; }
					div3(vsub(n0, o[0]), vsub(n1, o[1]), vsub(n2, o[2]), e0, e1, e2, q0, q1, q2, thr, a0, a1, a2);  // same cell, same edges; guards are moot on the fast path
					m = min3(a0, a1, a2);
				}
			}
			const float s = skip ? m : vadd(m, kEps);
			if (mode == kAdvNext || jump)
			{
				// tX,tY,tZ,tMin of Renderer.cuh:273-277 (a cluster skip leaves them stale) / 713-716 (tMin including +EPSILON):
				// all the normal ever asks is which of them equal tMin
				const float tm = jump ? s : m;
				fl = (fl & ~kFlEqMask) | (a0 == tm ? kFlEq0 : 0u) | (a1 == tm ? kFlEq0 << 1 : 0u) | (a2 == tm ? kFlEq0 << 2 : 0u);
			}
			o[0] = along(o[0], s, e0); o[1] = along(o[1], s, e1); o[2] = along(o[2], s, e2);
			// the tails of lit shadow rays are cluster skips / jumps and null-region skips through empty air (primary rays: kHzNever)
			if (VRM_HORIZON_AT == 0 && mode >= kAdvCluster && past_horizon()) { finish(result); return; }
			// grid_in_region((int)floorf(o)) of the jump (Renderer.cuh:719-723) and isRayInRegion(o) agree for every o
			if (skip || !ray_in_region(o)) { change_region(c); return; }
			g[0] = (int)o[0]; g[1] = (int)o[1]; g[2] = (int)o[2];  // == (int)floorf(o) inside a region
		}
		else
		{
			slot = (int)(seq & 3u);
			seq >>= 2;
			g[0] += slot == 0 ? (d[0] < 0.0f ? -1 : 1) : 0;
			g[1] += slot == 1 ? ad1 : 0;
			g[2] += slot == 2 ? ad2 : 0;
		}

		uint32_t col;
		const bool e = voxel_test(c, g[0], g[1], g[2], col);

		if (col != kEmpty)
		{
			if (!test) hit_after_advance(c, col, jump);
			else if constexpr (kLA)
			{
				const PermRuntime p = unpack_perm(fl);
				const float odS = pick3(slot, sd[0], sd[1], sd[2]);
				float p0 = ro[0], p1 = ro[1], p2 = ro[2];  // Renderer.cuh:899
				if (slot != 0)
				{
					// getLocalHitLocation, Renderer.cuh:753-758
					const float ooS = pick3(slot, o[0], o[1], o[2]);
					const float tl = odS > 0.0f ? vdiv(vsub(ceilf(ooS), ooS), odS) : vdiv(vsub(floorf(ooS), ooS), odS);
					p0 = along(o[0], tl, sd[0]); p1 = along(o[1], tl, sd[1]); p2 = along(o[2], tl, sd[2]);
				}
				record_hit(c, col, p0, p1, p2, p.axis(slot), copysignf(1.0f, -odS), true, g[0], g[1], g[2]);
			}
			return;
		}

		// no voxel here: decide the next micro-step
		if (!test)
		{
			if (!jump) st = e ? kAdvNext : kAdvCluster;
			else if (e)
			{
				if constexpr (kLA) resnap_after_jump();
			}
			// else: still no voxel space: another jump iteration (mode stays kAdvJump)
			return;
		}
		if constexpr (kLA)
		{
			if (!e)
			{
				// performVoxelSpaceJump (Renderer.cuh:808-810 -> 696): its while condition repeats the exist check of the failed
				// test on the same voxel -- same answer, only the counter sees it
				if (STATS) { c.st.nExist++; c.st.nExistFalse++; }
				st = kAdvJump;
			}
			else if (slot == 0)
			{
				// the longest axis was this iteration's last test: Renderer.cuh:903-908
				o[0] = ro[0]; o[1] = ro[1]; o[2] = ro[2];
				ro[0] = vadd(ro[0], sd[0]); ro[1] = vadd(ro[1], sd[1]); ro[2] = vadd(ro[2], sd[2]);
				ad1 = (int)ro[1] - g[1];
				ad2 = (int)ro[2] - g[2];
				st = kStHead;
			}
		}
	}

	// ---- kPpDefer: park the ray in the device queue ---------------------------------------------------------------------------
	struct Deferred
	{
		FlatRay ray;
		int32_t* hitOut;               // the pixel's hit-map slot (or null), from the context
		unsigned long long outAddr;    // where the colour goes: filled in by the kernel that queued the ray
		uint32_t outKind;              // 0: three RGB8 bytes, 1: one uint32 colour
		uint32_t pad;
	};
	// Called by the marching wrappers AFTER their loop for a ray that stopped in kStPark.  Returns the queue slot, or -1 when the
	// queue is full (the ray is then back in kStMain and the caller lets it crawl on like the reference).
	VRM_HD int park(RayCtx<ST, STATS>& c)
	{
#if defined(__CUDA_ARCH__)
		DeferHeader* h = static_cast<DeferHeader*>(c.deferQueue);
		const unsigned int slot = atomicAdd(&h->count, 1u);
		st = kAdvJump;  // only a cluster jump parks (do_main): the step that parked is redone
		if (slot >= h->capacity) return -1;
		Deferred* items = reinterpret_cast<Deferred*>(h + 1);
		items[slot].ray = *this;
		items[slot].hitOut = c.hitOut;
		items[slot].outAddr = 0ull;
		st = kStDone;
		return (int)slot;
#else
		st = kAdvJump;
		return -1;
#endif
	}

	// ---- region-face ping-pong fast-forward ---------------------------------------------------------------------------------
	// A second form of the reference's EPSILON crawl (vrm_core.cuh crawl_skip has the first).  Longest-axis cluster jump, one of
	// the short axes stuck on a cluster face (t = 0, so every jump iteration advances by EPSILON * direction only) and the other
	// short axis sitting exactly on a REGION face with a direction component too small to move it: the ray leaves the region
	// by a rounding error, is rebased to local 64 (or 0) in the neighbouring region, runs that region's prologue, loop head and
	// first voxel test (empty cluster), jumps again, leaves again ... two region changes per cycle, ~10^4 cycles per voxel of
	// progress along the longest axis, 10^5-10^6 iterations per ray (4 such pixels made a 1080p frame of the 2048^3 orbit take
	// 710 ms instead of ~2 ms; the reference's own kernels crawl the same way).
	// Per cycle only the longest-axis coordinate changes, by a constant number of ulps (as in crawl_skip); every decision of the
	// cycle is a monotone function of that coordinate (rounded sums / products with constants, truncations, comparisons).  So
	// if the FIRST and the LAST cycle of a span -- both executed here with the ordinary code on a copy of the ray -- take the
	// same decisions, every cycle in between does, and the ray can be moved to the end of the span: bit-identical to executing
	// the cycles.  The span keeps the coordinate inside its voxel and its binade.
	struct Discrete
	{
		int st, g0, g1, g2, ad1, ad2;
		int32_t ri;
		uint32_t ur0, ur1, ur2, seq, fl, o1, o2;
	};
	VRM_HD Discrete discrete() const
	{
		Discrete k;
		k.st = st; k.g0 = g[0]; k.g1 = g[1]; k.g2 = g[2]; k.ad1 = ad1; k.ad2 = ad2; k.ri = ri;
		k.ur0 = ur[0]; k.ur1 = ur[1]; k.ur2 = ur[2]; k.seq = seq; k.fl = fl & ~kFlEqMask; k.o1 = float_bits(o[1]); k.o2 = float_bits(o[2]);
		return k;
	}
	static VRM_HD bool same_discrete(const Discrete& a, const Discrete& b)
	{
		return a.st == b.st && a.g0 == b.g0 && a.g1 == b.g1 && a.g2 == b.g2 && a.ad1 == b.ad1 && a.ad2 == b.ad2 && a.ri == b.ri &&
		       a.ur0 == b.ur0 && a.ur1 == b.ur1 && a.ur2 == b.ur2 && a.seq == b.seq && a.fl == b.fl && a.o1 == b.o1 && a.o2 == b.o2;
	}

	// One half cycle, executed plainly: jump advance that leaves the region -> region entry -> prologue -> head -> first voxel
	// test, which must send the ray back into a jump.
	VRM_HD bool pingpong_half(RayCtx<ST, STATS>& c)
	{
		if constexpr (kLA)
		{
			if (st != kAdvJump) return false;
			do_main<true>(c);
			if (st != kStRegion) return false;
			do_region(c);
			if (st != kStHead) return false;
			do_head();
			if (st != kAdvNone) return false;
			do_main<true>(c);
			return st == kAdvJump;
		}
		return false;
	}

	// Returns true when the ray was moved forward by whole cycles (it is then again in kStMain / kAdvJump, before an advance).
	VRM_FLAT_COLD bool pingpong_skip(RayCtx<ST, STATS>& c)
	{
		if (!(thr == thr)) return false;
		const uint32_t xb = float_bits(o[0]), eb = xb >> 23;
		if (eb < 24u || eb > 140u) return false;
		const float c0 = vmul(kEps, sd[0]);
		const float cu = vmul(c0, bits_float((277u - eb) << 23));  // advance per iteration in ulps of o[0]
		if (!(fabsf(cu) < 1048576.0f)) return false;
		int q;
		const float cuFloor = floorf(cu);
		if (vsub(cu, cuFloor) == 0.5f)
		{
			if (xb & 1u) return false;  // exact tie from an odd mantissa: one ordinary iteration makes it even (see crawl_skip)
			const int k = (int)cuFloor;
			q = (k & 1) ? k + 1 : k;
		}
		else q = (int)rintf(cu);
		if (q == 0) return false;
		// o[0] must stay strictly inside its voxel (the prologue truncates it) and its binade (constant ulp)
		const int v0 = (int)o[0];
		uint32_t lo = float_bits((float)v0), hi = float_bits((float)(v0 + 1));
		const uint32_t blo = eb << 23, bhi = (eb + 1u) << 23;
		if (lo < blo) lo = blo;
		if (hi > bhi) hi = bhi;
		if (xb < lo || xb >= hi) return false;
		if (lo == blo) lo = blo + 1u;  // a step down must land strictly above the binade's first float (see crawl_skip)
		const uint32_t room = q > 0 ? (hi - 1u - xb) / (uint32_t)q : (xb >= lo ? (xb - lo) / (uint32_t)(-q) : 0u);  // advances that keep o[0] inside
		const uint32_t cycles = room / 2u;  // whole cycles that keep o[0] inside
		if (cycles < 4u) return false;
		const FlatRay start = *this;
		const Stats saved = c.st;
		const Discrete k0 = discrete();
		bool ok = pingpong_half(c);
		const Discrete kA = discrete();
		const uint32_t xA = float_bits(o[0]);
		ok = ok && (int32_t)(xA - xb) == q && pingpong_half(c);
		const Discrete kB = discrete();
		ok = ok && (int32_t)(float_bits(o[0]) - xA) == q && same_discrete(kB, k0);
		const Stats per = c.st;
		// Cycle number m (1-based) starts (m - 1) cycles after `start`.  "Cycle m takes the decisions of cycle 1" is monotone in m
		// (see above), so the cycles that do form a prefix 1..good: binary search for its end with one probed cycle per step.
		uint32_t good = 1u, bad = cycles + 1u;
		while (ok && bad - good > 1u)
		{
			const uint32_t mid = good + (bad - good) / 2u;
			*this = start;
			const uint32_t xl = xb + (mid - 1u) * 2u * (uint32_t)q;
			o[0] = bits_float(xl);
			bool same = pingpong_half(c) && same_discrete(discrete(), kA) && (int32_t)(float_bits(o[0]) - xl) == q;
			const uint32_t xm = float_bits(o[0]);
			same = same && pingpong_half(c) && same_discrete(discrete(), kB) && (int32_t)(float_bits(o[0]) - xm) == q;
			if (same) good = mid; else bad = mid;
		}
		if (ok && good >= 3u)
		{
			// the state after `good` cycles: execute cycle `good` once more (plainly) from its start
			*this = start;
			o[0] = bits_float(xb + (good - 1u) * 2u * (uint32_t)q);
			ok = pingpong_half(c) && pingpong_half(c);
		}
		else ok = false;
		if (!ok)
		{
			*this = start;
			c.st = saved;
			return false;
		}
		const uint32_t done = good;
		if (STATS)
		{
			// counters: `done` times what one cycle added
			const unsigned long long n = done;
			Stats t = saved;
			t.nExist += n * (per.nExist - saved.nExist); t.nExistFalse += n * (per.nExistFalse - saved.nExistFalse);
			t.nLookup += n * (per.nLookup - saved.nLookup); t.nLookupHit += n * (per.nLookupHit - saved.nLookupHit);
			t.nProbe2 += n * (per.nProbe2 - saved.nProbe2); t.nRegionReads += n * (per.nRegionReads - saved.nRegionReads);
			t.nCrawlSkipped = saved.nCrawlSkipped + n * (per.nExist - saved.nExist);
			c.st = t;
		}
		return true;
	}

	// Run the blocks the ray's state asks for, in program order.  Returns true when the pixel is resolved.
	template <int PP = kPpDefault>
	VRM_HD bool step(RayCtx<ST, STATS>& c)
	{
		if (st == kStHit) do_hit(c);
		if (st == kStRegion) do_region(c);
		if constexpr (kLA) { if (st == kStHead) do_head(); }
		if (st <= kStMainLast) do_main<false, PP>(c);
		return st == kStDone;
	}

	// step() with the warp-uniform fast paths taken per ray whenever they apply: what a warp whose lanes all qualify executes
	// (host harness: the CPU tier checks the fast paths against the oracle this way, tests/test_hostsim.py form "fast")
	template <int PP = kPpDefault>
	VRM_HD bool step_fast(RayCtx<ST, STATS>& c)
	{
		if constexpr (kLA && ST == kStorageVcs)
		{
			if (st == kAdvJump) { if (fast_jump(c)) return st == kStDone; }
			else if (st == kStRegion && ri == -1) { if (fast_nullskip(c)) return st == kStDone; }
			else if (st == kStHead || st == kAdvNone || ((VRM_FAST_LA & 2) == 0 && st == kStRegion)) { fast_la(c); return st == kStDone; }
		}
		return step<PP>(c);
	}

	// the marching blocks only (region -> head -> main); hits are shaded by the caller
	template <int PP = kPpDefault>
	VRM_HD void step_marching(RayCtx<ST, STATS>& c)
	{
		if (st == kStRegion) do_region(c);
		if constexpr (kLA) { if (st == kStHead) do_head(); }
		if (st <= kStMainLast) do_main<false, PP>(c);
	}
};

// One pass of the marching blocks for a whole warp (all 32 lanes call it; lanes that are not marching idle).
// VRM_REGION_VOTE / VRM_HEAD_VOTE > 0 (A/B variants): the region-entry / loop-head block of a pass runs only when enough lanes want it
// or nobody has anything else to do; the lanes that wait keep their state and run with the lanes that join them in a later pass.
// Progress: the main block always runs when a lane wants it; without such a lane the head block does; else the region block.
template <int ST, int ALGO, bool STATS, int PP>
VRM_HD void warp_march_pass(RayCtx<ST, STATS>& c, FlatRay<ST, ALGO, STATS>& ray)
{
#if defined(__CUDA_ARCH__) && (VRM_REGION_VOTE > 0 || VRM_HEAD_VOTE > 0)
	const unsigned wantRegion = __ballot_sync(0xFFFFFFFFu, ray.st == kStRegion);
	const unsigned others = __ballot_sync(0xFFFFFFFFu, ray.st == kStHead || ray.st <= kStMainLast);
	if (wantRegion != 0u && (VRM_REGION_VOTE <= 0 || __popc(wantRegion) >= VRM_REGION_VOTE || others == 0u)) { if (ray.st == kStRegion) ray.do_region(c); }
	if constexpr (ALGO != kAlgoOriginal)
	{
		const unsigned wantHead = __ballot_sync(0xFFFFFFFFu, ray.st == kStHead);
		const unsigned wantMain = __ballot_sync(0xFFFFFFFFu, ray.st <= kStMainLast);
		if (wantHead != 0u && (VRM_HEAD_VOTE <= 0 || __popc(wantHead) >= VRM_HEAD_VOTE || wantMain == 0u)) { if (ray.st == kStHead) ray.do_head(); }
	}
	if (ray.st <= kStMainLast) ray.template do_main<false, PP>(c);
#else
	if (ray.st <= kStHead) ray.template step_marching<PP>(c);
#endif
}

// Warp-cooperative form for the render kernels: all 32 lanes of a warp call it together (lanes without a pixel pass
// active = false) and one ballot per iteration decides what the warp runs.
// HIT BARRIER: lanes whose primary ray has hit wait in kStHit until every lane of the warp has hit or finished; the whole
// tile then shades and starts its shadow rays in the same iteration.  The shadow rays of a tile share one direction and
// neighbouring origins, so they walk in lockstep instead of being interleaved with late primary rays (measured on the 4K
// terrain frame, VCS + longest axis: 1.62 -> 1.53 ms; a further barrier at region changes measured no gain and was dropped).
// Only the interleaving of different rays' operations changes; every ray executes exactly the operations it always did.
// deferredSlot: the ray's slot in the defer queue when it was parked there (its colour is then not final), else -1
template <int ST, int ALGO, bool STATS, int PP>
VRM_HD uint32_t march_scene_flat_warp(RayCtx<ST, STATS>& c, bool active, const float* originW, const float* dirW, float scale, int& deferredSlot)
{
	FlatRay<ST, ALGO, STATS> ray;
	ray.st = kStDone; ray.result = 0;
	if (active) ray.start_primary(c, originW, dirW, scale);
#if defined(__CUDA_ARCH__)
#if VRM_FAST_PATHS
	if constexpr (ALGO != kAlgoOriginal && ST == kStorageVcs)
	{
		bool generic = false;  // warp-uniform: a lane's step did not qualify for the fast path it was offered
		for (;;)
		{
#if VRM_SMEM_MASK
			if (c.smMask)
			{
				// stage the cluster mask of the region the first marching lane is in (the lanes of a tile mostly share it)
				const unsigned inRegion = __ballot_sync(0xFFFFFFFFu, ray.st <= kStHead && ray.ri >= 0);
				if (inRegion != 0u)
				{
					const int32_t want = __shfl_sync(0xFFFFFFFFu, ray.ri, __ffs(inRegion) - 1);
					if (want != c.smRi)
					{
						__syncwarp();
						if ((threadIdx.x & 31u) < 16u) c.smMask[threadIdx.x & 31u] = ldg(c.sv.clusterMask + ((uint32_t)want * 16u + (threadIdx.x & 31u)));
						c.smRi = want;
						__syncwarp();
					}
				}
			}
#endif
			// what the warp's marching lanes (kStMain, kStRegion, kStHead) are about to do: a cluster jump, a null-region skip, longest-axis
			// stepping (loop head, a voxel test of the current iteration; with VRM_FAST_LA & 2 == 0 also a stored-region entry) or anything
			// else.
			constexpr unsigned kClsJump = 0x10u, kClsNull = 0x20u, kClsOther = 0x40u, kClsLa = 0x80u;
			const bool isJump = ray.st == kAdvJump, isNull = ray.st == kStRegion && ray.ri == -1;
#if VRM_FAST_LA
			const bool isLa = ray.st == kStHead || ray.st == kAdvNone || ((VRM_FAST_LA & 2) == 0 && ray.st == kStRegion && ray.ri != -1);
#if VRM_CLS_LUT
			// the class is a function of the state word alone (one nibble per state, already in place: kAdvNone la, kAdvNext other,
			// kAdvCluster other, kAdvJump jump, kAdvRegion other, kStRegion other (la when fast_la runs stored-region entries), kStHead la,
			// the rest 0) except for the null-region entry
			// (a clamped funnel shift: states 8 and 9 shift the table out completely)
			const unsigned nib = __funnelshift_rc((VRM_FAST_LA & 2) ? 0x84414480u : 0x88414480u, 0u, (unsigned)ray.st * 4u) & 0xF0u;
			const unsigned cls = isNull ? kClsNull : nib;
			(void)isJump; (void)isLa;
#else
			const unsigned cls = ray.st <= kStHead ? (isJump ? kClsJump : (isNull ? kClsNull : (isLa ? kClsLa : kClsOther))) : 0u;
#endif
#else
			const unsigned cls = ray.st <= kStHead ? (isJump ? kClsJump : (isNull ? kClsNull : kClsOther)) : 0u;
#endif
			const unsigned all = __reduce_or_sync(0xFFFFFFFFu, cls);
			// Four equality tests on one value become a jump table (a constant-bank load + BRX, ~17 times per tile, each a dependent
			// latency behind the reduction): the jump / null-region tests below read an opaque copy, so the compiler sees two chains of two.
			unsigned all2 = all;
#if defined(__CUDA_ARCH__)
			asm volatile("mov.u32 %0, %1;" : "=r"(all2) : "r"(all));
#endif
#if VRM_FAST_LA
			if (all == kClsLa)
			{
				for (;;)
				{
					ray.fast_la(c);
					if (VRM_FAST_LA & 4) break;
					const bool la = ray.st == kStHead || ray.st == kAdvNone || ((VRM_FAST_LA & 2) == 0 && ray.st == kStRegion && ray.ri != -1);
					const unsigned stay = __ballot_sync(0xFFFFFFFFu, la);
					const unsigned leave = __ballot_sync(0xFFFFFFFFu, ray.st <= kStHead && !la);
					if (leave != 0u || stay == 0u) break;
				}
				continue;
			}
#endif
			if (all == 0u)
			{
				// nobody is marching: every lane is waiting with a hit, done or parked
				if (!__any_sync(0xFFFFFFFFu, ray.st == kStHit)) break;
				if (ray.st == kStHit) ray.do_hit(c);
				continue;
			}
#if VRM_FAST_LOOPS
			// The warp stays in a fast block for as long as every marching lane still qualifies (two votes per pass instead of the
			// classification above): fast_jump leaves a lane in kStMain / kAdvJump, or in kStRegion / kStHead / kStHit; fast_nullskip
			// leaves it in kStRegion.
			if (all2 == kClsJump || all2 == kClsNull)
			{
				// a lane whose step did not qualify for the fast path it was offered (it changed nothing) sends the warp through the
				// generic pass below, once
				bool bad;
				if (all2 == kClsJump)
				{
					for (;;)
					{
						bool ok = true;
						if (ray.st == kAdvJump) ok = ray.fast_jump(c);
						const unsigned stay = __ballot_sync(0xFFFFFFFFu, ok && ray.st == kAdvJump);
						const unsigned leave = __ballot_sync(0xFFFFFFFFu, !ok || ray.st == kStRegion || ray.st == kStHead);
						if (leave != 0u || stay == 0u) { bad = __any_sync(0xFFFFFFFFu, !ok); break; }
					}
				}
				else
				{
					for (;;)
					{
						bool ok = true;
						if (ray.st == kStRegion) ok = ray.fast_nullskip(c);
						const unsigned stay = __ballot_sync(0xFFFFFFFFu, ok && ray.st == kStRegion && ray.ri == -1);
						const unsigned leave = __ballot_sync(0xFFFFFFFFu, !ok || (ray.st <= kStHead && !(ray.st == kStRegion && ray.ri == -1)));
						if (leave != 0u || stay == 0u) { bad = __any_sync(0xFFFFFFFFu, !ok); break; }
					}
				}
				if (!bad) continue;
			}
#else
			if (!generic && all == kClsJump)
			{
				bool ok = true;
				if (isJump) ok = ray.fast_jump(c);
				generic = __any_sync(0xFFFFFFFFu, !ok);
				continue;
			}
			if (!generic && all == kClsNull)
			{
				bool ok = true;
				if (isNull) ok = ray.fast_nullskip(c);
				generic = __any_sync(0xFFFFFFFFu, !ok);
				continue;
			}
#endif
			warp_march_pass<ST, ALGO, STATS, PP>(c, ray);
			generic = false;
		}
	}
	else
#endif
	for (;;)
	{
		const unsigned marching = __ballot_sync(0xFFFFFFFFu, ray.st <= kStHead);  // kStMain, kStRegion, kStHead
		if (marching != 0u)
		{
			warp_march_pass<ST, ALGO, STATS, PP>(c, ray);
			continue;
		}
		// nobody is marching: every lane is waiting with a hit, done or parked
		if (!__any_sync(0xFFFFFFFFu, ray.st == kStHit)) break;
		if (ray.st == kStHit) ray.do_hit(c);
	}
#else
	while (ray.st < kStDone) ray.template step<PP>(c);
#endif
	deferredSlot = -1;
	if constexpr (PP == kPpDefer && ST == kStorageVcs && ALGO != kAlgoOriginal)  // the only combination that can park (do_main)
	{
		if (ray.st == kStPark)
		{
			deferredSlot = ray.park(c);
			if (deferredSlot < 0) { while (ray.st < kStDone) ray.template step<kPpOff>(c); }  // queue full: crawl on like the reference
			else ray.result = 0u;
		}
	}
	return ray.result;
}

// PRIMARY phase only, warp-cooperative (render kernels with the shadow-ray queue, vrm_render.cu): every lane marches its primary ray
// until it has hit (kStHit, waiting to be shaded by the caller), finished (kStDone) or must be parked (kStPark).  No hit barrier is
// needed: the shadow rays run in their own kernel, compacted.
template <int ST, int ALGO, bool STATS, int PP>
VRM_HD void march_primary_flat_warp(RayCtx<ST, STATS>& c, bool active, const float* originW, const float* dirW, float scale, FlatRay<ST, ALGO, STATS>& ray)
{
	ray.st = kStDone; ray.result = 0;
	if (active) ray.start_primary(c, originW, dirW, scale);
#if defined(__CUDA_ARCH__)
	while (__any_sync(0xFFFFFFFFu, ray.st <= kStHead)) warp_march_pass<ST, ALGO, STATS, PP>(c, ray);
#else
	while (ray.st <= kStHead) ray.template step_marching<PP>(c);
#endif
}

// SHADOW phase of one queue record, warp-cooperative: returns the pixel's final colour (ss.lit or 0); the ray may end in kStPark.
template <int ST, int ALGO, bool STATS, int PP>
VRM_HD void march_shadow_flat_warp(RayCtx<ST, STATS>& c, bool active, const ShadowStart& ss, FlatRay<ST, ALGO, STATS>& ray)
{
	ray.st = kStDone; ray.result = 0;
	if (active) ray.start_shadow(c, ss);
#if defined(__CUDA_ARCH__)
	while (__any_sync(0xFFFFFFFFu, ray.st <= kStHead)) warp_march_pass<ST, ALGO, STATS, PP>(c, ray);
#else
	while (ray.st <= kStHead) ray.template step_marching<PP>(c);
#endif
}

// Convenience for single-ray callers (trace kernels, host sim): run the state machine to completion.
template <int ST, int ALGO, bool STATS, int PP = kPpDefault>
VRM_HD uint32_t march_scene_flat(RayCtx<ST, STATS>& c, const float* originW, const float* dirW, float scale, int& deferredSlot)
{
	FlatRay<ST, ALGO, STATS> ray;
	ray.start_primary(c, originW, dirW, scale);
	while (ray.st < kStDone) ray.template step<PP>(c);
	deferredSlot = -1;
	if constexpr (PP == kPpDefer && ST == kStorageVcs && ALGO != kAlgoOriginal)  // the only combination that can park (do_main)
	{
		if (ray.st == kStPark)
		{
			deferredSlot = ray.park(c);
			if (deferredSlot < 0) { while (ray.st < kStDone) ray.template step<kPpOff>(c); }  // queue full: crawl on like the reference
			else ray.result = 0u;
		}
	}
	return ray.result;
}

template <int ST, int ALGO, bool STATS>
VRM_HD uint32_t march_scene_flat(RayCtx<ST, STATS>& c, const float* originW, const float* dirW, float scale)
{
	int unused;
	return march_scene_flat<ST, ALGO, STATS, kPpDefault>(c, originW, dirW, scale, unused);
}

// The same with the fast paths taken whenever a ray qualifies (host harness)
template <int ST, int ALGO, bool STATS>
VRM_HD uint32_t march_scene_flat_fast(RayCtx<ST, STATS>& c, const float* originW, const float* dirW, float scale)
{
	FlatRay<ST, ALGO, STATS> ray;
	ray.start_primary(c, originW, dirW, scale);
	while (ray.st < kStDone) ray.template step_fast<kPpDefault>(c);
	return ray.result;
}

}  // namespace vrm
