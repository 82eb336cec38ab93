// vrm_core.cuh -- per-ray traversal core of the B200-native voxel raymarcher.
//
// Everything here is __host__ __device__ so that tests/hostsim can compile the very same source for the CPU and
// single-step it against the oracle; the product only ever runs it inside the sm_100a kernels of vrm_render.cu.
//
// Design (see DESIGN.md):
//  * "Walk space": a ray is stored with its axes permuted so that slot 0/1/2 are the longest/middle/shortest
//    direction axes (identity permutation for the "original" algorithm).  Every per-component operation of the
//    reference is axis-symmetric, so the arithmetic is bit-identical, but the longest-axis algorithm's
//    dynamically indexed gridValues[axis]/axisDiff[axis] (local-memory traffic in the reference build:
//    1092 LDL / 1844 STL, SURVEY.md §2.1) become plain registers.  Only the storage code and the region-table
//    index are computed through three per-ray shift/stride registers.
//  * No virtual dispatch, no function pointers: storage type and algorithm are template parameters.
//  * IEEE fp32 with NO contraction: every float op goes through vadd/vsub/vmul/vdiv (the *_rn intrinsics on the
//    device), mirroring the reference's operation order exactly (SURVEY.md §7 hard part 1).
//
// Reference file:line citations are relative to /root/reference/VoxelRaymarcher/src.
#pragma once

#ifndef VRM_SMEM_MASK
#define VRM_SMEM_MASK 0  // 1 (with VRM_VCS_FUSED_EXIST=0): per-warp shared-memory copy of the current region's cluster mask in the fused render kernel (measured, off)
#endif

#include <stdint.h>
#include <math.h>
#include <string.h>
#include <type_traits>

#if defined(__CUDACC__)
#define VRM_HD __host__ __device__ __forceinline__
#define VRM_HD_NOINLINE static __host__ __device__ __noinline__
#else
#define VRM_HD inline
#define VRM_HD_NOINLINE static inline
#endif

namespace vrm
{

constexpr float kEps = 0.0001f;                // EPSILON, geometry/VoxelFunctions.cuh:19
constexpr uint32_t kEmpty = 1u << 30;          // EMPTY_KEY / EMPTY_VAL, geometry/VoxelFunctions.cuh:20-21
constexpr uint32_t kContinue = kEmpty + 2u;    // CONTINUE_VAL, geometry/VoxelFunctions.cuh:23
constexpr int kRegion = 64;                    // BLOCK_SIZE, geometry/VoxelFunctions.cuh:24
constexpr int kStorageVcs = 0, kStorageHash = 1;  // StorageType, geometry/VoxelFunctions.cuh:37
constexpr int kAlgoLongestAxis = 0, kAlgoOriginal = 1;  // main/Main.cu:58-68
constexpr unsigned long long kEmptySlot = 0xFFFFFFFFFFFFFFFFull;
constexpr uint32_t kHeaderClusterExists = 0x80000000u;  // VCS header word, .y: the word's cluster holds at least one voxel (low 31 bits: index of the word's first colour)

// ---------------------------------------------------------------- non-contracting fp32

#if defined(__CUDA_ARCH__)
VRM_HD float vadd(float a, float b) { return __fadd_rn(a, b); }
VRM_HD float vsub(float a, float b) { return __fsub_rn(a, b); }
VRM_HD float vmul(float a, float b) { return __fmul_rn(a, b); }
VRM_HD float vdiv(float a, float b) { return __fdiv_rn(a, b); }
VRM_HD float vsqrt(float a) { return __fsqrt_rn(a); }
VRM_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return __umulhi(a, b); }
VRM_HD int popc32(uint32_t a) { return __popc(a); }
#else
// Host build (tests/hostsim only): compiled with -ffp-contract=off.
VRM_HD float vadd(float a, float b) { return a + b; }
VRM_HD float vsub(float a, float b) { return a - b; }
VRM_HD float vmul(float a, float b) { return a * b; }
VRM_HD float vdiv(float a, float b) { return a / b; }
VRM_HD float vsqrt(float a) { return sqrtf(a); }
VRM_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
VRM_HD int popc32(uint32_t a) { return __builtin_popcount(a); }
#endif

VRM_HD float min3(float a, float b, float c) { return fminf(a, fminf(b, c)); }
// o + t * d, the reference's  origin + (t * direction)  (math/Vector3.cuh:105-109,134-138)
VRM_HD float along(float o, float t, float d) { return vadd(o, vmul(t, d)); }

// ---------------------------------------------------------------- exact division by a per-ray constant
//
// The walk divides by the three direction components at every step ("t = (next - o) / d", Renderer.cuh:273-275 and
// siblings) and those divisors never change along a ray.  IEEE division (div.rn.f32) costs ~12 issue slots on sm_100a
// (MUFU.RCP + 5 FFMA + FCHK + slow-path branch); with y = RN(1/d) computed once per ray the correctly rounded quotient is
//     q0 = RN(x * y);  r = x - d * q0  (one FMA, exact);  q = RN(q0 + r * y)            (Markstein)
// i.e. 3 issue slots.  Before rounding, q0 + r*y = (x/d)(1 - e1*(e1+e2+e1*e2)) with |e1|,|e2| <= 2^-24, a relative
// perturbation below 2^-47; the result was checked equal to x/d for all 2^23 numerator mantissas against 200 000
// denominators (1.7e12 cases, incl. all-ones / sparse mantissas) and on 2.4e9 adversarial near-midpoint quotients.
// This is the SAME value as the reference's division, not an approximation: parity stays bit-exact.
//
// Preconditions (else fall back to div.rn): d normal with 2^-40 <= |d| <= 2^40 (so y, q are far from over/underflow) and
// every numerator either exactly 0 or |x| >= 2^-100 (so that the residual r cannot underflow).  One compare per step
// covers both: thr is 2^-100 for a "fast" ray and NaN otherwise, and the slow path is taken unless min|x_i| >= thr.
// (An exactly zero numerator also takes the slow path; it is rare -- a ray exactly on a cluster face.)
#if defined(__CUDA_ARCH__)
VRM_HD float vfma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
VRM_HD float vrcp(float a) { return __frcp_rn(a); }
#else
VRM_HD float vfma(float a, float b, float c) { return fmaf(a, b, c); }
VRM_HD float vrcp(float a) { return 1.0f / a; }
#endif

struct RayDir
{
	float d[3];   // direction, walk space
	float rd[3];  // RN(1 / d)
	float thr;    // fast-division threshold (see above)
};

VRM_HD bool dir_component_safe(float v)
{
	float a = fabsf(v);
	return a >= 9.094947017729282e-13f && a <= 1.099511627776e12f;  // 2^-40 .. 2^40 (false for 0, inf, NaN, denormals)
}

VRM_HD RayDir make_raydir(float d0, float d1, float d2)
{
	RayDir k;
	k.d[0] = d0; k.d[1] = d1; k.d[2] = d2;
	k.rd[0] = vrcp(d0); k.rd[1] = vrcp(d1); k.rd[2] = vrcp(d2);
	const bool fast = dir_component_safe(d0) && dir_component_safe(d1) && dir_component_safe(d2);
	k.thr = fast ? 7.888609052210118e-31f : NAN;  // 2^-100
	return k;
}

VRM_HD float div_by_const(float x, float d, float rd)
{
	float q0 = vmul(x, rd);
	float r = vfma(-d, q0, x);
	return vfma(r, rd, q0);
}

// a_i = x_i / d_i, bit-identical to IEEE division
VRM_HD void div3(float x0, float x1, float x2, const RayDir& k, float& a0, float& a1, float& a2)
{
	float m = fminf(fabsf(x0), fminf(fabsf(x1), fabsf(x2)));
	if (!(m >= k.thr))
	{
		a0 = vdiv(x0, k.d[0]); a1 = vdiv(x1, k.d[1]); a2 = vdiv(x2, k.d[2]);
	}
	else
	{
		a0 = div_by_const(x0, k.d[0], k.rd[0]); a1 = div_by_const(x1, k.d[1], k.rd[1]); a2 = div_by_const(x2, k.d[2], k.rd[2]);
	}
}

// VRM_COLD_OUTLINE=1 keeps IEEE division (and the crawl fast-forward) OUT of line: the slow branches below run for a handful of rays per frame, and three inlined div.rn
// expansions per site sit in the middle of the hot loop instruction stream.  Measured: no difference (1.588 vs 1.582 ms), so inline stays the default
#ifndef VRM_COLD_OUTLINE
#define VRM_COLD_OUTLINE 0
#endif
#if VRM_COLD_OUTLINE
VRM_HD_NOINLINE float vdiv_cold(float a, float b) { return vdiv(a, b); }
#else
VRM_HD float vdiv_cold(float a, float b) { return vdiv(a, b); }
#endif

// the same with the constants passed one by one (vrm_flat.cuh keeps them in individual registers)
VRM_HD void div3(float x0, float x1, float x2, float d0, float d1, float d2, float r0, float r1, float r2, float thr, float& a0, float& a1, float& a2)
{
	float m = fminf(fabsf(x0), fminf(fabsf(x1), fabsf(x2)));
	if (!(m >= thr))
	{
		a0 = vdiv_cold(x0, d0); a1 = vdiv_cold(x1, d1); a2 = vdiv_cold(x2, d2);
	}
	else
	{
		a0 = div_by_const(x0, d0, r0); a1 = div_by_const(x1, d1, r1); a2 = div_by_const(x2, d2, r2);
	}
}

VRM_HD float div1(float x, float d, float rd, float thr)
{
	if (!(fabsf(x) >= thr)) return vdiv_cold(x, d);
	return div_by_const(x, d, rd);
}

VRM_HD float div1(float x, const RayDir& k, int i)
{
	float ax = fabsf(x);
	if (!(ax >= k.thr)) return vdiv(x, k.d[i]);
	return div_by_const(x, k.d[i], k.rd[i]);
}

// ---------------------------------------------------------------- scene description (device pointers)

struct Lighting
{
	float dir[3];    // LIGHT_DIRECTION
	float color[3];  // LIGHT_COLOR
	float pos[3];    // LIGHT_POSITION
	int usePoint;    // USE_POINT_LIGHT
	int useShadows;  // USE_SHADOWS
};

// The light direction prepared for the shadow rays of the state machine (vrm_flat.cuh make_light_walk; host-computed):
// id* = world axis order (original-algorithm shadow routine), la* = ranked longest / middle / shortest order.
struct LightWalk
{
	float idD[3], idR[3], idThr;
	float laD[3], laR[3], laSD[3], laSR[3], laThr;
	uint32_t laPerm;  // pack_perm() of the ranked order
};

// ---- shadow horizon map --------------------------------------------------------------------------------------------------
// A shadow ray's whole result is one bit (colour * !inShadow) and it travels along the light direction n.  The map is a 2D grid on
// the plane perpendicular to n; a cell holds an upper bound of dot(X, n) over every point X of every occupied 8^3 cluster whose
// projection, widened by kHorizonR, covers the cell.  A shadow ray looks its start point up once (every later point of its line
// projects to the same place) and, once its depth along n is past the cell's value plus kHorizonMargin, no voxel test it can still
// make can find an occupied cluster: it finishes lit, exactly as the full walk out of the scene would.
// Coordinates are relative to the region table's origin (64 * minCoord), so scenes near +-2^23 lose nothing.
//
// kHorizonR bounds how far off the ray's exact line a tested voxel can lie, kHorizonMargin how far AHEAD along n (both in voxels):
//   - any point of a tested voxel cube [g, g + 1]^3 lies within sqrt(3) of the ray point g was taken from (truncation);
//   - the longest-axis walk tests g + axisDiff, taken from its origin `ro`, which runs up to one scaled step (|sd| <= sqrt(3)) ahead
//     of o; its prologue steps back by at most one voxel, and the first voxel test after entering a region takes the voxel under the
//     rebased position (coordinate up to 64, aliased into the same cluster grid);
//   - fp32 drift of the walk in region-local coordinates: each advance rounds every coordinate by <= 2^-18 (|o| <= 64) and a ray
//     makes far fewer than 10^4 advances outside crawls; a crawl (t = 0 on a face) cannot slide along a face for more than one
//     iteration per axis when every non-zero |n_i| >= kHorizonMinComponent (kEps * |n_i| moves the coordinate off the face), which
//     horizon_setup requires -- other lights get no map;
//   - projection and lookup in fp32 (coordinates < 2^18): < 0.05; the splat adds one more voxel of padding for it.
// sqrt(3) + sqrt(3) + 1 + drift < 4.5: R = 5 and margin = 5 voxels.  (The cell is 8+ voxels wide, so a larger R costs little.)
constexpr float kHorizonR = 5.0f;
constexpr float kHorizonMargin = 5.0f;
constexpr float kHorizonClusterR = 6.92820323f;    // 4 * sqrt(3): circumradius of an 8^3 cluster around its centre
constexpr double kHorizonMinComponent = 0.0625;    // lights with 0 < |n_i| < this get no map (see above)
constexpr uint32_t kHorizonMaxCells = 2048;        // per side: the cell grows past 8 voxels for scenes wider than that
constexpr int32_t kHorizonEmpty = (int32_t)0x80808080u;  // a cell no cluster covers (below every real value; a byte memset fills it)

struct HorizonView
{
	const int32_t* cells;  // [nv][nu] ceil(max dot(X, n)) over the covering clusters, kHorizonEmpty if none; null: no map (rays walk out)
	float n[3];            // unit light direction, world axes
	float e1[3], e2[3];    // orthonormal basis of the plane perpendicular to n
	float u0, v0, invCell; // cell (iu, iv) = floor((dot(X, e1) - u0) * invCell), floor((dot(X, e2) - v0) * invCell)
	uint32_t nu, nv;
	int axis;              // world axis of the largest |n_i|: the coordinate a shadow ray's threshold is stated in
};

// Grid for a scene of diameter D regions and light direction dir (host, double).  Returns false when the light gets no map.
inline bool horizon_setup(const float* dir, uint32_t D, uint32_t permAxis0, HorizonView& h)
{
	h.cells = nullptr;
	const double l = sqrt((double)dir[0] * dir[0] + (double)dir[1] * dir[1] + (double)dir[2] * dir[2]);
	if (!(l > 0.0) || D == 0u) return false;
	double n[3];
	for (int i = 0; i < 3; i++)
	{
		n[i] = dir[i] / l;
		if (n[i] != 0.0 && fabs(n[i]) < kHorizonMinComponent) return false;
	}
	const int k = fabs(n[0]) <= fabs(n[1]) ? (fabs(n[0]) <= fabs(n[2]) ? 0 : 2) : (fabs(n[1]) <= fabs(n[2]) ? 1 : 2);  // least aligned axis
	double a[3] = {0.0, 0.0, 0.0};
	a[k] = 1.0;
	double e1[3] = {n[1] * a[2] - n[2] * a[1], n[2] * a[0] - n[0] * a[2], n[0] * a[1] - n[1] * a[0]};
	const double l1 = sqrt(e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2]);
	for (int i = 0; i < 3; i++) e1[i] /= l1;
	const double e2[3] = {n[1] * e1[2] - n[2] * e1[1], n[2] * e1[0] - n[0] * e1[2], n[0] * e1[1] - n[1] * e1[0]};
	const double side = 64.0 * D, pad = kHorizonClusterR + kHorizonR + 2.0;
	double umin = 1e300, umax = -1e300, vmin = 1e300, vmax = -1e300;
	for (int c = 0; c < 8; c++)
	{
		const double p[3] = {(c & 1) ? side : 0.0, (c & 2) ? side : 0.0, (c & 4) ? side : 0.0};
		const double u = p[0] * e1[0] + p[1] * e1[1] + p[2] * e1[2], v = p[0] * e2[0] + p[1] * e2[1] + p[2] * e2[2];
		umin = fmin(umin, u); umax = fmax(umax, u); vmin = fmin(vmin, v); vmax = fmax(vmax, v);
	}
	umin -= pad; vmin -= pad; umax += pad; vmax += pad;
	double cell = 8.0;
	while ((umax - umin) / cell >= kHorizonMaxCells || (vmax - vmin) / cell >= kHorizonMaxCells) cell *= 2.0;
	for (int i = 0; i < 3; i++) { h.n[i] = (float)n[i]; h.e1[i] = (float)e1[i]; h.e2[i] = (float)e2[i]; }
	h.u0 = (float)umin; h.v0 = (float)vmin; h.invCell = (float)(1.0 / cell);  // (a power of two)
	h.nu = (uint32_t)((umax - umin) / cell) + 1u;
	h.nv = (uint32_t)((vmax - vmin) / cell) + 1u;
	h.axis = (int)permAxis0;  // rank_axes' longest axis of the light (ties broken as the shadow rays' walk space breaks them)
	return true;
}

// One occupied cluster (cx, cy, cz: cluster coordinates relative to the table origin, 8 voxels each) -> max into every cell its
// widened projection touches.  `update(cellIndex, value)` is atomicMax on the device, a plain max on the host.
template <class F>
VRM_HD void horizon_splat(const HorizonView& h, uint32_t cx, uint32_t cy, uint32_t cz, F update)
{
	const double p[3] = {8.0 * cx + 4.0, 8.0 * cy + 4.0, 8.0 * cz + 4.0};
	const double u = p[0] * h.e1[0] + p[1] * h.e1[1] + p[2] * h.e1[2] - h.u0;
	const double v = p[0] * h.e2[0] + p[1] * h.e2[1] + p[2] * h.e2[2] - h.v0;
	const double depth = p[0] * h.n[0] + p[1] * h.n[1] + p[2] * h.n[2];
	const double rr = (double)kHorizonClusterR + (double)kHorizonR + 1.0;  // + 1: fp32 projection at lookup
	const int32_t val = (int32_t)ceil(depth + (double)kHorizonClusterR + 1.0);
	const double ic = h.invCell;
	int iu0 = (int)floor((u - rr) * ic), iu1 = (int)floor((u + rr) * ic), iv0 = (int)floor((v - rr) * ic), iv1 = (int)floor((v + rr) * ic);
	iu0 = iu0 < 0 ? 0 : iu0; iv0 = iv0 < 0 ? 0 : iv0;
	iu1 = iu1 >= (int)h.nu ? (int)h.nu - 1 : iu1; iv1 = iv1 >= (int)h.nv ? (int)h.nv - 1 : iv1;
	for (int iv = iv0; iv <= iv1; iv++)
		for (int iu = iu0; iu <= iu1; iu++) update((uint32_t)iv * h.nu + (uint32_t)iu, val);
}

struct HashRegionDesc  // 16 bytes, one LDG.128 per region entry
{
	uint32_t slotBase;  // first 64-bit slot of table 1; table 2 follows at slotBase + n
	uint32_t n;         // slots per table
	uint32_t seed1, seed2;
};

struct SceneView
{
	const int32_t* regionTable;  // D^3 entries: dense region index or -1 (index = ux + uy*D + uz*D*D, VoxelSceneCPU.cuh:61-62)
	uint32_t diameter;
	int32_t minCoord;
	// cuckoo hash table ("two-level": region directory -> per-region pair of tables)
	const HashRegionDesc* hashDesc;
	const unsigned long long* slots;  // (hash_key << 32) | rgb ; kEmptySlot when free
	// voxel cluster store
	const uint2* headers;         // [region][512 clusters][16 words] {occupancy mask, index of the word's first colour}
	const uint32_t* clusterMask;  // [region][16] : bit c set <=> cluster c holds at least one voxel
	const uint32_t* values;       // colours, sorted by (region, cluster, in-cluster code)
};

struct Stats
{
	unsigned long long nExist, nExistFalse, nLookup, nLookupHit, nProbe2, nRegionReads;
	unsigned long long nCrawlSkipped;  // cluster-skip iterations replaced by crawl_skip (already included in nExist / nExistFalse)
};

// ---------------------------------------------------------------- axis permutation ("walk space")

// Walk slot i holds world axis axis(i).  cs(i) = shift of that axis inside a 9-bit cluster / in-cluster code
// (x:6, y:3, z:0 -- VoxelClusterStore.cuh:21-24); ks(i) = its shift inside the hash key (x:14, y:7, z:0 -- hash_key below).
struct PermIdentity
{
	VRM_HD int axis(int i) const { return i; }
	VRM_HD int cs(int i) const { return 6 - 3 * i; }
	VRM_HD int ks(int i) const { return 14 - 7 * i; }
	VRM_HD uint32_t stride(int i, uint32_t D) const { return i == 0 ? 1u : (i == 1 ? D : D * D); }
};

struct PermRuntime
{
	int a0, a1, a2;
	VRM_HD int axis(int i) const { return i == 0 ? a0 : (i == 1 ? a1 : a2); }
	VRM_HD int cs(int i) const { return 6 - 3 * axis(i); }
	VRM_HD int ks(int i) const { return 14 - 7 * axis(i); }
	VRM_HD uint32_t stride(int i, uint32_t D) const
	{
		int a = axis(i);
		return a == 0 ? 1u : (a == 1 ? D : D * D);
	}
};
template <class P> constexpr bool kIsIdentityPerm = false;
template <> constexpr bool kIsIdentityPerm<PermIdentity> = true;

// Ray::convertRayToLongestAxisDirection, renderer/rays/Ray.cuh:19-71 (strict '>' tie rules): slot 0 = longest,
// slot 1 = "shortAxis1" (middle), slot 2 = "shortAxis2" (shortest).
VRM_HD PermRuntime rank_axes(float dx, float dy, float dz)
{
	float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
	PermRuntime p;
	if (ax > ay && ax > az) { p.a0 = 0; if (ay > az) { p.a1 = 1; p.a2 = 2; } else { p.a1 = 2; p.a2 = 1; } }
	else if (ay > az)       { p.a0 = 1; if (ax > az) { p.a1 = 0; p.a2 = 2; } else { p.a1 = 2; p.a2 = 0; } }
	else                    { p.a0 = 2; if (ax > ay) { p.a1 = 0; p.a2 = 1; } else { p.a1 = 1; p.a2 = 0; } }
	return p;
}

template <class T> VRM_HD T pick3(int a, T v0, T v1, T v2) { return a == 0 ? v0 : (a == 1 ? v1 : v2); }

// world (x,y,z) -> walk slots
template <class P, class T> VRM_HD void to_walk(const P& p, const T* xyz, T* w)
{
	w[0] = pick3(p.axis(0), xyz[0], xyz[1], xyz[2]);
	w[1] = pick3(p.axis(1), xyz[0], xyz[1], xyz[2]);
	w[2] = pick3(p.axis(2), xyz[0], xyz[1], xyz[2]);
}
// walk slots -> world (x,y,z)
template <class P, class T> VRM_HD void to_world(const P& p, const T* w, T* xyz)
{
	int a0 = p.axis(0), a1 = p.axis(1);
	xyz[0] = a0 == 0 ? w[0] : (a1 == 0 ? w[1] : w[2]);
	xyz[1] = a0 == 1 ? w[0] : (a1 == 1 ? w[1] : w[2]);
	xyz[2] = a0 == 2 ? w[0] : (a1 == 2 ? w[1] : w[2]);
}

// ---------------------------------------------------------------- storage access

// Slot index inside one table: multiply-shift hashing with a per-region random ODD multiplier (the "seed"; universal for
// the high bits of key * seed mod 2^32) followed by a multiply-high range reduction -- two integer instructions per table
// instead of the reference's two signed mixing functions and four integer modulos per probe
// (CuckooHashTable.cuh:62,69,181-202).  The builder re-draws the multipliers of a region whose insertion cycles.
VRM_HD uint32_t hash_slot1(uint32_t key, uint32_t seed, uint32_t n) { return mulhi32((key + 1u) * seed, n); }
VRM_HD uint32_t hash_slot2(uint32_t key, uint32_t seed, uint32_t n) { return mulhi32((key + 1u) * seed, n); }

// "A coordinate of 64".  A ray that leaves a region through a low face at -tiny is rebased to 64 - tiny, which rounds to exactly
// 64.0f for tiny < 2^-19: the longest-axis walk then tests up to two voxels with a coordinate of 64 before its grid values are
// back inside the region (the original algorithm never does: it tests isRayInRegion first).  In the reference such a lookup is
// always empty for y or z = 64 -- its cluster id aliases into a neighbouring cluster, which only doesVoxelSpaceExist sees, and its
// key matches nothing (x = 64 indexes past its 512-entry cluster table: undefined there).  Here:
//  * hash table: the key has a spare bit per coordinate (hash_key below), so 64 matches nothing -- no extra instruction;
//  * VCS: the longest-axis test sites (vrm_flat.cuh voxel_test, lookup_voxel below with a run-time permutation) reject the
//    coordinate AFTER the value load behind the occupancy bit -- only a lookup that found something executes it, the walk through
//    empty space pays nothing (measured: 1.504 ms before and after).  VRM_COORD64_EMPTY=0 removes it.
#ifndef VRM_COORD64_EMPTY
#define VRM_COORD64_EMPTY 1
#endif
#ifndef VRM_HASH_INCR_KEY
#define VRM_HASH_INCR_KEY 1  // nested longest-axis walk over the hash table: the lookup key is kept up to date by the test loop (march_longest_axis)
#endif
#ifndef VRM_HASH_CLUSTER_FILTER
#define VRM_HASH_CLUSTER_FILTER 1
#endif
template <class T> VRM_HD T ldg(const T* p);
// The hash key of a region-local voxel: x << 14 | y << 7 | z -- SEVEN bits per coordinate although a stored voxel needs six.  The
// traversal can ask for a coordinate of exactly 64 (a ray rebased onto the far face of a region); the reference's key for it
// (VoxelFunctions.cuh:41-46: x << 20 | y << 10 | z) matches no stored voxel, and with the spare bit neither does this one --
// a 6-bit field would carry into its neighbour and could match a voxel of the next row.  Costs nothing: same instructions.
constexpr int kHashKeyBits = 7;
VRM_HD uint32_t hash_key(uint32_t x, uint32_t y, uint32_t z) { return (x << (2 * kHashKeyBits)) | (y << kHashKeyBits) | z; }
// key -> cluster id (x/8) << 6 | (y/8) << 3 | z/8 -> bit of the region's mask (a coordinate of 64 lands in row 0 of its axis:
// whatever the filter answers there, the key comparison still fails)
VRM_HD bool hash_cluster_occupied(const uint32_t* clusterMask, uint32_t ri, uint32_t key)
{
	const uint32_t t = key >> 3;
	const uint32_t cid = (t & 7u) | ((t >> 4) & 0x38u) | ((t >> 8) & 0x1C0u);
	return ((ldg(clusterMask + (ri * 16u + (cid >> 5))) >> (cid & 31u)) & 1u) != 0u;
}

// ---- reading the stored voxels back (vrm_voxels_out.cu): the inverses of the two layouts ----
// hash_key inverse: region-local x, y, z of a stored key
VRM_HD void hash_key_decode(uint32_t key, uint32_t& x, uint32_t& y, uint32_t& z)
{
	constexpr uint32_t m = (1u << kHashKeyBits) - 1u;
	x = key >> (2 * kHashKeyBits); y = (key >> kHashKeyBits) & m; z = key & m;
}
// A hash slot holds (hash_key << 32) | colour, or kEmptySlot.  A region's slots are table 1 and table 2 back to back:
// [base1, base1 + 2n) of SceneView::slots (load_region below), and after the build every one is a stored voxel of the region or free.
VRM_HD bool slot_used(unsigned long long e) { return e != kEmptySlot; }
VRM_HD uint32_t slot_key(unsigned long long e) { return (uint32_t)(e >> 32); }
VRM_HD uint32_t slot_colour(unsigned long long e) { return (uint32_t)e; }
// VCS: cluster (cx, cy, cz) of a region (cluster coordinates 0..7) -> cluster id, bit of the region's 512-bit cluster mask
VRM_HD uint32_t vcs_cluster_id(uint32_t cx, uint32_t cy, uint32_t cz) { return (cx << 6) | (cy << 3) | cz; }
// header word w (0..15) of cluster cid of dense region ri
VRM_HD size_t vcs_header_index(uint32_t ri, uint32_t cid, uint32_t w) { return ((size_t)ri * 512 + cid) * 16 + w; }
// Header word w covers the in-cluster codes 32w .. 32w + 31 (code = x%8 << 6 | y%8 << 3 | z%8): x%8 = w >> 1, y%8 = (w & 1) * 4 + bit / 8,
// z%8 = bit % 8 -- a z-range is a byte mask, a y-range selects bytes, an x-range selects word pairs.  Mask of the bits of word w whose
// voxel lies in the cluster-local box [x0, x1) x [y0, y1) x [z0, z1) (0 <= lo < hi <= 8 per axis).
VRM_HD uint32_t vcs_word_box_mask(uint32_t w, uint32_t x0, uint32_t x1, uint32_t y0, uint32_t y1, uint32_t z0, uint32_t z1)
{
	const uint32_t x = w >> 1, yb = (w & 1u) * 4u;
	if (x < x0 || x >= x1) return 0u;
	const uint32_t zb = (0xFFu << z0) & ~(0xFFu << z1) & 0xFFu;
	// bytes b = 0..3 hold y = yb + b: keep those with y0 <= y < y1
	const uint32_t bLo = y0 > yb ? y0 - yb : 0u, bHi = y1 > yb ? (y1 - yb < 4u ? y1 - yb : 4u) : 0u;
	if (bLo >= bHi) return 0u;
	const uint32_t bytes = (0xFFFFFFFFu >> (32u - 8u * (bHi - bLo))) << (8u * bLo);
	return (zb * 0x01010101u) & bytes;
}
// in-cluster coordinates of bit `bit` of header word w
VRM_HD void vcs_word_bit_xyz(uint32_t w, uint32_t bit, uint32_t& x, uint32_t& y, uint32_t& z)
{
	x = w >> 1; y = (w & 1u) * 4u + (bit >> 3); z = bit & 7u;
}
// index into SceneView::values of the colour behind a SET bit of a header word {occupancy mask, index of the word's first colour}
VRM_HD uint32_t vcs_colour_index(uint32_t hx, uint32_t hy, uint32_t bit) { return (hy & ~kHeaderClusterExists) + popc32(hx & ((1u << bit) - 1u)); }

template <int ST> struct RegionRef;

template <> struct RegionRef<kStorageHash>
{
	uint32_t base1, base2;  // first slot of table 1 / table 2 (32-bit indices into SceneView::slots: one IMAD.WIDE per probe)
	uint32_t n, seed1, seed2;
	uint32_t ri;            // dense region index (cluster-mask filter)
};

template <> struct RegionRef<kStorageVcs>
{
	uint32_t ri;  // dense region index: header / cluster-mask addresses are formed from it at each use (one register, not two pointers)
};

template <int ST> VRM_HD RegionRef<ST> load_region(const SceneView& sv, int32_t ri);

template <> VRM_HD RegionRef<kStorageHash> load_region<kStorageHash>(const SceneView& sv, int32_t ri)
{
#if defined(__CUDA_ARCH__)
	uint4 raw = __ldg(reinterpret_cast<const uint4*>(sv.hashDesc) + ri);
	HashRegionDesc d = {raw.x, raw.y, raw.z, raw.w};
#else
	HashRegionDesc d = sv.hashDesc[ri];
#endif
	RegionRef<kStorageHash> r;
	r.base1 = d.slotBase;
	r.base2 = d.slotBase + d.n;
	r.n = d.n; r.seed1 = d.seed1; r.seed2 = d.seed2;
	r.ri = (uint32_t)ri;
	return r;
}

template <> VRM_HD RegionRef<kStorageVcs> load_region<kStorageVcs>(const SceneView& sv, int32_t ri)
{
	RegionRef<kStorageVcs> r;
	r.ri = (uint32_t)ri;
	return r;
}

template <class T> VRM_HD T ldg(const T* p)
{
#if defined(__CUDA_ARCH__)
	return __ldg(p);
#else
	return *p;
#endif
}

// ---------------------------------------------------------------- per-ray context

template <int ST, bool STATS> struct RayCtx
{
	SceneView sv;
	Lighting light;
	LightWalk lw;  // only the state machine of vrm_flat.cuh reads it
	float translation[3];
	// First voxel found by this pixel's rays (global x,y,z, flag) -- SURVEY.md F6.  Every lookup site of the reference returns
	// on the first stored voxel and the shadow ray only starts after the primary hit, so "the first non-empty lookup" IS the
	// primary ray's hit.  Nested traversal (vrm_core.cuh): recorded by lookup_voxel in hit[].  State machine (vrm_flat.cuh):
	// recorded at the hit site (record_hit_voxel) straight through hitOut (nullable; the kernels point it at the pixel's slot
	// of the hit map, so no registers stay live for it; the host harness points it at hit[]).
	int32_t* hitOut;
	int32_t hit[4];
	// Queue of rays handed to the resume kernel (vrm_flat.cuh kPpDefer, vrm_render.cu resume_kernel); null = none
	void* deferQueue;
	// 1: a hit whose shaded colour is already black starts no shadow ray (Renderer.cuh:314-315: 0 * !isInShadow = 0 whatever the shadow
	// ray finds).  0 (host harness, reference-comparable event counters): every hit's shadow ray is traced, as the reference does.
	uint32_t skipDead;
	// Shadow horizon map (null cells: none).  Set only by the kernels that run the state machine of vrm_flat.cuh, and never for
	// reference-comparable event counters (it ends lit shadow rays before the reference's walk does).
	HorizonView hv;
#if VRM_SMEM_MASK
	// A/B form (north-star "shared-memory staging of cluster headers", DESIGN.md 3.2): the warp's copy of ONE region's 512-bit
	// cluster-exists mask in shared memory and the region it belongs to (warp-uniform; -1 = none).  Filled by march_scene_flat_warp.
	uint32_t* smMask;
	int32_t smRi;
#endif
	Stats st;

	VRM_HD void reset()
	{
#if VRM_SMEM_MASK
		smMask = nullptr; smRi = -1;
#endif
		hit[0] = hit[1] = hit[2] = hit[3] = 0;
		deferQueue = nullptr;
		skipDead = 0u;
		hv.cells = nullptr;
		if (STATS) { st.nExist = st.nExistFalse = st.nLookup = st.nLookupHit = st.nProbe2 = st.nRegionReads = st.nCrawlSkipped = 0; }
	}
};

// StorageStructure::doesVoxelSpaceExist (storage/StorageStructure.cuh:36-39,49-52; VoxelClusterStore.cuh:93-99)
template <int ST, bool STATS, class P>
VRM_HD bool space_exists(RayCtx<ST, STATS>& c, const RegionRef<ST>& r, const P& p, int g0, int g1, int g2)
{
	bool e = true;
	if constexpr (ST == kStorageVcs)
	{
		const RegionRef<kStorageVcs>& rv = r;
		uint32_t cid = ((uint32_t)(g0 >> 3) << p.cs(0)) | ((uint32_t)(g1 >> 3) << p.cs(1)) | ((uint32_t)(g2 >> 3) << p.cs(2));
		e = (ldg(c.sv.clusterMask + ((size_t)rv.ri * 16 + (cid >> 5))) >> (cid & 31)) & 1u;
	}
	if (STATS) { c.st.nExist++; if (!e) c.st.nExistFalse++; }
	return e;
}

// StorageStructure::lookupVoxel (CuckooHashTable.cuh:59-76; VoxelClusterStore.cuh:101-135): colour or kEmpty.
// g0..g2 are region-local coordinates in walk order; reg[] the region in walk order (for the hit record).
// The nested traversal records the pixel's first stored voxel here, in c.hit (SURVEY.md F6); the state machine of
// vrm_flat.cuh has its own fused test site and records at the hit site instead.
// The cuckoo lookup on a ready-made key (lookup_voxel below; the nested longest-axis walk keeps the key up to date itself).
template <bool STATS>
VRM_HD uint32_t lookup_hash_key(RayCtx<kStorageHash, STATS>& c, const RegionRef<kStorageHash>& rh, uint32_t key)
{
	uint32_t v = kEmpty;
#if VRM_HASH_CLUSTER_FILTER
	// negative filter: a voxel whose 8^3 cluster holds no voxel at all cannot be in the table, and the 64-byte mask of the
	// region answers that from L1 -- most lookups of a walk through open space never touch the (much larger) slot arrays.
	// The traversal is untouched (the hash table's doesVoxelSpaceExist stays true: no cluster is ever skipped).
	if (hash_cluster_occupied(c.sv.clusterMask, rh.ri, key))
#endif
	{
		// both probes are issued before either compare: a miss (the common case) costs one round trip, not two
		unsigned long long e1 = ldg(c.sv.slots + (rh.base1 + hash_slot1(key, rh.seed1, rh.n)));
		unsigned long long e2 = ldg(c.sv.slots + (rh.base2 + hash_slot2(key, rh.seed2, rh.n)));
		if ((uint32_t)(e1 >> 32) == key) v = (uint32_t)e1;
		else if ((uint32_t)(e2 >> 32) == key) v = (uint32_t)e2;
	}
	if (STATS) c.st.nProbe2++;
	return v;
}

// A lookup found a stored voxel: the pixel's first one is its hit (see RayCtx::hit)
template <int ST, bool STATS, class P>
VRM_HD void note_lookup_hit(RayCtx<ST, STATS>& c, const P& p, const int* reg, int g0, int g1, int g2)
{
	if (STATS) c.st.nLookupHit++;
	if (!c.hit[3])
	{
		int gw[3] = {reg[0] * kRegion + g0, reg[1] * kRegion + g1, reg[2] * kRegion + g2};
		int gx[3];
		to_world(p, gw, gx);
		c.hit[0] = gx[0]; c.hit[1] = gx[1]; c.hit[2] = gx[2]; c.hit[3] = 1;
	}
}

template <int ST, bool STATS, class P>
VRM_HD uint32_t lookup_voxel(RayCtx<ST, STATS>& c, const RegionRef<ST>& r, const P& p, const int* reg, int g0, int g1, int g2)
{
	uint32_t v = kEmpty;
	if constexpr (ST == kStorageHash)
	{
		const uint32_t key = ((uint32_t)g0 << p.ks(0)) | ((uint32_t)g1 << p.ks(1)) | ((uint32_t)g2 << p.ks(2));
		v = lookup_hash_key(c, r, key);
	}
	else
	{
		const RegionRef<kStorageVcs>& rv = r;
		uint32_t cid = ((uint32_t)(g0 >> 3) << p.cs(0)) | ((uint32_t)(g1 >> 3) << p.cs(1)) | ((uint32_t)(g2 >> 3) << p.cs(2));
		uint32_t code = ((uint32_t)(g0 & 7) << p.cs(0)) | ((uint32_t)(g1 & 7) << p.cs(1)) | ((uint32_t)(g2 & 7) << p.cs(2));
		uint2 h = ldg(c.sv.headers + (((size_t)rv.ri * 512 + cid) * 16 + (code >> 5)));
		uint32_t bit = code & 31;
		if ((h.x >> bit) & 1u)
		{
			v = ldg(c.sv.values + (h.y & ~kHeaderClusterExists) + popc32(h.x & ((1u << bit) - 1u)));
			// "a coordinate of 64" (above): only the longest-axis walk (the one with a run-time permutation) can ask for it; applied
			// after the load behind the occupancy bit, like the state machine's test site (vrm_flat.cuh voxel_test)
			if constexpr (VRM_COORD64_EMPTY && !kIsIdentityPerm<P>) { if (((uint32_t)g0 | (uint32_t)g1 | (uint32_t)g2) & 64u) v = kEmpty; }
		}
	}
	if (STATS) c.st.nLookup++;
	if (v != kEmpty) note_lookup_hit(c, p, reg, g0, g1, g2);
	return v;
}

// The hit map entry of a primary hit: region (walk order) * 64 + region-local voxel (walk order), stored in WORLD axes.
template <int ST, bool STATS, class P>
VRM_HD void record_hit_voxel(RayCtx<ST, STATS>& c, const P& p, const int* reg, int g0, int g1, int g2)
{
	if (!c.hitOut) return;
	int gw[3] = {reg[0] * kRegion + g0, reg[1] * kRegion + g1, reg[2] * kRegion + g2};
	int gx[3];
	to_world(p, gw, gx);
	c.hitOut[0] = gx[0]; c.hitOut[1] = gx[1]; c.hitOut[2] = gx[2]; c.hitOut[3] = 1;
}

// VoxelScene::isRayInScene + getRegionStorageStructure (renderer/Renderer.cuh:29-44): -2 = outside the table,
// -1 = empty region, else dense region index.
template <int ST, bool STATS, class P>
VRM_HD int32_t region_entry(RayCtx<ST, STATS>& c, const P& p, const int* reg)
{
	uint32_t D = c.sv.diameter;
	uint32_t u0 = (uint32_t)(reg[0] - c.sv.minCoord), u1 = (uint32_t)(reg[1] - c.sv.minCoord), u2 = (uint32_t)(reg[2] - c.sv.minCoord);
	if (!(u0 < D && u1 < D && u2 < D)) return -2;
	if (STATS) c.st.nRegionReads++;
	return ldg(c.sv.regionTable + (u0 * p.stride(0, D) + u1 * p.stride(1, D) + u2 * p.stride(2, D)));
}

// ---------------------------------------------------------------- lighting (renderer/Renderer.cuh:57-86,237-258)

VRM_HD uint32_t vec_to_rgb(float r, float g, float b)  // VoxelFunctions.cuh:76-82
{
	uint32_t ir = (uint32_t)vmul(r, 255.0f), ig = (uint32_t)vmul(g, 255.0f), ib = (uint32_t)vmul(b, 255.0f);
	return (ir << 16) | (ig << 8) | ib;
}

// normalAxis / normalSign are in WORLD axes; hitLocal = hit position in region-local WORLD axes; regW = region (world axes)
VRM_HD uint32_t apply_lighting(const Lighting& L, const float* translation, uint32_t voxelColor, int normalAxis, float normalSign,
                               const float* hitLocal, const int* regW)
{
	float cr = vdiv((float)(voxelColor >> 16), 255.0f);           // VoxelFunctions.cuh:54-74
	float cg = vdiv((float)((voxelColor >> 8) & 0xFF), 255.0f);
	float cb = vdiv((float)(voxelColor & 0xFF), 255.0f);
	float n[3] = {0.0f, 0.0f, 0.0f};
	n[0] = normalAxis == 0 ? normalSign : 0.0f;
	n[1] = normalAxis == 1 ? normalSign : 0.0f;
	n[2] = normalAxis == 2 ? normalSign : 0.0f;
	if (L.usePoint)  // Renderer.cuh:68-86
	{
		float t[3];
		for (int i = 0; i < 3; i++)
		{
			float regionWorld = vadd(translation[i], (float)(regW[i] * kRegion));  // Renderer.cuh:413
			float hit = vadd(regionWorld, hitLocal[i]);                              // Renderer.cuh:88-91
			t[i] = vsub(L.pos[i], hit);
		}
		float distance = vsqrt(vadd(vadd(vmul(t[0], t[0]), vmul(t[1], t[1])), vmul(t[2], t[2])));
		float ld[3] = {vdiv(t[0], distance), vdiv(t[1], distance), vdiv(t[2], distance)};
		float attenuation = vdiv(1.0f, vadd(vadd(1.0f, vmul(0.045f, distance)), vmul(0.0075f, vmul(distance, distance))));
		float diff = fmaxf(vadd(vadd(vmul(n[0], ld[0]), vmul(n[1], ld[1])), vmul(n[2], ld[2])), 0.0f);
		float r = vmul(vmul(attenuation, vmul(diff, L.color[0])), cr);
		float g = vmul(vmul(attenuation, vmul(diff, L.color[1])), cg);
		float b = vmul(vmul(attenuation, vmul(diff, L.color[2])), cb);
		return vec_to_rgb(r, g, b);
	}
	// Renderer.cuh:57-66
	float diff = fmaxf(vadd(vadd(vmul(n[0], L.dir[0]), vmul(n[1], L.dir[1])), vmul(n[2], L.dir[2])), 0.0f);
	return vec_to_rgb(vmul(cr, vmul(diff, L.color[0])), vmul(cg, vmul(diff, L.color[1])), vmul(cb, vmul(diff, L.color[2])));
}

// getNormalFromTValues (Renderer.cuh:237-247) evaluated in walk space: the reference tests X, then Y, else Z,
// so pick the lowest WORLD axis whose t equals tMin, falling back to Z.
template <class P> VRM_HD int normal_axis_from_t(const P& p, float t0, float t1, float t2, float tMin)
{
	int m = 0;
	if (t0 == tMin) m |= 1 << p.axis(0);
	if (t1 == tMin) m |= 1 << p.axis(1);
	if (t2 == tMin) m |= 1 << p.axis(2);
	return (m & 1) ? 0 : ((m & 2) ? 1 : 2);
}

// ---------------------------------------------------------------- shared walk helpers

VRM_HD uint32_t float_bits(float f)
{
#if defined(__CUDA_ARCH__)
	return __float_as_uint(f);
#else
	uint32_t u;
	memcpy(&u, &f, 4);
	return u;
#endif
}
// isRayInRegion, Renderer.cuh:93-98: 0 <= o_i < 64 on all axes.  Non-negative floats order like their bit patterns and
// every negative float, NaN and +-inf has a pattern >= bits(64.0f), so three float range tests (seven instructions) are one
// unsigned max and one compare.  The only value the two forms disagree on is -0.0f (in range for the reference), which a
// position can never take: canonical_zero() removes it where a ray starts and sums / differences cannot produce it.
VRM_HD bool ray_in_region(const float* o)
{
	uint32_t a = float_bits(o[0]), b = float_bits(o[1]), c = float_bits(o[2]);
	uint32_t m = a > b ? a : b;
	m = m > c ? m : c;
	return m < 0x42800000u;
}
// -0.0f -> +0.0f, every other value unchanged.  Invisible to the reference's arithmetic (a zero's sign is never observed:
// no division by a position, no copysign of one), see ray_in_region.
VRM_HD float canonical_zero(float v) { return vadd(v, 0.0f); }
VRM_HD bool grid_in_region(int x, int y, int z)  // Renderer.cuh:436-439
{
	return (uint32_t)x < (uint32_t)kRegion && (uint32_t)y < (uint32_t)kRegion && (uint32_t)z < (uint32_t)kRegion;
}
VRM_HD float next_edge(float d, float v)  // Renderer.cuh:47-55,263-265
{
	return d > 0.0f ? vadd(ceilf(v), kEps) : vsub(floorf(v), kEps);
}
template <bool GUARD> VRM_HD float t_to(float next, float o, float d)  // Renderer.cuh:113-115 (guarded) / 273-275
{
	float t = vdiv(vsub(next, o), d);
	if (GUARD) t = (d != 0.0f) ? t : INFINITY;
	return t;
}
// the three t values of one advance: (next_i - o_i) / d_i with the ray's exact-division constants
template <bool GUARD> VRM_HD void t_to3(const RayDir& k, float n0, float n1, float n2, const float* o, float& a0, float& a1, float& a2)
{
	div3(vsub(n0, o[0]), vsub(n1, o[1]), vsub(n2, o[2]), k, a0, a1, a2);
	if (GUARD)
	{
		a0 = (k.d[0] != 0.0f) ? a0 : INFINITY; a1 = (k.d[1] != 0.0f) ? a1 : INFINITY; a2 = (k.d[2] != 0.0f) ? a2 : INFINITY;
	}
}
VRM_HD int cluster_edge(float d, int v)  // Renderer.cuh:293-295
{
	return d > 0.0f ? ((v / 8) + 1) * 8 : (v / 8) * 8;
}

// cluster_edge for a voxel coordinate known to be non-negative (every call site inside a region: v in [0, 64)): the
// truncating division is then a mask.  Same value as cluster_edge.
VRM_HD int cluster_edge_u(float d, int v)
{
	return (int)(((uint32_t)v & ~7u) + (d > 0.0f ? 8u : 0u));
}

VRM_HD float bits_float(uint32_t u)
{
#if defined(__CUDA_ARCH__)
	return __uint_as_float(u);
#else
	float f;
	memcpy(&f, &u, 4);
	return f;
#endif
}

// next_edge for a direction component that is NOT ZERO (every component of a ray whose fast-division threshold is finite): the sign
// bit of d decides, and ceilf(v) + EPSILON = -(floorf(-v) - EPSILON) exactly (negation is exact, round-to-nearest is symmetric), so
// the two roundings + two sums + select of next_edge become one conditional sign flip, one rounding, one sum and the flip back.
VRM_HD float next_edge_nz(float d, float v)
{
	const uint32_t flip = ~float_bits(d) & 0x80000000u;
	return bits_float(float_bits(vsub(floorf(bits_float(float_bits(v) ^ flip)), kEps)) ^ flip);
}

// ---- "crawl" fast-forward ---------------------------------------------------------------------------------------------
// A reference pathology that dominates whole frames: a cluster skip towards a NEGATIVE direction component d_j with
// |d_j| < ~5e-3 lands the ray EXACTLY on the cluster face (o_j + EPSILON * d_j rounds back to the face), the voxel (int)o_j
// still belongs to the same empty cluster, and from then on every skip iteration has t_j = 0, so the ray advances by only
// EPSILON * d per iteration: ~10^5 iterations to crawl across one 8-voxel cluster (Renderer.cuh:293-304 / 707-721).  Any
// view whose frustum contains a direction with a zero component has a few pixel columns of such rays (measured: 470 ms
// instead of 2.8 ms for a 4K terrain frame; 196 ms per 1080p frame on the 2048^3 orbit), and the reference's own kernels
// crawl the same way.
// While the ray stays inside the cluster cell, each iteration is exactly  o_i <- RN(o_i + c_i),  c_i = RN(EPSILON * d_i).
// Inside one binade a float advances by a constant whole number q_i of ulps per such addition (q_i = nearest integer to
// c_i / ulp; on an exact tie the even one of the two neighbours, once the mantissa is even), i.e. its bit pattern advances by q_i.  So M iterations are one integer multiply-add
// per axis: the result is bit-identical to executing them.  M is chosen so that all M skipped positions stay strictly
// inside the cell and the binade; the step that leaves the cell is then executed normally.
// Returns M (0 = nothing skipped).  v = voxel whose cluster is being skipped; the caller guarantees (int)o lies in that cell.
VRM_HD int crawl_skip(float* o, const float* dir, float thr, int v0, int v1, int v2)
{
	if (!(thr == thr)) return 0;  // only rays on the exact-division fast path (no zero / tiny direction components)
	const int v[3] = {v0, v1, v2};
	int q[3];
	int best = 0x7FFFFFFF;
	bool stuck = false;
#pragma unroll
	for (int i = 0; i < 3; i++)
	{
		const float y = o[i];
		const uint32_t yb = float_bits(y), eb = yb >> 23;
		if (eb < 24u || eb > 140u) return 0;  // zero, denormal, tiny, negative (sign bit), inf / NaN
		const float c = vmul(kEps, dir[i]);
		const float cu = vmul(c, bits_float((277u - eb) << 23));  // c / ulp(y), exact power-of-two scaling
		if (!(fabsf(cu) < 1048576.0f)) return 0;
		int qi;
		const float cuFloor = floorf(cu);
		if (vsub(cu, cuFloor) == 0.5f)
		{
			// exact tie: y + c lies midway between two floats and rounds to the one with the even mantissa.  From an even
			// mantissa that is the even one of {floor(cu), floor(cu) + 1} ulps, and the mantissa stays even, so the step is
			// constant from then on; from an odd mantissa one ordinary step makes it even (no skip this time)
			if (yb & 1u) return 0;
			const int k = (int)cuFloor;
			qi = (k & 1) ? k + 1 : k;
		}
		else qi = (int)rintf(cu);
		const int cell = v[i] & ~7;
		uint32_t lo = float_bits((float)cell), hi = float_bits((float)(cell + 8));
		const uint32_t blo = eb << 23, bhi = (eb + 1u) << 23;
		// A step DOWN must land strictly above the binade's first float: the exact sum of a step that "lands on" the power of two
		// can lie below it, where the floats are twice as dense, and then rounds to one of those instead (a differential run
		// against the oracle found 32.0 vs 31.9999981)
		if (lo < blo) lo = blo;
		if (hi > bhi) hi = bhi;
		if (yb < lo || yb >= hi) return 0;  // (int)o is not in the cell being skipped
		if (lo == blo) lo = blo + 1u;       // lowest pattern a step down may land on
		int m;
		if (qi > 0) m = (int)((hi - 1u - yb) / (uint32_t)qi);
		else if (qi < 0) m = yb >= lo ? (int)((yb - lo) / (uint32_t)(-qi)) : 0;
		else
		{
			// "does not move" must hold for the addition itself: from a power of two a negative c steps into the binade below, whose
			// floats are twice as dense, so |c| between a quarter and half an ulp of y DOES move it (found by a differential run
			// against the oracle: a ray starting on local coordinate 16.0)
			if (vadd(y, c) != y) return 0;
			m = 0x7FFFFFFF;
			if ((float)cluster_edge(dir[i], v[i]) == y) stuck = true;  // this axis sits on its cluster face and cannot move: t_i = 0
		}
		best = m < best ? m : best;
		q[i] = qi;
	}
	if (!stuck || best < 1 || best == 0x7FFFFFFF) return 0;
#pragma unroll
	for (int i = 0; i < 3; i++) o[i] = bits_float(float_bits(o[i]) + (uint32_t)(best * q[i]));
	return best;
}

VRM_HD int crawl_skip(float* o, const RayDir& k, int v0, int v1, int v2) { return crawl_skip(o, k.d, k.thr, v0, v1, v2); }

// Out-of-line form for the state machine: position and direction travel by value / through a small struct so that the
// caller's registers are not forced into local memory.
struct CrawlResult { float o0, o1, o2; int skipped; };
#if VRM_COLD_OUTLINE
VRM_HD_NOINLINE
#else
VRM_HD
#endif
CrawlResult crawl_skip_cold(float o0, float o1, float o2, float d0, float d1, float d2, float thr, int v0, int v1, int v2)
{
	float o[3] = {o0, o1, o2};
	const float d[3] = {d0, d1, d2};
	CrawlResult r;
	r.skipped = crawl_skip(o, d, thr, v0, v1, v2);
	r.o0 = o[0]; r.o1 = o[1]; r.o2 = o[2];
	return r;
}

// Renderer.cuh:421-429: move region coordinates by floor(o / 64) and rebase the local position
VRM_HD void rebase_region(float* o, int* reg)
{
	for (int i = 0; i < 3; i++)
	{
		int diff = (int)floorf(vmul(o[i], 0.015625f));  // o / 64: 1/64 is a power of two, so the product is the same correctly rounded value
		reg[i] += diff;
		o[i] = vmul(1.0f, vsub(o[i], (float)(diff * kRegion)));  // convertRayToLocalSpace(.., scale 1), Ray.cuh:14-17
	}
}

// A NaN position (only reachable when a direction component is exactly +0 in the unguarded divisions: -inf * 0) makes
// the reference's host build leave the scene -- (int)NaN is INT_MIN there -- whereas CUDA's saturating conversion gives 0
// and the reference's own kernels (and a literal translation) would spin forever.  Follow the host build: NaN = outside.
VRM_HD bool position_sane(const float* o) { return o[0] == o[0] && o[1] == o[1] && o[2] == o[2]; }

// Null-region skip, Renderer.cuh:384-410 (GUARD: 185-211).  On return ri >= 0 (a stored region) or -2 (left the scene).
template <int ST, bool STATS, class P, bool GUARD>
VRM_HD int32_t skip_null_regions(RayCtx<ST, STATS>& c, const P& p, float* o, const RayDir& k, int* reg, int32_t ri)
{
	const float* d = k.d;
	while (ri == -1)
	{
		float n0 = d[0] > 0.0f ? vadd((float)kRegion, kEps) : vsub(0.0f, kEps);
		float n1 = d[1] > 0.0f ? vadd((float)kRegion, kEps) : vsub(0.0f, kEps);
		float n2 = d[2] > 0.0f ? vadd((float)kRegion, kEps) : vsub(0.0f, kEps);
		float a0, a1, a2;
		t_to3<GUARD>(k, n0, n1, n2, o, a0, a1, a2);
		float tMin = min3(a0, a1, a2);
		o[0] = along(o[0], tMin, d[0]); o[1] = along(o[1], tMin, d[1]); o[2] = along(o[2], tMin, d[2]);
		rebase_region(o, reg);
		ri = position_sane(o) ? region_entry(c, p, reg) : -2;
	}
	// (The caller's tests of the returned entry are merged with this loop's into a three-way jump table in the hash-table kernels.  Hiding
	// the value behind an opaque copy removes the BRX -- and cost VCS + original 7 % on the sparse 2048^3 orbit, 98.9 -> 106.3 ms, for
	// nothing measurable on the hash table: left as the compiler wants it.)
	return ri;
}

// ---------------------------------------------------------------- "original" traversal

// The step loop shared by rayMarchVoxelGrid (Renderer.cuh:260-336, GUARD=false) and shadowRayMarchVoxelGrid
// (Renderer.cuh:100-172, GUARD=true).  Returns the raw voxel colour or kEmpty; t[0..3] = the OUTER tX,tY,tZ,tMin
// of the hit step (stale after a cluster skip, exactly as in the reference, SURVEY.md §7 hard part 3).
// NZ: the caller knows that no direction component is zero (k.thr is finite): next_edge_nz, and the zero-direction guards of the
// shadow routine (Renderer.cuh:113-115) are moot.
template <int ST, bool STATS, class P, bool GUARD_, bool NZ>
VRM_HD uint32_t march_steps_t(RayCtx<ST, STATS>& c, const RegionRef<ST>& r, const P& p, float* o, const RayDir& k, const int* reg, float* t)
{
	constexpr bool GUARD = GUARD_ && !NZ;
	const float* d = k.d;
	float t0, t1, t2;
	t_to3<GUARD>(k, NZ ? next_edge_nz(d[0], o[0]) : next_edge(d[0], o[0]), NZ ? next_edge_nz(d[1], o[1]) : next_edge(d[1], o[1]), NZ ? next_edge_nz(d[2], o[2]) : next_edge(d[2], o[2]), o, t0, t1, t2);
	float tMin = min3(t0, t1, t2);
	float s = vadd(tMin, kEps);
	o[0] = along(o[0], s, d[0]); o[1] = along(o[1], s, d[1]); o[2] = along(o[2], s, d[2]);
	while (ray_in_region(o))
	{
		int v0 = (int)o[0], v1 = (int)o[1], v2 = (int)o[2];
		if (!space_exists(c, r, p, v0, v1, v2))
		{
			float u0, u1, u2;
			t_to3<GUARD>(k, (float)cluster_edge(d[0], v0), (float)cluster_edge(d[1], v1), (float)cluster_edge(d[2], v2), o, u0, u1, u2);
			float mu = min3(u0, u1, u2);
			if (mu == 0.0f)
			{
				const int skipped = crawl_skip(o, k, v0, v1, v2);
				if (skipped > 0)
				{
					if (STATS) { c.st.nExist += skipped; c.st.nExistFalse += skipped; c.st.nCrawlSkipped += skipped; }
					t_to3<GUARD>(k, (float)cluster_edge(d[0], v0), (float)cluster_edge(d[1], v1), (float)cluster_edge(d[2], v2), o, u0, u1, u2);
					mu = min3(u0, u1, u2);
				}
			}
			float su = vadd(mu, kEps);
			o[0] = along(o[0], su, d[0]); o[1] = along(o[1], su, d[1]); o[2] = along(o[2], su, d[2]);
			continue;
		}
		uint32_t col = lookup_voxel(c, r, p, reg, v0, v1, v2);
		if (col != kEmpty)
		{
			t[0] = t0; t[1] = t1; t[2] = t2; t[3] = tMin;
			return col;
		}
		t_to3<GUARD>(k, NZ ? next_edge_nz(d[0], o[0]) : next_edge(d[0], o[0]), NZ ? next_edge_nz(d[1], o[1]) : next_edge(d[1], o[1]), NZ ? next_edge_nz(d[2], o[2]) : next_edge(d[2], o[2]), o, t0, t1, t2);
		tMin = min3(t0, t1, t2);
		s = vadd(tMin, kEps);
		o[0] = along(o[0], s, d[0]); o[1] = along(o[1], s, d[1]); o[2] = along(o[2], s, d[2]);
	}
	return kEmpty;
}

#ifndef VRM_STEPS_NZ
#define VRM_STEPS_NZ 1
#endif
template <int ST, bool STATS, class P, bool GUARD>
VRM_HD uint32_t march_steps(RayCtx<ST, STATS>& c, const RegionRef<ST>& r, const P& p, float* o, const RayDir& k, const int* reg, float* t)
{
#if VRM_STEPS_NZ
	if (k.thr == k.thr) return march_steps_t<ST, STATS, P, GUARD, true>(c, r, p, o, k, reg, t);  // per-ray constant: no direction component is zero
#endif
	return march_steps_t<ST, STATS, P, GUARD, false>(c, r, p, o, k, reg, t);
}

// What a primary march reports on a hit; lighting and the shadow ray are applied ONCE, in march_scene, instead of
// at each of the reference's eight hit sites (keeps the kernel small and the warp converged).
struct HitInfo
{
	float pos[3];   // hit position, region-local, walk space (the "rayOrigin" handed to applyLighting / the shadow ray)
	int nAxisW;     // normal axis in WORLD axes
	float nSign;    // +-1
	int laShadow;   // 1: isInShadowRayMarchVoxelSceneLongestAxis, 0: isInShadowOriginalRayMarch
};

// rayMarchVoxelGrid, Renderer.cuh:260-336 (the hit's lighting + shadow are applied by the caller)
template <int ST, bool STATS, class P>
VRM_HD uint32_t march_original(RayCtx<ST, STATS>& c, const RegionRef<ST>& r, const P& p, float* o, const RayDir& k, const int* reg, HitInfo& h)
{
	const float* d = k.d;
	float t[4];
	uint32_t col = march_steps<ST, STATS, P, false>(c, r, p, o, k, reg, t);
	if (col == kEmpty) return kEmpty;
	h.nAxisW = normal_axis_from_t(p, t[0], t[1], t[2], t[3]);  // Renderer.cuh:312
	float dn = p.axis(0) == h.nAxisW ? d[0] : (p.axis(1) == h.nAxisW ? d[1] : d[2]);
	h.nSign = copysignf(1.0f, -dn);
	h.pos[0] = o[0]; h.pos[1] = o[1]; h.pos[2] = o[2];        // Renderer.cuh:314-315
	h.laShadow = 0;
	return col;
}

// ---------------------------------------------------------------- "longest axis" traversal (walk slot 0 = L, 1 = M, 2 = S)

// Ray::convertRayToLongestAxisDirection's scaling (Ray.cuh:37,52,67,69): direction * (1 / |longest component|).  The
// reference recomputes it at every region entry from the same direction, so it is a per-ray constant.
VRM_HD RayDir scaled_raydir(const RayDir& k)
{
	float s = vdiv(1.0f, fabsf(k.d[0]));
	return make_raydir(vmul(s, k.d[0]), vmul(s, k.d[1]), vmul(s, k.d[2]));
}

struct LaState
{
	float oo[3], od[3];  // oldRay origin / longest-axis-scaled direction
	float ro[3];         // ray origin (its direction equals od)
	int g[3], ad[3];     // gridValues, axisDiff
};

// performVoxelSpaceJump (Renderer.cuh:696-751) / performShadowVoxelSpaceJump (Renderer.cuh:441-492)
template <int ST, bool STATS, bool SHADOW>
VRM_HD uint32_t voxel_space_jump(RayCtx<ST, STATS>& c, const RegionRef<ST>& r, const PermRuntime& p, LaState& s, const RayDir& ko, float* origO, const int* reg, HitInfo& h)
{
	float t0 = 0.0f, t1 = 0.0f, t2 = 0.0f, tMin = 0.0f;
	while (!space_exists(c, r, p, s.g[0], s.g[1], s.g[2]))
	{
		t_to3<false>(ko, (float)cluster_edge(s.od[0], s.g[0]), (float)cluster_edge(s.od[1], s.g[1]), (float)cluster_edge(s.od[2], s.g[2]), s.oo, t0, t1, t2);
		float mj = min3(t0, t1, t2);
		if (mj == 0.0f)
		{
			const int skipped = crawl_skip(s.oo, ko, s.g[0], s.g[1], s.g[2]);  // checks that oldRay's voxel is in gridValues' cluster cell
			if (skipped > 0)
			{
				if (STATS) { c.st.nExist += skipped; c.st.nExistFalse += skipped; c.st.nCrawlSkipped += skipped; }
				t_to3<false>(ko, (float)cluster_edge(s.od[0], s.g[0]), (float)cluster_edge(s.od[1], s.g[1]), (float)cluster_edge(s.od[2], s.g[2]), s.oo, t0, t1, t2);
				mj = min3(t0, t1, t2);
			}
		}
		tMin = vadd(mj, kEps);
		s.oo[0] = along(s.oo[0], tMin, s.od[0]); s.oo[1] = along(s.oo[1], tMin, s.od[1]); s.oo[2] = along(s.oo[2], tMin, s.od[2]);
		s.g[0] = (int)floorf(s.oo[0]); s.g[1] = (int)floorf(s.oo[1]); s.g[2] = (int)floorf(s.oo[2]);
		if (!grid_in_region(s.g[0], s.g[1], s.g[2]))
		{
			origO[0] = s.oo[0]; origO[1] = s.oo[1]; origO[2] = s.oo[2];
			return kEmpty;
		}
	}
	uint32_t col = lookup_voxel(c, r, p, reg, s.g[0], s.g[1], s.g[2]);
	if (col != kEmpty)
	{
		if (!SHADOW)
		{
			// tMin already carries +EPSILON (Renderer.cuh:716,736), so this normally falls through to the Z normal
			h.nAxisW = normal_axis_from_t(p, t0, t1, t2, tMin);
			float dn = p.axis(0) == h.nAxisW ? s.od[0] : (p.axis(1) == h.nAxisW ? s.od[1] : s.od[2]);
			h.nSign = copysignf(1.0f, -dn);
			h.pos[0] = s.oo[0]; h.pos[1] = s.oo[1]; h.pos[2] = s.oo[2];  // Renderer.cuh:737-738
			h.laShadow = 1;
		}
		return col;
	}
	// re-snap to the longest axis, Renderer.cuh:742-747
	float tNext = div1(vsub(s.od[0] > 0.0f ? ceilf(s.oo[0]) : floorf(s.oo[0]), s.oo[0]), ko, 0);
	float tt = vadd(tNext, kEps);
	s.ro[0] = along(s.oo[0], tt, s.od[0]); s.ro[1] = along(s.oo[1], tt, s.od[1]); s.ro[2] = along(s.oo[2], tt, s.od[2]);
	s.ad[1] = (int)s.ro[1] - s.g[1];
	s.ad[2] = (int)s.ro[2] - s.g[2];
	return kContinue;
}

// rayMarchVoxelGridLongestAxis (Renderer.cuh:760-915) / shadowRayMarchVoxelGridLongestAxis (Renderer.cuh:495-631).
// o/d/reg are in walk space of p (slot 0 = longest axis of d).
//
// The reference spells the per-iteration voxel tests out as four sub-cases with seven copies of the same
// "bump one axis, test the voxel space, look the voxel up" unit.  Here the sub-case only selects the ORDER of
// slots to test (packed 2 bits each into `seq`); one shared test site then runs 1-3 times.  Same tests in the same
// order, but lanes of a warp that are in different sub-cases execute the same instructions instead of serialising.
// a voxel test of the longest-axis walk found a voxel: where, and which face (Renderer.cuh:818-822, 899, 753-758)
VRM_HD void la_test_hit(const PermRuntime& p, const LaState& s, int slot, HitInfo& h)
{
	float odS = pick3(slot, s.od[0], s.od[1], s.od[2]);
	h.nAxisW = p.axis(slot);
	h.nSign = copysignf(1.0f, -odS);
	if (slot == 0) { h.pos[0] = s.ro[0]; h.pos[1] = s.ro[1]; h.pos[2] = s.ro[2]; }  // Renderer.cuh:899
	else
	{
		// getLocalHitLocation, Renderer.cuh:753-758
		float ooS = pick3(slot, s.oo[0], s.oo[1], s.oo[2]);
		float tl = odS > 0.0f ? vdiv(vsub(ceilf(ooS), ooS), odS) : vdiv(vsub(floorf(ooS), ooS), odS);
		h.pos[0] = along(s.oo[0], tl, s.od[0]); h.pos[1] = along(s.oo[1], tl, s.od[1]); h.pos[2] = along(s.oo[2], tl, s.od[2]);
	}
	h.laShadow = 1;
}

template <int ST, bool STATS, bool SHADOW>
VRM_HD uint32_t march_longest_axis(RayCtx<ST, STATS>& c, const RegionRef<ST>& r, const PermRuntime& p, float* o, const RayDir& k, const RayDir& ko, const int* reg, HitInfo& h)
{
	const float* d = k.d;
	LaState s;
	s.od[0] = ko.d[0]; s.od[1] = ko.d[1]; s.od[2] = ko.d[2];  // scaled direction: constant along the ray, see scaled_raydir
	s.oo[0] = o[0]; s.oo[1] = o[1]; s.oo[2] = o[2];
	s.g[0] = (int)o[0]; s.g[1] = (int)o[1]; s.g[2] = (int)o[2];
	s.ad[0] = d[0] < 0.0f ? -1 : 1;
	// snap the longest axis to the grid, Renderer.cuh:776-779
	float t = s.ad[0] > 0 ? vdiv(vsub(vadd(vadd((float)s.g[0], kEps), 1.0f), o[0]), 1.0f)
	                      : vdiv(vsub(vsub((float)s.g[0], kEps), o[0]), -1.0f);
	s.ro[0] = along(s.oo[0], t, s.od[0]); s.ro[1] = along(s.oo[1], t, s.od[1]); s.ro[2] = along(s.oo[2], t, s.od[2]);
	s.ad[1] = (int)s.ro[1] - s.g[1];
	s.ad[2] = (int)s.ro[2] - s.g[2];
	const bool roundDown = s.od[1] < 0.0f;  // Renderer.cuh:784
	// Hash table (VRM_HASH_INCR_KEY): every voxel of the walk is looked up (doesVoxelSpaceExist is always true, nothing is skipped),
	// so the test loop keeps the lookup KEY up to date -- one add of the tested slot's step, ad << ks -- instead of bumping three grid
	// values and packing them again for every test; the grid values are unpacked from the key once per iteration (and at a hit).
	// Fields are 7 bits wide and the grid values stay in [0, 64], so sums and ORs of the fields agree.
	constexpr bool kIncrKey = VRM_HASH_INCR_KEY && ST == kStorageHash;
	uint32_t key = 0u, kst1 = 0u, kst2 = 0u;
	const int ks0 = p.ks(0), ks1 = p.ks(1), ks2 = p.ks(2);
	const uint32_t kst0 = (uint32_t)s.ad[0] << ks0;
	if constexpr (kIncrKey) key = ((uint32_t)s.g[0] << ks0) | ((uint32_t)s.g[1] << ks1) | ((uint32_t)s.g[2] << ks2);

	while (grid_in_region(s.g[0] + s.ad[0], s.g[1] + s.ad[1], s.g[2] + s.ad[2]))
	{
		// slots to test this iteration, first test in the low bits; the longest axis (slot 0) is always last
		uint32_t seq;
		int nTests;
		if (s.ad[2] != 0 && s.ad[1] != 0)  // Renderer.cuh:792-805
		{
			float rounded = roundDown ? floorf(s.oo[1]) : ceilf(s.oo[1]);
			float t1 = div1(vsub(rounded, s.oo[1]), ko, 1);
			float shortestPosition = vadd(s.oo[2], vmul(s.od[2], t1));
			int shorterDiff = (int)floorf(shortestPosition) - s.g[2];
			seq = shorterDiff != 0 ? (2u | (1u << 2)) : (1u | (2u << 2));
			nTests = 3;
		}
		else if (s.ad[1] != 0) { seq = 1u; nTests = 2; }  // Renderer.cuh:844
		else if (s.ad[2] != 0) { seq = 2u; nTests = 2; }  // Renderer.cuh:865
		else { seq = 0u; nTests = 1; }
		bool again = false;
		if constexpr (kIncrKey)
		{
			kst1 = (uint32_t)s.ad[1] << ks1; kst2 = (uint32_t)s.ad[2] << ks2;
			for (int i = 0; i < nTests; i++)
			{
				const int slot = (int)(seq & 3u);
				seq >>= 2;
				key += slot == 0 ? kst0 : (slot == 1 ? kst1 : kst2);
				if (STATS) c.st.nExist++;  // space_exists: always true for the hash table
				const uint32_t col = lookup_hash_key(c, r, key);
				if (STATS) c.st.nLookup++;
				if (col != kEmpty)
				{
					s.g[0] = (int)((key >> ks0) & 127u); s.g[1] = (int)((key >> ks1) & 127u); s.g[2] = (int)((key >> ks2) & 127u);
					note_lookup_hit(c, p, reg, s.g[0], s.g[1], s.g[2]);
					if (!SHADOW) la_test_hit(p, s, slot, h);
					return col;
				}
			}
			s.g[0] = (int)((key >> ks0) & 127u); s.g[1] = (int)((key >> ks1) & 127u); s.g[2] = (int)((key >> ks2) & 127u);
		}
		else
		for (int i = 0; i < nTests; i++)
		{
			int slot = (int)(seq & 3u);
			seq >>= 2;
			s.g[0] += slot == 0 ? s.ad[0] : 0;
			s.g[1] += slot == 1 ? s.ad[1] : 0;
			s.g[2] += slot == 2 ? s.ad[2] : 0;
			if (!space_exists(c, r, p, s.g[0], s.g[1], s.g[2]))
			{
				uint32_t j = voxel_space_jump<ST, STATS, SHADOW>(c, r, p, s, ko, o, reg, h);
				if (j != kContinue) return j;
				again = true;  // `continue` of the reference's while loop
				break;
			}
			uint32_t col = lookup_voxel(c, r, p, reg, s.g[0], s.g[1], s.g[2]);
			if (col != kEmpty)
			{
				if (!SHADOW) la_test_hit(p, s, slot, h);
				return col;
			}
		}
		if (again) continue;
		// Renderer.cuh:903-908
		s.oo[0] = s.ro[0]; s.oo[1] = s.ro[1]; s.oo[2] = s.ro[2];
		s.ro[0] = vadd(s.ro[0], s.od[0]); s.ro[1] = vadd(s.ro[1], s.od[1]); s.ro[2] = vadd(s.ro[2], s.od[2]);
		s.ad[1] = (int)s.ro[1] - s.g[1];
		s.ad[2] = (int)s.ro[2] - s.g[2];
	}
	// Renderer.cuh:911-914 / 627-630: finish the region with the original algorithm from oldRay's origin
	o[0] = s.oo[0]; o[1] = s.oo[1]; o[2] = s.oo[2];
	if (SHADOW)
	{
		float tt[4];
		return march_steps<ST, STATS, PermRuntime, true>(c, r, p, o, k, reg, tt);
	}
	return march_original<ST, STATS, PermRuntime>(c, r, p, o, k, reg, h);
}

// isInShadowOriginalRayMarch (Renderer.cuh:174-235; LA = false, zero-direction guards) and
// isInShadowRayMarchVoxelSceneLongestAxis (Renderer.cuh:633-694; LA = true, no guards in the region walk).
// originW / regW are in WORLD axes; the walk itself runs in the permutation of the light direction.
template <int ST, bool STATS, bool LA>
VRM_HD bool in_shadow(RayCtx<ST, STATS>& c, const float* originW, const int* regW)
{
	if (!c.light.useShadows) return false;
	using P = typename std::conditional<LA, PermRuntime, PermIdentity>::type;
	P p;
	if constexpr (LA) p = rank_axes(c.light.dir[0], c.light.dir[1], c.light.dir[2]);
	float o[3], d[3];
	int reg[3];
	to_walk(p, originW, o); to_walk(p, c.light.dir, d); to_walk(p, regW, reg);
	// the light direction is the same for every shadow ray: these constants are loop-invariant for the whole kernel
	const RayDir k = make_raydir(d[0], d[1], d[2]);
	RayDir ko = k;
	if constexpr (LA) ko = scaled_raydir(k);
	int32_t ri = region_entry(c, p, reg);
	while (ri != -2)
	{
		ri = skip_null_regions<ST, STATS, P, !LA>(c, p, o, k, reg, ri);
		if (ri == -2) return false;
		RegionRef<ST> r = load_region<ST>(c.sv, ri);
		uint32_t col;
		if constexpr (LA)
		{
			HitInfo unused;
			col = march_longest_axis<ST, STATS, true>(c, r, p, o, k, ko, reg, unused);
		}
		else
		{
			float t[4];
			col = march_steps<ST, STATS, P, true>(c, r, p, o, k, reg, t);
		}
		if (col != kEmpty) return true;
		rebase_region(o, reg);
		ri = position_sane(o) ? region_entry(c, p, reg) : -2;
	}
	return false;
}

// ---------------------------------------------------------------- scene walk

// What a pixel's shadow phase starts from: the hit position and its region in WORLD axes, the shaded colour that survives when the
// light is visible, and which of the reference's two shadow routines the hit site calls.  Also the record of the shadow-ray queue
// between the primary and the shadow kernel (vrm_render.cu).
struct ShadowStart
{
	float hitW[3];
	int regW[3];
	uint32_t lit;   // applyLighting(...) of the hit
	int la;         // 1: isInShadowRayMarchVoxelSceneLongestAxis, 0: isInShadowOriginalRayMarch
};

// rayMarchVoxelScene (Renderer.cuh:338-434) / rayMarchVoxelSceneLongestAxis (Renderer.cuh:917-1010) up to and including the hit's
// lighting; the shadow ray (`* !isInShadow...`, Renderer.cuh:314-315,821-822,...) is the caller's second phase (shadow_nested).
// originW/dirW: WORLD ray (before the scene transform).  Returns true on a hit (ss filled in), false for background.
template <int ST, int ALGO, bool STATS>
VRM_HD bool march_scene_primary(RayCtx<ST, STATS>& c, const float* originW, const float* dirW, float scale, ShadowStart& ss)
{
	using P = typename std::conditional<ALGO == kAlgoOriginal, PermIdentity, PermRuntime>::type;
	P p;
	if constexpr (ALGO != kAlgoOriginal) p = rank_axes(dirW[0], dirW[1], dirW[2]);
	// Ray::convertRayToLocalSpace, Ray.cuh:14-17
	float sW[3] = {canonical_zero(vmul(scale, vsub(originW[0], c.translation[0]))), canonical_zero(vmul(scale, vsub(originW[1], c.translation[1]))),
	               canonical_zero(vmul(scale, vsub(originW[2], c.translation[2])))};
	float o[3], d[3];
	to_walk(p, sW, o); to_walk(p, dirW, d);
	int reg[3] = {(int)floorf(vmul(o[0], 0.015625f)), (int)floorf(vmul(o[1], 0.015625f)), (int)floorf(vmul(o[2], 0.015625f))};
	const int minC = c.sv.minCoord;
	const uint32_t D = c.sv.diameter;
	// scene-entry loop, Renderer.cuh:349-373
	while (reg[0] - minC < 0 || reg[1] - minC < 0 || reg[2] - minC < 0 ||
	       (uint32_t)(reg[0] - minC) > D - 1 || (uint32_t)(reg[1] - minC) > D - 1 || (uint32_t)(reg[2] - minC) > D - 1)
	{
		int far = (int)(D + (uint32_t)minC);
		float t0 = vdiv(vsub((float)((d[0] < 0.0f ? far : minC) * kRegion), o[0]), d[0]);
		float t1 = vdiv(vsub((float)((d[1] < 0.0f ? far : minC) * kRegion), o[1]), d[1]);
		float t2 = vdiv(vsub((float)((d[2] < 0.0f ? far : minC) * kRegion), o[2]), d[2]);
		if (t0 <= 0.0f) t0 = INFINITY;
		if (t1 <= 0.0f) t1 = INFINITY;
		if (t2 <= 0.0f) t2 = INFINITY;
		float tMin = min3(t0, t1, t2);
		if (tMin == INFINITY) return false;
		float s = vadd(tMin, kEps);
		o[0] = along(o[0], s, d[0]); o[1] = along(o[1], s, d[1]); o[2] = along(o[2], s, d[2]);
		reg[0] = (int)floorf(vmul(o[0], 0.015625f)); reg[1] = (int)floorf(vmul(o[1], 0.015625f)); reg[2] = (int)floorf(vmul(o[2], 0.015625f));
	}
	// to region-local coordinates, Renderer.cuh:376-378
	for (int i = 0; i < 3; i++) o[i] = vmul(1.0f, vsub(o[i], (float)(reg[i] * kRegion)));
	const RayDir k = make_raydir(d[0], d[1], d[2]);
	RayDir ko = k;
	if constexpr (ALGO != kAlgoOriginal) ko = scaled_raydir(k);
	int32_t ri = region_entry(c, p, reg);
	// Every lane marches its PRIMARY ray to a hit or out of the scene -- the loop has one exit, so the warp reconverges behind it.
	// Executed as the reference nests it (shadow march inside the hit branch inside the region loop) the shadow rays of a warp ran one
	// hit time after the other: 11.9 of 32 threads active in the shadow half of the hash table kernels (profiles/r01j).
	uint32_t col = kEmpty;
	HitInfo h;
	while (ri != -2)
	{
		ri = skip_null_regions<ST, STATS, P, false>(c, p, o, k, reg, ri);
		if (ri == -2) break;
		RegionRef<ST> r = load_region<ST>(c.sv, ri);
		if constexpr (ALGO == kAlgoOriginal) col = march_original<ST, STATS, P>(c, r, p, o, k, reg, h);
		else col = march_longest_axis<ST, STATS, false>(c, r, p, o, k, ko, reg, h);
		if (col != kEmpty) break;
		rebase_region(o, reg);
		ri = position_sane(o) ? region_entry(c, p, reg) : -2;
	}
	if (col == kEmpty) return false;
	// applyLighting(...)  (Renderer.cuh:314-315,821-822,...)
	to_world(p, h.pos, ss.hitW); to_world(p, reg, ss.regW);
	ss.lit = apply_lighting(c.light, c.translation, col, h.nAxisW, h.nSign, ss.hitW, ss.regW);
	ss.la = ALGO == kAlgoOriginal ? 0 : h.laShadow;
	return true;
}

// ... * !isInShadow...(Ray(hit, LIGHT_DIRECTION), currentRegion): which routine depends on the hit site (SURVEY.md 8a18)
template <int ST, int ALGO, bool STATS>
VRM_HD bool shadow_nested(RayCtx<ST, STATS>& c, const ShadowStart& ss)
{
	if constexpr (ALGO == kAlgoOriginal) return in_shadow<ST, STATS, false>(c, ss.hitW, ss.regW);
	else return ss.la ? in_shadow<ST, STATS, true>(c, ss.hitW, ss.regW) : in_shadow<ST, STATS, false>(c, ss.hitW, ss.regW);
}

// Both phases for one ray (trace kernels, host sim).  Returns the pixel colour (0 = background).
template <int ST, int ALGO, bool STATS>
VRM_HD uint32_t march_scene(RayCtx<ST, STATS>& c, const float* originW, const float* dirW, float scale)
{
	ShadowStart ss;
	if (!march_scene_primary<ST, ALGO, STATS>(c, originW, dirW, scale, ss)) return 0;
	return ss.lit * (uint32_t)!shadow_nested<ST, ALGO, STATS>(c, ss);
}

// calculateWorldRay (Renderer.cuh:1013-1022) + Camera::generateRay (Camera.cuh:25-29).  cam = 15 floats.  len = |o - eye|, the
// world distance from the camera origin to the ray's image-plane origin o.
VRM_HD void primary_ray(const float* cam, uint32_t x, uint32_t y, uint32_t W, uint32_t H, float* o, float* d, float& len)
{
	float u = vdiv(vadd((float)x, 0.5f), (float)W);
	float v = vdiv(vadd((float)(H - y), 0.5f), (float)H);
	float rel[3];
	for (int i = 0; i < 3; i++)
	{
		o[i] = vadd(vadd(cam[3 + i], vmul(u, cam[6 + i])), vmul(v, cam[9 + i]));
		rel[i] = vsub(o[i], cam[i]);
	}
	len = vsqrt(vadd(vadd(vmul(rel[0], rel[0]), vmul(rel[1], rel[1])), vmul(rel[2], rel[2])));
	d[0] = vdiv(rel[0], len); d[1] = vdiv(rel[1], len); d[2] = vdiv(rel[2], len);
}

VRM_HD void primary_ray(const float* cam, uint32_t x, uint32_t y, uint32_t W, uint32_t H, float* o, float* d)
{
	float len;
	primary_ray(cam, x, y, W, H, o, d, len);
}

// ---------------------------------------------------------------- hit surfaces (vrm_hit_surface_*, DESIGN.md §3.6)
//
// Depth and entered face of a reported hit record hit = {x, y, z, flag} for the WORLD ray origin P, unit direction D: the exact ray
// against the slabs of the hit voxel in local units, s = scale * (P - translation) as march_scene_primary transforms the origin.  For
// every axis a with D_a != 0: t_a = (f_a - s_a) / D_a with f_a = D_a > 0 ? h_a : h_a + 1; t = the largest t_a, ties to the earlier
// axis; face = 1 + 2a + (D_a < 0), so 1..6 = -x, +x, -y, +y, -z, +z, the outward normal of the face the ray enters through.
//   depth = len + t / scale  (withLen: a camera ray, len from primary_ray -- the world distance from the eye along the pixel's ray)
//         = t / scale        (a traced ray: the world ray parameter, P + depth * D is the entry point)
// flag 0: +inf and face 0.  No axis with D_a != 0: NaN and face 0 (no camera ray).  Not clamped: a depth below len (below 0 for a
// trace) means the origin lies inside the hit voxel, or the reference walk's drift reported a voxel the exact ray only grazes.
// This one function is the definition: the sm_100a kernel (vrm_surface.cu) and the CPU tests' host build both call it.
VRM_HD float hit_surface(const int32_t* hit, const float* P, const float* D, const float* translation, float scale, float len, bool withLen,
                         uint32_t& face)
{
	face = 0u;
	if (hit[3] == 0) return INFINITY;
	float t = 0.0f;
	for (int a = 0; a < 3; a++)
	{
		if (D[a] == 0.0f) continue;
		const float s = vmul(scale, vsub(P[a], translation[a]));
		const float f = (float)(D[a] > 0.0f ? hit[a] : hit[a] + 1);
		const float ta = vdiv(vsub(f, s), D[a]);
		if (face == 0u || ta > t) { t = ta; face = 1u + 2u * (uint32_t)a + (D[a] < 0.0f ? 1u : 0u); }
	}
	if (face == 0u) return NAN;
	const float q = vdiv(t, scale);
	return withLen ? vadd(len, q) : q;
}

// ---------------------------------------------------------------- exact ray casts (vrm_cast_*, DESIGN.md §3.7)
//
// The first STORED voxel along the exact ray within a parameter interval, with its entry depth, face and colour.  The definition is the
// cell-by-cell walk of include/vrm_b200.h "exact ray casts" in the local frame s = scale * (P - translation), tau = scale * t:
//   plane k of axis a (D_a != 0) is crossed at tau_a(k) = (k - s_a) / D_a (hit_surface's expression; monotone in k, not strictly once
//   |k - s_a| passes ~2^23), the walk starts in the cell after every crossing with tau <= tau0 and repeatedly takes the smallest next
//   crossing, ties to the earlier axis, until it passes tau1.  At one tau the walk therefore makes all of x's crossings, then y's, then
//   z's, so the walk's state right after axis m crosses a plane at tau X is: axis m in the cell behind that plane, every earlier axis in
//   the cell after all its crossings <= X, every later axis in the cell after all its crossings < X (cast_search).  That is what makes
//   the leaps below exact: out of a null 64^3 region, out of an 8^3 cluster whose mask bit is clear, and into the region table's box,
//   each leap lands in the state the cell-by-cell walk has right after it crosses the exit (entry) plane -- including ties between axes
//   and runs of equal tau on one axis.  Cells are stepped one by one only inside occupied clusters.
// This one function is the definition: the sm_100a kernel (vrm_cast.cu) and the CPU tests' host build both call it.

struct CastResult
{
	int32_t hit[4];   // global voxel x, y, z and 1; all 0 for a miss
	float depth;      // world ray parameter (views: distance from the eye); +inf for a miss
	uint32_t face;    // 1..6 = -x, +x, -y, +y, -z, +z of the entered face; 0 for a hit in the start cell and for a miss
	uint32_t colour;  // the stored colour (exactly what vrm_lookup returns); kEmpty for a miss
};

// tau of plane k on one axis, through the ray's exact division (bit-identical to vdiv)
VRM_HD float cast_tau(int k, float s, float d, float rd, float thr) { return div1(vsub((float)k, s), d, rd, thr); }

// The cell of one axis after every crossing with tau <= X (strict: tau < X), searched in [lo, hi]: the largest m there with
// P(m) = (d < 0) == (strict ? tau(m) >= X : tau(m) > X), true for every m up to the answer as tau is monotone.  lo - 1 when P fails on
// all of [lo, hi] (the cell lies below lo); hi when the cell is hi or above.  The first probe is the rounded position s + X d, which
// is off by at most one cell except in runs of equal tau, so a search usually costs two divisions.
VRM_HD int cast_search(float s, float d, float rd, float thr, float X, bool strict, int lo, int hi)
{
	const bool neg = d < 0.0f;
	auto P = [&](int m) {
		const float t = cast_tau(m, s, d, rd, thr);
		return neg == (strict ? t >= X : t > X);
	};
	const float e = vadd(s, vmul(X, d));
	const int k = e >= (float)hi ? hi : (e >= (float)lo ? (int)floorf(e) : lo);
	int a = lo - 1, b = hi;  // the answer lies in [a, b]
	if (P(k)) a = k; else b = k - 1;
	if (a < b)
	{
		const int m = a == k ? k + 1 : k - 1;
		if (P(m)) a = m; else b = m - 1;
	}
	while (a < b)
	{
		const int m = a + (b - a + 1) / 2;
		if (P(m)) a = m; else b = m - 1;
	}
	return a;
}

// The cuckoo lookup with the found flag kept apart from the colour (a voxel may be stored with the colour kEmpty)
VRM_HD bool cast_hash_probe(const SceneView& sv, const RegionRef<kStorageHash>& r, uint32_t key, uint32_t& colour)
{
	const unsigned long long e1 = ldg(sv.slots + (r.base1 + hash_slot1(key, r.seed1, r.n)));
	const unsigned long long e2 = ldg(sv.slots + (r.base2 + hash_slot2(key, r.seed2, r.n)));
	if (slot_key(e1) == key) { colour = slot_colour(e1); return true; }
	if (slot_key(e2) == key) { colour = slot_colour(e2); return true; }
	return false;
}

// One ray.  P, D: world origin and direction; [tNear, tFar]: the interval of the world ray parameter.  withLen (views): depth = len +
// tau / scale, len for a start-cell hit; otherwise depth = tau / scale, tNear for a start-cell hit.
template <int ST>
VRM_HD void cast_ray(const SceneView& sv, const float* P, const float* D, const float* tr, float scale, float tNear, float tFar, float len,
                     bool withLen, CastResult& res)
{
	res.hit[0] = res.hit[1] = res.hit[2] = res.hit[3] = 0;
	res.depth = INFINITY; res.face = 0u; res.colour = kEmpty;
	if (!(isfinite(P[0]) && isfinite(P[1]) && isfinite(P[2]) && isfinite(D[0]) && isfinite(D[1]) && isfinite(D[2]) && isfinite(tNear)) ||
	    tFar != tFar || tNear > tFar)
		return;
	float s[3];
	for (int a = 0; a < 3; a++) s[a] = vmul(scale, vsub(P[a], tr[a]));
	const float tau0 = vmul(tNear, scale), tau1 = vmul(tFar, scale);
	// an overflowing local origin or start (huge coordinates, a non-finite translation) has no cell: a miss
	if (!(isfinite(s[0]) && isfinite(s[1]) && isfinite(s[2]) && isfinite(tau0))) return;
	RayDir k = make_raydir(D[0], D[1], D[2]);
	// the fast division also needs its quotients far from overflow: |k - s| < 2^65, |q| < 2^105
	if (!(fabsf(s[0]) < 1.8446744e19f && fabsf(s[1]) < 1.8446744e19f && fabsf(s[2]) < 1.8446744e19f)) k.thr = NAN;
	const int L = kRegion * sv.minCoord, Hb = L + kRegion * (int)sv.diameter;  // the region table's box [L, Hb)^3
	auto tau = [&](int a, int plane) { return cast_tau(plane, s[a], k.d[a], k.rd[a], k.thr); };
	auto next = [&](int a, int cell) { return tau(a, k.d[a] > 0.0f ? cell + 1 : cell); };  // the next crossing out of `cell`
	auto search = [&](int a, float X, bool strict, int lo, int hi) { return cast_search(s[a], k.d[a], k.rd[a], k.thr, X, strict, lo, hi); };
	auto inBox = [&](int v) { return v >= L && v < Hb; };

	// start cell: the cell after every crossing with tau <= tau0 (searched in [L - 1, Hb]: only its cell inside the box matters)
	int c[3];
	for (int a = 0; a < 3; a++)
	{
		if (k.d[a] == 0.0f)
		{
			const float fl = floorf(s[a]);
			if (!(fl >= (float)L && fl < (float)Hb)) return;  // the axis never moves: the ray never enters the box
			c[a] = (int)fl;
		}
		else c[a] = search(a, tau0, false, L - 1, Hb);
	}
	float t = tau0;
	uint32_t face = 0u;
	if (!(inBox(c[0]) && inBox(c[1]) && inBox(c[2])))
	{
		// leap to the box: its entry is the latest per-axis entry crossing (ties: the later axis crosses last)
		int m = -1;
		float E = 0.0f;
		for (int a = 0; a < 3; a++)
		{
			if (k.d[a] == 0.0f || inBox(c[a])) continue;
			if ((c[a] < L) != (k.d[a] > 0.0f)) return;  // outside and moving away
			const float Ea = tau(a, c[a] < L ? L : Hb);
			if (m < 0 || Ea >= E) { E = Ea; m = a; }
		}
		if (!(E <= tau1)) return;
		for (int b = 0; b < 3; b++)
		{
			if (b == m || k.d[b] == 0.0f) continue;
			c[b] = search(b, E, b > m, L - 1, Hb);
			if (!inBox(c[b])) return;  // another axis left the box before this one entered it
		}
		c[m] = k.d[m] > 0.0f ? L : Hb - 1;
		t = E;
		face = 1u + 2u * (uint32_t)m + (k.d[m] < 0.0f ? 1u : 0u);
	}
	float nt[3];
	for (int a = 0; a < 3; a++) nt[a] = k.d[a] != 0.0f ? next(a, c[a]) : 0.0f;

	// Leap to the exit of the aligned cube of side S around c: the first exit crossing (ties: the earlier axis), the crossing axis into
	// the cell behind it, the others by cast_search inside the cube.  false: the walk ends (past tau1, no moving axis, out of the box).
	auto leap = [&](int S) -> bool {
		int m = -1;
		float X = 0.0f;
		for (int a = 0; a < 3; a++)
		{
			if (k.d[a] == 0.0f) continue;
			const int lo = c[a] & -S;
			const float Xa = tau(a, k.d[a] > 0.0f ? lo + S : lo);
			if (m < 0 || Xa < X) { X = Xa; m = a; }
		}
		if (m < 0 || !(X <= tau1)) return false;
		for (int b = 0; b < 3; b++)
		{
			if (b == m || k.d[b] == 0.0f) continue;
			const int lo = c[b] & -S;
			c[b] = search(b, X, b > m, lo, lo + S - 1);
			nt[b] = next(b, c[b]);
		}
		c[m] = k.d[m] > 0.0f ? (c[m] & -S) + S : (c[m] & -S) - 1;
		nt[m] = next(m, c[m]);
		t = X;
		face = 1u + 2u * (uint32_t)m + (k.d[m] < 0.0f ? 1u : 0u);
		return inBox(c[m]);
	};
	// One crossing of the cell-by-cell walk.  false: the walk ends.
	auto step = [&]() -> bool {
		int m = -1;
		for (int a = 0; a < 3; a++)
			if (k.d[a] != 0.0f && (m < 0 || nt[a] < nt[m])) m = a;
		if (m < 0 || !(nt[m] <= tau1)) return false;
		t = nt[m];
		face = 1u + 2u * (uint32_t)m + (k.d[m] < 0.0f ? 1u : 0u);
		c[m] += k.d[m] > 0.0f ? 1 : -1;
		nt[m] = next(m, c[m]);
		return inBox(c[m]);
	};

	const uint32_t Dm = sv.diameter;
	for (;;)  // regions
	{
		const uint32_t u0 = (uint32_t)(c[0] - L) >> 6, u1 = (uint32_t)(c[1] - L) >> 6, u2 = (uint32_t)(c[2] - L) >> 6;
		const int32_t ri = ldg(sv.regionTable + (u0 + u1 * Dm + u2 * Dm * Dm));
		if (ri < 0)
		{
			if (!leap(kRegion)) return;
			continue;
		}
		const RegionRef<ST> r = load_region<ST>(sv, ri);
		const int rg0 = c[0] & -kRegion, rg1 = c[1] & -kRegion, rg2 = c[2] & -kRegion;
		auto inRegion = [&]() { return (c[0] & -kRegion) == rg0 && (c[1] & -kRegion) == rg1 && (c[2] & -kRegion) == rg2; };
		for (;;)  // clusters of the region
		{
			const uint32_t cid = vcs_cluster_id((uint32_t)(c[0] - rg0) >> 3, (uint32_t)(c[1] - rg1) >> 3, (uint32_t)(c[2] - rg2) >> 3);
			if (!((ldg(sv.clusterMask + (r.ri * 16u + (cid >> 5))) >> (cid & 31u)) & 1u))
			{
				if (!leap(8)) return;
				if (!inRegion()) break;
				continue;
			}
			const int cl0 = c[0] & -8, cl1 = c[1] & -8, cl2 = c[2] & -8;
			uint32_t wordAt = 0xFFFFFFFFu;  // VCS: the header word in hand (32 cells' occupancy)
			uint2 h = {0u, 0u};
			for (;;)  // cells of the cluster
			{
				const uint32_t x = (uint32_t)(c[0] - rg0), y = (uint32_t)(c[1] - rg1), z = (uint32_t)(c[2] - rg2);
				bool found;
				uint32_t colour = kEmpty;
				if constexpr (ST == kStorageVcs)
				{
					const uint32_t code = ((x & 7u) << 6) | ((y & 7u) << 3) | (z & 7u);
					if (code >> 5 != wordAt) { wordAt = code >> 5; h = ldg(sv.headers + vcs_header_index(r.ri, cid, wordAt)); }
					const uint32_t bit = code & 31u;
					found = (h.x >> bit) & 1u;
					if (found) colour = ldg(sv.values + vcs_colour_index(h.x, h.y, bit));
				}
				else found = cast_hash_probe(sv, r, hash_key(x, y, z), colour);
				if (found)
				{
					res.hit[0] = c[0]; res.hit[1] = c[1]; res.hit[2] = c[2]; res.hit[3] = 1;
					res.face = face;
					res.colour = colour;
					if (face == 0u) res.depth = withLen ? len : tNear;
					else { const float q = vdiv(t, scale); res.depth = withLen ? vadd(len, q) : q; }
					return;
				}
				if (!step()) return;
				if ((c[0] & -8) != cl0 || (c[1] & -8) != cl1 || (c[2] & -8) != cl2) break;
			}
			if (!inRegion()) break;
		}
	}
}

}  // namespace vrm
