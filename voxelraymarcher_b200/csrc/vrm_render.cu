// vrm_render.cu -- render / trace / lookup kernels (sm_100a).  Replaces rayMarchSceneOriginal and
// rayMarchSceneJumpAxis (renderer/Renderer.cuh:1033-1063) and their launch (main/Main.cu:105-163).
//
// One thread per pixel; a warp owns an 8x4 pixel tile (coherent primary rays: neighbouring pixels walk the same
// clusters, so their lookups share 128-byte lines), a 128-thread CTA owns a 32x4 row of four tiles, blockIdx.z is the
// view.  Storage type and algorithm are template parameters: four specialised kernels instead of the reference's two
// kernels with virtual storage dispatch (the specialisation the reference's own dead OptimizedFunctions.cuh aimed at).
// Compile with -fmad=false as a second line of defence; the core already spells every float op with *_rn intrinsics.
#include "vrm_internal.h"

#include <cstdlib>
#include "vrm_flat.cuh"
#include "vrm_lean.cuh"
#include "../../include/vrm_b200.h"

using namespace vrm;

namespace
{

// Tunables (A/B builds: make VARIANT_FLAGS=-DVRM_... OUT=...; the defaults are the measured choices, DESIGN.md 3.2)
#ifndef VRM_BLOCK_TILES_Y
#define VRM_BLOCK_TILES_Y 1
#endif
#ifndef VRM_BLOCK_TILES_X
#define VRM_BLOCK_TILES_X 4
#endif
#ifndef VRM_HIT_BARRIER
#define VRM_HIT_BARRIER 1  // VCS + longest axis state machine: 1 = a tile shades and starts its shadow rays together (march_scene_flat_warp), 0 = independent lanes
#endif
#ifndef VRM_TRACE_HIT_BARRIER
#define VRM_TRACE_HIT_BARRIER 0  // the same for trace_rays (arbitrary rays)
#endif
#ifndef VRM_WARP_STORE
#define VRM_WARP_STORE 1        // fused form (VCS + longest axis): per-warp stores when the frame is in this GPU's memory (1.398 -> 1.377 ms; with 9 CTAs per SM 1.363)
#endif
#ifndef VRM_WARP_STORE_QUEUE
#define VRM_WARP_STORE_QUEUE 0  // the same for the nested-loop render kernels of the shadow-ray queue pipelines
#endif
#ifndef VRM_FLAT_LA_MINBLOCKS
#define VRM_FLAT_LA_MINBLOCKS 4
#endif

#ifndef VRM_FUSED_CTAS
#define VRM_FUSED_CTAS 9   // > 0: resident CTAs per SM the fused form (FORM 2) is compiled for, 0: VRM_FLAT_LA_MINBLOCKS * 2.  Measured with the fast paths in
                           // place: 7 (72 registers, no spills) 1.439 ms, 8 (64) 1.398, 9 (56, ~0.5 KB of spills) 1.379, 10 (48) 1.404 -- occupancy beats the spills up to 36 warps
#endif
#ifndef VRM_TILE_W
#define VRM_TILE_W 8
#endif
constexpr int kTileW = VRM_TILE_W, kTileH = 32 / VRM_TILE_W;          // pixels per warp
constexpr int kBlockTilesX = VRM_BLOCK_TILES_X, kBlockTilesY = VRM_BLOCK_TILES_Y;
constexpr int kBlockW = kTileW * kBlockTilesX;  // 32
constexpr int kBlockH = kTileH * kBlockTilesY;  // 8
constexpr int kRenderThreads = kBlockW * kBlockH;  // 128 threads = a 32x4 pixel row of four tiles: measured 2.5-3 % faster than 32x8 for every combination (fewer warps parked at the CTA barrier behind a slow tile)

struct RenderArgs
{
	SceneView sv;
	Lighting light;
	LightWalk lw;
	float translation[3];
	float scale;
	const float* cams;  // nViews x 15
	float cam0[15];     // camInline: the camera of a single-view launch travels in the kernel arguments (constant bank): no upload, no loads
	uint32_t camInline;
	uint32_t W, H;
	size_t viewPixels;     // pixel slots between the outputs of consecutive views (W * H, or a multiple of it for interleaved view sharding)
	size_t rgbViewPixels;  // the same for the frame array `rgb` alone (it differs when the frames are rendered into the handle's local buffer first)
	float invW, invH;      // RN(1 / W), RN(1 / H) (host): exact division by a constant in primary_ray_flat
	uint32_t rgbLocal;     // host side only: the frame `rgb` points into this GPU's own memory (selects the per-warp store kernels)
	uint32_t rowWordsOk;   // 1 when every 32-pixel row segment starts on a 4-byte boundary (W * 3 % 4 == 0 and an aligned base)
	uint32_t rowBulkOk;    // 1 when every such segment also starts on a 16-byte boundary and the frame is not in this GPU's memory: the CTA-staged rows leave as bulk async copies
	uint32_t yBase, yEnd;  // rows rendered by this launch (a band of the frame: vrm_render overlaps the D2H copy of band k with band k+1)
	uint8_t* rgb;       // nViews x H x W x 3
	int32_t* hits;      // nullable, nViews x H x W x 4
	Stats* stats;       // nullable
	void* defer;        // DeferHeader + records: rays parked for resume_kernel (vrm_flat.cuh kPpDefer)
	unsigned int* queue;   // persistent kernel: next unclaimed pixel slot
	uint32_t tilesX, tilesPerView, nViews;
	uint32_t* parkBits;    // lean kernels: one bit per ray (index (view * H + y) * W + x) that must be re-traced by resume_lean_kernel
	unsigned int* parkCtl; // {parked rays, resume blocks done}
	int4* shadowItems;     // shadow-ray queue (two int4 per record), null when shadows are off
	unsigned int* shadowCtl;  // {records queued, next record to claim}
	uint32_t shadowCap;
	uint32_t skipDead;     // 1: a hit whose shaded colour is already black queues no shadow ray (0 * !shadow = 0)
	HorizonView hv;        // shadow horizon map (cells null: none); read by the fused kernel (FORM 2) only
};

// ---- shadow-ray queue ------------------------------------------------------------------------------------------------------------
// The render kernels trace PRIMARY rays only.  A pixel whose ray hit is shaded there and its shadow ray -- start position and region in
// world axes, the shaded colour, which of the reference's two shadow routines the hit site calls -- is appended to a queue in device
// memory (one ballot + one atomicAdd per warp); shadow_kernel then walks the queued rays 32 consecutive records per warp.  Why: only
// ~30 % of the pixels of the terrain frame hit anything and lit pixels' shadow rays are long while shadowed ones end early, so inside
// the tile that found the hits the shadow phase ran at 11.8 of 32 lanes (hash table kernels, profiles/r02c) -- half of the frame time.
// All shadow rays share one direction, so consecutive records (neighbouring pixels of a tile, tiles of a CTA) stay coherent.  Same
// operations per ray as before; the frame receives the shaded colour first and shadow_kernel blacks out the pixels whose light is
// blocked (Renderer.cuh:314-315: colour * !isInShadow).
struct ShadowArgs
{
	SceneView sv;
	Lighting light;
	LightWalk lw;
	float translation[3];
	const int4* items;
	unsigned int* ctl;
	uint32_t cap;
	uint32_t skipDead;     // 1: a record whose shaded colour is already black is not traced (0 * !shadow = 0); 0: trace everything (reference-comparable event counters)
	uint8_t* rgb;          // frame: the record's pixel number indexes RGB8 triples ...
	uint32_t* colour;      // ... or (trace_rays) one uint32 colour per ray when this is not null
	Stats* stats;
	void* defer;
};

template <class Args>
__device__ __forceinline__ void shadow_enqueue(const Args& a, bool hit, const ShadowStart& ss, uint32_t pixel)
{
	const bool want = hit && !(a.skipDead && ss.lit == 0u);
	const unsigned m = __ballot_sync(0xFFFFFFFFu, want);
	if (m == 0u) return;
	const unsigned lane = threadIdx.x & 31u;
	const int leader = __ffs(m) - 1;
	unsigned base = 0;
	if ((int)lane == leader) base = atomicAdd(a.shadowCtl, (unsigned)__popc(m));
	base = __shfl_sync(0xFFFFFFFFu, base, leader);
	if (want)
	{
		const unsigned i = base + __popc(m & ((1u << lane) - 1u));
		if (i < a.shadowCap)  // (the launch wrapper sizes the queue for every pixel of the launch)
		{
			a.shadowItems[2 * (size_t)i] = make_int4(__float_as_int(ss.hitW[0]), __float_as_int(ss.hitW[1]), __float_as_int(ss.hitW[2]), ss.regW[0]);
			a.shadowItems[2 * (size_t)i + 1] = make_int4(ss.regW[1], ss.regW[2], (int)pixel, (int)(ss.lit | (ss.la ? 0x80000000u : 0u)));
		}
	}
}

template <bool STATS, int ST>
__device__ __forceinline__ void flush_stats(const RayCtx<ST, STATS>& c, Stats* out)
{
	if constexpr (STATS)
	{
		unsigned long long v[7] = {c.st.nExist, c.st.nExistFalse, c.st.nLookup, c.st.nLookupHit, c.st.nProbe2, c.st.nRegionReads, c.st.nCrawlSkipped};
#pragma unroll
		for (int k = 0; k < 7; k++)
		{
			unsigned long long x = v[k];
			for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, o);
			if ((threadIdx.x & 31) == 0 && x) atomicAdd(reinterpret_cast<unsigned long long*>(out) + k, x);
		}
	}
}

// a ray parked by FlatRay::defer: tell the resume kernel where its colour goes
template <class Ray>
__device__ __forceinline__ void park_output(void* queue, int slot, const void* out, uint32_t kind)
{
	typename Ray::Deferred* items = reinterpret_cast<typename Ray::Deferred*>(static_cast<DeferHeader*>(queue) + 1);
	items[slot].outAddr = reinterpret_cast<unsigned long long>(out);
	items[slot].outKind = kind;
}

struct ResumeArgs
{
	SceneView sv;
	Lighting light;
	LightWalk lw;
	float translation[3];
	Stats* stats;
	void* defer;
};

// Continues the rays the render / trace kernels parked (region-face ping-pong, vrm_flat.cuh): a handful per frame at most,
// each worth 10^5-10^6 iterations of the reference, fast-forwarded here in place.  One thread per ray; ONE block, which also
// re-arms the queue for the next launch (so the render path needs no memset).
constexpr int kResumeThreads = 256;
template <int ST, int ALGO, bool STATS>
__global__ void __launch_bounds__(kResumeThreads) resume_kernel(const ResumeArgs a)
{
	using Ray = FlatRay<ST, ALGO, STATS>;
	DeferHeader* h = static_cast<DeferHeader*>(a.defer);
	typename Ray::Deferred* items = reinterpret_cast<typename Ray::Deferred*>(h + 1);
	const unsigned int n = h->count < h->capacity ? h->count : h->capacity;
	RayCtx<ST, STATS> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
	{
		Ray ray = items[i].ray;
		c.hitOut = items[i].hitOut;
		while (ray.st != kStDone) ray.template step<kPpInline>(c);
		const uint32_t color = ray.result;
		if (items[i].outKind == 0u)
		{
			uint8_t* px = reinterpret_cast<uint8_t*>(items[i].outAddr);
			px[0] = (uint8_t)(color >> 16); px[1] = (uint8_t)((color >> 8) & 0xFF); px[2] = (uint8_t)(color & 0xFF);
		}
		else *reinterpret_cast<uint32_t*>(items[i].outAddr) = color;
	}
	__syncthreads();
	if (threadIdx.x == 0) h->count = 0u;
	if constexpr (STATS)
	{
		// lanes leave the loop together (uniform trip count per warp is not guaranteed): plain atomics
		unsigned long long v[7] = {c.st.nExist, c.st.nExistFalse, c.st.nLookup, c.st.nLookupHit, c.st.nProbe2, c.st.nRegionReads, c.st.nCrawlSkipped};
		for (int k = 0; k < 7; k++) if (v[k]) atomicAdd(reinterpret_cast<unsigned long long*>(a.stats) + k, v[k]);
	}
}

// Bulk asynchronous copy shared -> global (the TMA unit's non-tensor form).  A CTA whose last instruction is an ordinary store into
// page-locked host memory or a peer GPU keeps its slot on the SM until PCIe / NVLink has acknowledged the store; a bulk copy is handed
// to the copy unit, and the CTA only waits until its shared memory has been READ (cp.async.bulk.wait_group.read) before it leaves.
// dst and src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_store_row(void* dst, const void* src, uint32_t bytes)
{
	const uint32_t s = (uint32_t)__cvta_generic_to_shared(src);
	asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(s), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_store_commit_and_release()
{
	asm volatile("cp.async.bulk.commit_group;" ::: "memory");
	asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// FORM 0: nested loops, primary rays only (shadow rays go to the queue); 1: state machine, primary rays only; 2: state machine with the
// shadow ray in the kernel behind a hit barrier (march_scene_flat_warp) -- the default for VCS + longest axis, see launch_render_t
// WSTORE: every warp writes its own 8x4 tile (four 24-byte row segments) and leaves -- no CTA barrier, so a warp that finishes early does
// not wait for the slowest tile of its CTA (14 % of the warp-samples of the fused kernel sat at that barrier, profiles/r02g).  Chosen
// when the frame lives in this GPU's memory; frames in page-locked host memory or on a peer GPU keep the CTA-staged 96-byte rows
// (fewer, larger transactions over PCIe / NVLink).
template <int ST, int ALGO, bool STATS, int FORM, bool WSTORE>
__global__ void __launch_bounds__(kRenderThreads, (FORM == 2 && VRM_FUSED_CTAS > 0) ? VRM_FUSED_CTAS : ((FORM != 0 && ALGO != kAlgoOriginal) ? VRM_FLAT_LA_MINBLOCKS : (ST == kStorageHash ? (ALGO == kAlgoOriginal ? 6 : 5) : (ALGO == kAlgoOriginal ? 6 : 4))) * 8 / (VRM_BLOCK_TILES_Y * VRM_BLOCK_TILES_X)) render_kernel(const RenderArgs a)
{
	constexpr bool FLATLOOP = FORM != 0;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t lx = (warp % kBlockTilesX) * kTileW + (lane & (kTileW - 1)), ly = (warp / kBlockTilesX) * kTileH + (lane / kTileW);
	const uint32_t x0 = blockIdx.x * kBlockW, y0 = a.yBase + blockIdx.y * kBlockH;
	const uint32_t x = x0 + lx, y = y0 + ly;
	const bool inside = x < a.W && y < a.yEnd;
	// The CTA's 32x4 pixels are staged in shared memory and written as 4 rows of 96 contiguous bytes (24 words per row,
	// one STG.32 per thread) instead of three scattered byte stores per pixel (Renderer.cuh:1027-1030); this is also what makes
	// writing the frame straight into pinned host memory (vrm_render) efficient.
	__shared__ __align__(16) uint32_t staged[kBlockH][kBlockW * 3 / 4];
	RayCtx<ST, STATS> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	uint32_t color = 0;
	bool hit = false;
	ShadowStart ss;
	ss.hitW[0] = ss.hitW[1] = ss.hitW[2] = 0.0f; ss.regW[0] = ss.regW[1] = ss.regW[2] = 0; ss.lit = 0u; ss.la = 0;
	const size_t pixel = (size_t)blockIdx.z * a.viewPixels + (size_t)y * a.W + x;        // hit map slot
	const size_t pixelOut = (size_t)blockIdx.z * a.rgbViewPixels + (size_t)y * a.W + x;  // frame slot (also the shadow record's)
	if constexpr (FLATLOOP)
	{
		// warp-cooperative state machine (vrm_flat.cuh): every lane takes part in the votes, lanes outside the image just idle
		float o[3] = {0.0f, 0.0f, 0.0f}, d[3] = {0.0f, 0.0f, 0.0f};
		if (inside)
		{
			float camv[15];
			if (a.camInline)
			{
#pragma unroll
				for (int i = 0; i < 15; i++) camv[i] = a.cam0[i];
			}
			else
			{
				const float* cam = a.cams + (size_t)blockIdx.z * 15;
#pragma unroll
				for (int i = 0; i < 15; i++) camv[i] = __ldg(cam + i);
			}
			primary_ray_flat(camv, x, y, a.W, a.H, a.invW, a.invH, o, d);
			if (a.hits)
			{
				// the hit map slot is cleared here and filled at the hit site (record_hit_voxel)
				c.hitOut = a.hits + 4 * pixel;
				*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
			}
		}
		c.deferQueue = a.defer;
		if constexpr (FORM == 2)
		{
			c.skipDead = a.skipDead;
			c.hv = a.hv;
#if VRM_SMEM_MASK
			__shared__ uint32_t stagedMask[kRenderThreads / 32][16];
			c.smMask = stagedMask[warp];
#endif
			// both phases here: lanes that hit wait at the hit barrier, the tile then shades and walks its shadow rays together
			int slot;
			color = march_scene_flat_warp<ST, ALGO, STATS, kPpDefer>(c, inside, o, d, a.scale, slot);
			if (slot >= 0) park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.rgb + 3 * pixelOut, 0u);
		}
		else
		{
		FlatRay<ST, ALGO, STATS> ray;
		march_primary_flat_warp<ST, ALGO, STATS, kPpDefer>(c, inside, o, d, a.scale, ray);
		if (ray.st == kStHit)
		{
			ray.shade_hit(c, ss);
			hit = true;
			color = ss.lit;
		}
		else if (ray.st == kStPark)
		{
			// region-face ping-pong (vrm_flat.cuh): the ray goes to the resume kernel, which finishes it -- shadow ray included
			const int slot = ray.park(c);
			if (slot >= 0) park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.rgb + 3 * pixelOut, 0u);
			else { while (ray.st < kStDone) ray.template step<kPpOff>(c); color = ray.result; }  // queue full: crawl on like the reference
		}
		else color = ray.result;
		}
	}
	else if (inside)
	{
		float camv[15];
		if (a.camInline)
		{
#pragma unroll
			for (int i = 0; i < 15; i++) camv[i] = a.cam0[i];
		}
		else
		{
			const float* cam = a.cams + (size_t)blockIdx.z * 15;
#pragma unroll
			for (int i = 0; i < 15; i++) camv[i] = __ldg(cam + i);
		}
		float o[3], d[3];
		primary_ray(camv, x, y, a.W, a.H, o, d);
		hit = march_scene_primary<ST, ALGO, STATS>(c, o, d, a.scale, ss);
		color = hit ? ss.lit : 0u;
		if (a.hits) reinterpret_cast<int4*>(a.hits)[pixel] = make_int4(c.hit[0], c.hit[1], c.hit[2], c.hit[3]);
	}
	// the shadow ray of a hit goes to the queue; without shadows (USE_SHADOWS false, Main.cu:41) the shaded colour is final
	if constexpr (FORM != 2) { if (a.shadowItems) shadow_enqueue(a, hit, ss, (uint32_t)pixelOut); }
	// writeColorToFramebuffer, Renderer.cuh:1024-1031 (red = colour >> 16, unmasked, then narrowed to a byte)
	if constexpr (WSTORE)
	{
	// per-warp staging: each warp writes its own 8x4 tile as four 24-byte row segments, no CTA barrier
	const uint32_t tx0 = x0 + (warp % kBlockTilesX) * kTileW, ty0 = y0 + (warp / kBlockTilesX) * kTileH;
	const bool wholeTile = tx0 + kTileW <= a.W && ty0 + kTileH <= a.yEnd && a.rowWordsOk;
	if (wholeTile)
	{
		uint32_t (*mine)[kTileW * 3 / 4] = reinterpret_cast<uint32_t (*)[kTileW * 3 / 4]>(&staged[0][0]) + warp * kTileH;
		uint8_t* sb = reinterpret_cast<uint8_t*>(&mine[lane / kTileW][0]) + (lane & (kTileW - 1)) * 3;
		sb[0] = (uint8_t)(color >> 16); sb[1] = (uint8_t)((color >> 8) & 0xFF); sb[2] = (uint8_t)(color & 0xFF);
		__syncwarp();
		if (lane < kTileH * (kTileW * 3 / 4))
		{
			const uint32_t row = lane / (kTileW * 3 / 4), w = lane % (kTileW * 3 / 4);
			uint32_t* dst = reinterpret_cast<uint32_t*>(a.rgb + ((size_t)blockIdx.z * a.rgbViewPixels + (size_t)(ty0 + row) * a.W + tx0) * 3);
			dst[w] = mine[row][w];
		}
	}
	else if (inside)
	{
		const size_t p = pixelOut;
		a.rgb[3 * p] = (uint8_t)(color >> 16);
		a.rgb[3 * p + 1] = (uint8_t)((color >> 8) & 0xFF);
		a.rgb[3 * p + 2] = (uint8_t)(color & 0xFF);
	}
	}
	else
	{
	const bool wholeBlock = x0 + kBlockW <= a.W && y0 + kBlockH <= a.yEnd && a.rowWordsOk;
	if (wholeBlock)
	{
		uint8_t* sb = reinterpret_cast<uint8_t*>(&staged[ly][0]) + lx * 3;
		sb[0] = (uint8_t)(color >> 16); sb[1] = (uint8_t)((color >> 8) & 0xFF); sb[2] = (uint8_t)(color & 0xFF);
		if (a.rowBulkOk)
		{
			// remote frame: one bulk async copy per 96-byte row segment, issued by the first kBlockH threads
			asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
			__syncthreads();
			if (threadIdx.x < kBlockH)
			{
				bulk_store_row(a.rgb + ((size_t)blockIdx.z * a.rgbViewPixels + (size_t)(y0 + threadIdx.x) * a.W + x0) * 3, &staged[threadIdx.x][0], kBlockW * 3);
				bulk_store_commit_and_release();
			}
		}
		else
		{
		__syncthreads();
		if (threadIdx.x < kBlockH * (kBlockW * 3 / 4))
		{
			const uint32_t row = threadIdx.x / (kBlockW * 3 / 4), w = threadIdx.x % (kBlockW * 3 / 4);
			uint32_t* dst = reinterpret_cast<uint32_t*>(a.rgb + ((size_t)blockIdx.z * a.rgbViewPixels + (size_t)(y0 + row) * a.W + x0) * 3);
			dst[w] = staged[row][w];
		}
		}
	}
	else if (inside)
	{
		const size_t p = pixelOut;
		a.rgb[3 * p] = (uint8_t)(color >> 16);
		a.rgb[3 * p + 1] = (uint8_t)((color >> 8) & 0xFF);
		a.rgb[3 * p + 2] = (uint8_t)(color & 0xFF);
	}
	}
	flush_stats<STATS>(c, a.stats);
}

// The queued shadow rays: a persistent grid, every warp claims 32 consecutive records at a time.
#ifndef VRM_SHADOW_MINBLOCKS
#define VRM_SHADOW_MINBLOCKS 4
#endif
constexpr int kShadowThreads = 128;
template <int ST, int ALGO, bool STATS, bool FLAT>
__global__ void __launch_bounds__(kShadowThreads, (FLAT ? VRM_SHADOW_MINBLOCKS : (ALGO == kAlgoOriginal ? 6 : 5)) * 256 / kShadowThreads) shadow_kernel(const ShadowArgs a)
{
	const unsigned lane = threadIdx.x & 31u;
	const unsigned queued = a.ctl[0];
	const unsigned count = queued < a.cap ? queued : a.cap;
	RayCtx<ST, STATS> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	c.deferQueue = a.defer;
	for (;;)
	{
		unsigned base = 0;
		if (lane == 0) base = atomicAdd(a.ctl + 1, 32u);
		base = __shfl_sync(0xFFFFFFFFu, base, 0);
		if (base >= count) break;
		const unsigned i = base + lane;
		bool active = i < count;
		ShadowStart ss;
		ss.hitW[0] = ss.hitW[1] = ss.hitW[2] = 0.0f; ss.regW[0] = ss.regW[1] = ss.regW[2] = 0; ss.lit = 0u; ss.la = 0;
		uint32_t pixel = 0;
		if (active)
		{
			const int4 v0 = __ldg(a.items + 2 * (size_t)i), v1 = __ldg(a.items + 2 * (size_t)i + 1);
			ss.hitW[0] = __int_as_float(v0.x); ss.hitW[1] = __int_as_float(v0.y); ss.hitW[2] = __int_as_float(v0.z);
			ss.regW[0] = v0.w; ss.regW[1] = v1.x; ss.regW[2] = v1.y;
			pixel = (uint32_t)v1.z;
			ss.lit = (uint32_t)v1.w & 0x7FFFFFFFu;
			ss.la = ((uint32_t)v1.w >> 31) ? 1 : 0;
		}
		uint32_t final = ss.lit;
		if constexpr (FLAT)
		{
			FlatRay<ST, ALGO, STATS> ray;
			march_shadow_flat_warp<ST, ALGO, STATS, kPpDefer>(c, active, ss, ray);
			if (active)
			{
				if (ray.st == kStPark)
				{
					const int slot = ray.park(c);
					if (slot >= 0)  // the resume kernel writes the pixel
					{
						if (a.colour) park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.colour + pixel, 1u);
						else park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.rgb + 3 * (size_t)pixel, 0u);
						final = ss.lit;
					}
					else { while (ray.st < kStDone) ray.template step<kPpOff>(c); final = ray.result; }
				}
				else final = ray.result;
			}
		}
		else
		{
			if (active && shadow_nested<ST, ALGO, STATS>(c, ss)) final = 0u;
		}
		if (active && final != ss.lit)
		{
			// the light is blocked: the shaded colour the render kernel stored becomes black
			if (a.colour) a.colour[pixel] = final;
			else
			{
				uint8_t* px = a.rgb + 3 * (size_t)pixel;
				px[0] = (uint8_t)(final >> 16); px[1] = (uint8_t)((final >> 8) & 0xFF); px[2] = (uint8_t)(final & 0xFF);
			}
		}
	}
	flush_stats<STATS>(c, a.stats);
}

// The same queue walked with LANE-LEVEL REFILL: a lane whose shadow ray has ended takes the next record as soon as enough lanes of its
// warp are free (one atomicAdd per refill), so short (blocked) and long (light reaches the sky) shadow rays no longer make a warp
// wait for its longest one.  Shadow rays share one direction and consecutive records are neighbouring pixels, so the mixture a warp
// holds stays coherent.  The state machine of vrm_flat.cuh for every combination (one micro-step per pass).
#ifndef VRM_SHADOW_REFILL_MIN
#define VRM_SHADOW_REFILL_MIN 8
#endif
template <int ST, int ALGO, bool STATS>
__global__ void __launch_bounds__(kShadowThreads, (ALGO == kAlgoOriginal ? 6 : VRM_SHADOW_MINBLOCKS) * 256 / kShadowThreads) shadow_refill_kernel(const ShadowArgs a)
{
	const unsigned lane = threadIdx.x & 31u;
	const unsigned queued = a.ctl[0];
	const unsigned count = queued < a.cap ? queued : a.cap;
	RayCtx<ST, STATS> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	c.deferQueue = a.defer;
	FlatRay<ST, ALGO, STATS> ray;
	ray.st = kStDone; ray.result = 0u;
	bool have = false, dry = false;  // dry is warp-uniform: the queue has no unclaimed record left
	uint32_t pixel = 0, lit = 0;
	for (;;)
	{
		// a ray that ended in the last pass: its pixel keeps the shaded colour or turns black
		if (have && ray.st >= kStDone)
		{
			uint32_t final = ray.result;
			bool write = true;
			if (ray.st == kStPark)
			{
				const int slot = ray.park(c);
				if (slot >= 0)  // the resume kernel writes the pixel
				{
					if (a.colour) park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.colour + pixel, 1u);
					else park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.rgb + 3 * (size_t)pixel, 0u);
					write = false;
				}
				else { while (ray.st < kStDone) ray.template step<kPpOff>(c); final = ray.result; }
			}
			if (write && final != lit)
			{
				if (a.colour) a.colour[pixel] = final;
				else
				{
					uint8_t* px = a.rgb + 3 * (size_t)pixel;
					px[0] = (uint8_t)(final >> 16); px[1] = (uint8_t)((final >> 8) & 0xFF); px[2] = (uint8_t)(final & 0xFF);
				}
			}
			have = false;
			ray.st = kStDone;
		}
		const unsigned freeMask = __ballot_sync(0xFFFFFFFFu, !have);
		const int nFree = __popc(freeMask);
		if (!dry && (nFree >= VRM_SHADOW_REFILL_MIN || nFree == 32))
		{
			unsigned base = 0;
			const int leader = __ffs(freeMask) - 1;
			if ((int)lane == leader) base = atomicAdd(a.ctl + 1, (unsigned)nFree);
			base = __shfl_sync(0xFFFFFFFFu, base, leader);
			if (base + (unsigned)nFree >= count) dry = true;
			if (!have)
			{
				const unsigned i = base + __popc(freeMask & ((1u << lane) - 1u));
				if (i < count)
				{
					const int4 v0 = __ldg(a.items + 2 * (size_t)i), v1 = __ldg(a.items + 2 * (size_t)i + 1);
					ShadowStart ss;
					ss.hitW[0] = __int_as_float(v0.x); ss.hitW[1] = __int_as_float(v0.y); ss.hitW[2] = __int_as_float(v0.z);
					ss.regW[0] = v0.w; ss.regW[1] = v1.x; ss.regW[2] = v1.y;
					pixel = (uint32_t)v1.z;
					lit = (uint32_t)v1.w & 0x7FFFFFFFu;
					ss.lit = lit;
					ss.la = ((uint32_t)v1.w >> 31) ? 1 : 0;
					ray.start_shadow(c, ss);
					have = true;
				}
			}
		}
		if (!__any_sync(0xFFFFFFFFu, have)) break;  // nothing in flight: the refill above found the queue empty
		warp_march_pass<ST, ALGO, STATS, kPpDefer>(c, ray);
	}
	flush_stats<STATS>(c, a.stats);
}

// ---- persistent-thread ray queue + warp-level state scheduling ------------------------------------------------------
// Pixel slots are numbered tile-major: slot = (view * tilesPerView + tile) * 32 + pixel-in-8x4-tile, so that 32 consecutive
// slots are one warp-coherent tile.  The tiles are those of the launch's band, rows [yBase, yEnd), as in the grid kernels.
// Every lane owns one FlatRay state machine (vrm_flat.cuh).  Per iteration the warp votes (__match_any_sync groups lanes by state, __reduce_min_sync picks the largest group) and runs ONLY that state's
// code block; lanes in other states wait for their turn, lanes whose pixel is resolved vote for a refill, which claims the
// next slots with one warp-aggregated atomicAdd.  Divergent ray lengths and phases therefore cost idle lanes only while a
// state is in the minority, instead of serialising every loop nest as the nested kernels do.
constexpr int kPersistThreads = 128;

template <int ST, int ALGO, bool STATS>
__global__ void __launch_bounds__(kPersistThreads) render_scheduled_kernel(const RenderArgs a)
{
	const unsigned lane = threadIdx.x & 31u;
	const unsigned total = a.nViews * a.tilesPerView * 32u;
	RayCtx<ST, STATS> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	c.skipDead = a.skipDead;
	FlatRay<ST, ALGO, STATS> ray;
	ray.st = kStDone;
	size_t pixel = 0;
	bool exhausted = false;  // warp-uniform: the queue has run dry
	for (;;)
	{
		// the block a lane wants to run: 0 main (any advance mode), 1 region, 2 head, 3 hit, 4 done (5 parked: never, kPpOff)
		constexpr int bMain = 0, bRegion = 1, bHit = 3, bDone = 4;
		const int st = ray.st <= kStMainLast ? bMain : ray.st - kStMainLast;
		const bool votes = !(st == bDone && exhausted);
		const int ballotState = votes ? st : 7;
		const unsigned peers = __match_any_sync(0xFFFFFFFFu, ballotState);
		const int key = votes ? (((32 - __popc(peers)) << 3) | st) : ((32 << 3) | 7);
		const int best = __reduce_min_sync(0xFFFFFFFFu, key);
		const int run = best & 7;
		if (run == 7) break;  // every lane is idle and the queue is dry
		if (run == bDone)
		{
			// refill: the idle lanes are the largest group
			const unsigned idleMask = __ballot_sync(0xFFFFFFFFu, st == bDone);
			const int want = __popc(idleMask);
			const int leader = __ffs(idleMask) - 1;
			unsigned base = 0;
			if ((int)lane == leader) base = atomicAdd(a.queue, (unsigned)want);
			base = __shfl_sync(0xFFFFFFFFu, base, leader);
			if (base + want >= total) exhausted = true;
			if (st == bDone)
			{
				const unsigned slot = base + __popc(idleMask & ((1u << lane) - 1u));
				if (slot < total)
				{
					const unsigned tile = slot >> 5, inTile = slot & 31u;
					const unsigned view = tile / a.tilesPerView, t = tile - view * a.tilesPerView;
					const uint32_t x = (t % a.tilesX) * kTileW + (inTile & (kTileW - 1));
					const uint32_t y = a.yBase + (t / a.tilesX) * kTileH + (inTile / kTileW);
					if (x < a.W && y < a.yEnd)
					{
						const float* cam = a.cams + (size_t)view * 15;
						float camv[15];
#pragma unroll
						for (int i = 0; i < 15; i++) camv[i] = __ldg(cam + i);
						float o[3], d[3];
						primary_ray(camv, x, y, a.W, a.H, o, d);
						pixel = (size_t)view * a.viewPixels + (size_t)y * a.W + x;
						if (a.hits)
						{
							c.hitOut = a.hits + 4 * pixel;
							*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
						}
						ray.start_primary(c, o, d, a.scale);
						if (ray.st == kStDone)  // missed the scene's bounding cube altogether
						{
							a.rgb[3 * pixel] = 0; a.rgb[3 * pixel + 1] = 0; a.rgb[3 * pixel + 2] = 0;
						}
					}
				}
			}
			continue;
		}
		if (st == run)
		{
			if (run == bMain) ray.template do_main<false, kPpOff>(c);
			else if (run == bRegion) ray.do_region(c);
			else if (run == bHit) ray.do_hit(c);
			else if constexpr (ALGO != kAlgoOriginal) ray.do_head();
			if (ray.st == kStDone)
			{
				const uint32_t color = ray.result;
				// writeColorToFramebuffer, Renderer.cuh:1024-1031
				a.rgb[3 * pixel] = (uint8_t)(color >> 16);
				a.rgb[3 * pixel + 1] = (uint8_t)((color >> 8) & 0xFF);
				a.rgb[3 * pixel + 2] = (uint8_t)(color & 0xFF);
			}
		}
	}
	flush_stats<STATS>(c, a.stats);
}

struct TraceArgs
{
	SceneView sv;
	Lighting light;
	LightWalk lw;
	float translation[3];
	float scale;
	const float* rays;  // n x 6
	unsigned long long n;
	uint32_t* colour;
	int32_t* hits;
	Stats* stats;
	void* defer;
	uint32_t* parkBits;    // lean kernels: one bit per ray that must be re-traced by resume_lean_trace_kernel
	unsigned int* parkCtl;
	unsigned long long first;  // first ray of this launch (a ray list is traced in launches of at most 2^30 rays: 32-bit queue records)
	int4* shadowItems;     // shadow-ray queue, as in RenderArgs; the record's pixel field is the ray's index minus `first`
	unsigned int* shadowCtl;
	uint32_t shadowCap;
	uint32_t skipDead;
	HorizonView hv;        // shadow horizon map (cells null: none); read by trace_fused_kernel only
	const uint32_t* order; // null: thread t of the launch traces ray first + t; else ray first + order[t] (rays ordered for coherence, below)
};

// ---- ray ordering for trace_rays -----------------------------------------------------------------------------------------------------
// Caller-supplied rays arrive in the caller's order (BASELINE configs[4]: one random direction per pixel): the 32 rays of a warp then
// walk 32 unrelated paths and a warp instruction serves 6 of its 32 lanes (profiles/r02z_ncu_trace_config5_vcs_longestaxis.json).
// Rays are independent, so WHICH thread traces which ray is free: a launch first sorts its ray indices by a 26-bit key -- origin region
// parity (3 bits), cube-map face of the direction (3 bits), Morton code of the two minor direction components over the major one
// (2 x 10 bits) -- with the builder's radix sort (3 passes), and thread t traces ray order[t]: a warp then holds a small patch of
// direction space from one neighbourhood, like a tile of primary rays.  Colours, hit records and shadow-queue records carry the ray's
// own index, so results land where the caller expects them; every ray executes exactly what it always did.
__device__ __forceinline__ uint32_t spread10(uint32_t v)
{
	v &= 0x3FFu;
	v = (v | (v << 8)) & 0x00FF00FFu;
	v = (v | (v << 4)) & 0x0F0F0F0Fu;
	v = (v | (v << 2)) & 0x33333333u;
	v = (v | (v << 1)) & 0x55555555u;
	return v;
}

__global__ void ray_key_kernel(const float* __restrict__ rays, unsigned long long first, uint32_t m, float tx, float ty, float tz, float scale,
                               uint32_t* __restrict__ keys, uint32_t* __restrict__ vals)
{
	const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= m) return;
	const float* r = rays + 6 * (first + t);
	const float o0 = (r[0] - tx) * scale, o1 = (r[1] - ty) * scale, o2 = (r[2] - tz) * scale;
	const float d0 = r[3], d1 = r[4], d2 = r[5];
	const float a0 = fabsf(d0), a1 = fabsf(d1), a2 = fabsf(d2);
	int major = 0;
	float am = a0, u = d1, v = d2, dm = d0;
	if (a1 > am) { major = 1; am = a1; u = d0; v = d2; dm = d1; }
	if (a2 > am) { major = 2; am = a2; u = d0; v = d1; dm = d2; }
	const float inv = am > 0.0f ? 1.0f / am : 0.0f;
	// (a sort key, not traversal arithmetic: any value is a valid key, NaN / inf just land in the clamped corners)
	const uint32_t qu = (uint32_t)fminf(fmaxf((u * inv * 0.5f + 0.5f) * 1023.0f, 0.0f), 1023.0f);
	const uint32_t qv = (uint32_t)fminf(fmaxf((v * inv * 0.5f + 0.5f) * 1023.0f, 0.0f), 1023.0f);
	const uint32_t face = (uint32_t)major * 2u + (dm < 0.0f ? 1u : 0u);
	const uint32_t cell = ((uint32_t)(int)floorf(o0 * 0.015625f) & 1u) | (((uint32_t)(int)floorf(o1 * 0.015625f) & 1u) << 1) | (((uint32_t)(int)floorf(o2 * 0.015625f) & 1u) << 2);
	keys[t] = (cell << 23) | (face << 20) | (spread10(qu) << 1) | spread10(qv);
	vals[t] = t;
}
constexpr int kRayKeyBits = 26;

// Incoherent rays are latency-bound: occupancy is worth more than a few spilled registers (measured, 1024^3 shells, 8.3 M rays:
// VCS + original 9.37 ms at 54 registers / 4 CTAs, 8.82 at 48 / 5, 8.31 at 40 / 6; VCS + longest axis 16.77 at 78 / 3, 14.14 at 64 / 4, 14.50 at 48 / 5).
#ifndef VRM_TRACE_LA_MINBLOCKS
#define VRM_TRACE_LA_MINBLOCKS 4
#endif
#ifndef VRM_TRACE_ORIG_MINBLOCKS
#define VRM_TRACE_ORIG_MINBLOCKS 6
#endif
template <int ST, int ALGO, bool STATS, bool FLATLOOP>
__global__ void __launch_bounds__(256, ALGO == kAlgoOriginal ? VRM_TRACE_ORIG_MINBLOCKS : VRM_TRACE_LA_MINBLOCKS) trace_kernel(const TraceArgs a)
{
	// PRIMARY phase of caller-supplied rays (rayMarchVoxelScene[LongestAxis] called per ray, SURVEY.md 8d-5); a hit is shaded and its
	// shadow ray queued for shadow_kernel, exactly as in render_kernel.  Incoherent rays: every lane runs its own loop.
	const unsigned long long t = a.first + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
	const bool live = t < a.n;
	const unsigned long long i = (live && a.order) ? a.first + __ldg(a.order + (t - a.first)) : t;  // the ray this thread traces
	RayCtx<ST, STATS> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	bool hit = false;
	ShadowStart ss;
	ss.hitW[0] = ss.hitW[1] = ss.hitW[2] = 0.0f; ss.regW[0] = ss.regW[1] = ss.regW[2] = 0; ss.lit = 0u; ss.la = 0;
	if (live)
	{
		const float o[3] = {__ldg(a.rays + 6 * i), __ldg(a.rays + 6 * i + 1), __ldg(a.rays + 6 * i + 2)};
		const float d[3] = {__ldg(a.rays + 6 * i + 3), __ldg(a.rays + 6 * i + 4), __ldg(a.rays + 6 * i + 5)};
		uint32_t colour = 0;
		if constexpr (FLATLOOP)
		{
			if (a.hits)
			{
				c.hitOut = a.hits + 4 * i;
				*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
			}
			c.deferQueue = a.defer;
			FlatRay<ST, ALGO, STATS> ray;
			ray.start_primary(c, o, d, a.scale);
			while (ray.st <= kStHead) ray.template step_marching<kPpDefer>(c);
			if (ray.st == kStHit) { ray.shade_hit(c, ss); hit = true; colour = ss.lit; }
			else if (ray.st == kStPark)
			{
				const int slot = ray.park(c);
				if (slot >= 0) park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.colour + i, 1u);
				else { while (ray.st < kStDone) ray.template step<kPpOff>(c); colour = ray.result; }
			}
			else colour = ray.result;
		}
		else
		{
			hit = march_scene_primary<ST, ALGO, STATS>(c, o, d, a.scale, ss);
			colour = hit ? ss.lit : 0u;
			if (a.hits) reinterpret_cast<int4*>(a.hits)[i] = make_int4(c.hit[0], c.hit[1], c.hit[2], c.hit[3]);
		}
		a.colour[i] = colour;
	}
	if (a.shadowItems) shadow_enqueue(a, hit, ss, (uint32_t)(i - a.first));
	flush_stats<STATS>(c, a.stats);
}

// Ordered rays (ray_key_kernel) are coherent like the primary rays of a tile, so VCS + longest axis traces them the way render_kernel
// does: the warp-cooperative state machine with its fast blocks, primary and shadow ray in one kernel behind the hit barrier.
constexpr int kTraceFusedThreads = 128;
template <int ST, int ALGO, bool STATS>
__global__ void __launch_bounds__(kTraceFusedThreads, VRM_FUSED_CTAS > 0 ? VRM_FUSED_CTAS : 8) trace_fused_kernel(const TraceArgs a)
{
	const unsigned long long t = a.first + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
	const bool live = t < a.n;
	const unsigned long long i = (live && a.order) ? a.first + __ldg(a.order + (t - a.first)) : t;
	RayCtx<ST, STATS> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	c.deferQueue = a.defer;
	c.skipDead = a.skipDead;
	c.hv = a.hv;
	float o[3] = {0.0f, 0.0f, 0.0f}, d[3] = {0.0f, 0.0f, 0.0f};
	if (live)
	{
		for (int k = 0; k < 3; k++) { o[k] = __ldg(a.rays + 6 * i + k); d[k] = __ldg(a.rays + 6 * i + 3 + k); }
		if (a.hits)
		{
			c.hitOut = a.hits + 4 * i;
			*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
		}
	}
	int slot;
	const uint32_t colour = march_scene_flat_warp<ST, ALGO, STATS, kPpDefer>(c, live, o, d, a.scale, slot);
	if (live)
	{
		if (slot >= 0) park_output<FlatRay<ST, ALGO, STATS>>(a.defer, slot, a.colour + i, 1u);
		a.colour[i] = colour;
	}
	flush_stats<STATS>(c, a.stats);
}


// ---- lean state machine (vrm_lean.cuh) ------------------------------------------------------------------------------------------
// Same tile mapping and staged stores as render_kernel; per-ray constants in shared memory ([vector][thread]); rays that need a
// slow path flag themselves in a bitmap and are re-traced by resume_lean_kernel.
#ifndef VRM_LEAN_MINBLOCKS
#define VRM_LEAN_MINBLOCKS 4
#endif
__device__ __forceinline__ void park_ray(uint32_t* bits, unsigned int* ctl, unsigned long long rayIndex)
{
	atomicOr(bits + (rayIndex >> 5), 1u << (unsigned)(rayIndex & 31ull));
	atomicAdd(ctl, 1u);
}

template <int ST, int ALGO>
__global__ void __launch_bounds__(kRenderThreads, VRM_LEAN_MINBLOCKS * 8 / (VRM_BLOCK_TILES_Y * VRM_BLOCK_TILES_X)) render_lean_kernel(const RenderArgs a)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t lx = (warp % kBlockTilesX) * kTileW + (lane & (kTileW - 1)), ly = (warp / kBlockTilesX) * kTileH + (lane / kTileW);
	const uint32_t x0 = blockIdx.x * kBlockW, y0 = a.yBase + blockIdx.y * kBlockH;
	const uint32_t x = x0 + lx, y = y0 + ly;
	const bool inside = x < a.W && y < a.yEnd;
	__shared__ uint32_t staged[kBlockH][kBlockW * 3 / 4];
	__shared__ Vec4 consts[kKcVectors][kRenderThreads];
	Vec4* kc = &consts[0][threadIdx.x];
	RayCtx<ST, false> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	float o[3] = {0.0f, 0.0f, 0.0f}, d[3] = {0.0f, 0.0f, 0.0f};
	if (inside)
	{
		const float* cam = a.cams + (size_t)blockIdx.z * 15;
		float camv[15];
#pragma unroll
		for (int i = 0; i < 15; i++) camv[i] = __ldg(cam + i);
		primary_ray_flat(camv, x, y, a.W, a.H, a.invW, a.invH, o, d);
		if (a.hits)
		{
			c.hitOut = a.hits + 4 * ((size_t)blockIdx.z * a.viewPixels + (size_t)y * a.W + x);
			*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
		}
	}
	LeanRay<ST, ALGO, false, kRenderThreads> ray;
	const bool finished = march_scene_lean_warp<ST, ALGO, false, kRenderThreads>(c, kc, inside, o, d, a.scale, ray);
	if (!finished) park_ray(a.parkBits, a.parkCtl, ((unsigned long long)blockIdx.z * a.H + y) * a.W + x);
	const uint32_t color = ray.result;
	// writeColorToFramebuffer, Renderer.cuh:1024-1031 (red = colour >> 16, unmasked, then narrowed to a byte)
	const bool wholeBlock = x0 + kBlockW <= a.W && y0 + kBlockH <= a.yEnd && a.rowWordsOk;
	if (wholeBlock)
	{
		uint8_t* sb = reinterpret_cast<uint8_t*>(&staged[ly][0]) + lx * 3;
		sb[0] = (uint8_t)(color >> 16); sb[1] = (uint8_t)((color >> 8) & 0xFF); sb[2] = (uint8_t)(color & 0xFF);
		__syncthreads();
		if (threadIdx.x < kBlockH * (kBlockW * 3 / 4))
		{
			const uint32_t row = threadIdx.x / (kBlockW * 3 / 4), w = threadIdx.x % (kBlockW * 3 / 4);
			uint32_t* dst = reinterpret_cast<uint32_t*>(a.rgb + ((size_t)blockIdx.z * a.viewPixels + (size_t)(y0 + row) * a.W + x0) * 3);
			dst[w] = staged[row][w];
		}
	}
	else if (inside)
	{
		size_t p = (size_t)blockIdx.z * a.viewPixels + (size_t)y * a.W + x;
		a.rgb[3 * p] = (uint8_t)(color >> 16);
		a.rgb[3 * p + 1] = (uint8_t)((color >> 8) & 0xFF);
		a.rgb[3 * p + 2] = (uint8_t)(color & 0xFF);
	}
}

constexpr int kLeanTraceThreads = 128;
template <int ST, int ALGO>
__global__ void __launch_bounds__(kLeanTraceThreads, VRM_LEAN_MINBLOCKS) trace_lean_kernel(const TraceArgs a)
{
	const unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
	__shared__ Vec4 consts[kKcVectors][kLeanTraceThreads];
	Vec4* kc = &consts[0][threadIdx.x];
	if (i >= a.n) return;
	RayCtx<ST, false> c;
	c.sv = a.sv;
	c.light = a.light;
	c.lw = a.lw;
	c.hitOut = nullptr;
	c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
	c.reset();
	const float o[3] = {__ldg(a.rays + 6 * i), __ldg(a.rays + 6 * i + 1), __ldg(a.rays + 6 * i + 2)};
	const float d[3] = {__ldg(a.rays + 6 * i + 3), __ldg(a.rays + 6 * i + 4), __ldg(a.rays + 6 * i + 5)};
	if (a.hits)
	{
		c.hitOut = a.hits + 4 * i;
		*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
	}
	LeanRay<ST, ALGO, false, kLeanTraceThreads> ray;
	const bool finished = march_scene_lean<ST, ALGO, false, kLeanTraceThreads>(c, kc, o, d, a.scale, ray);
	if (!finished) park_ray(a.parkBits, a.parkCtl, i);
	a.colour[i] = ray.result;
}

// The rays the lean kernels flagged, re-traced from their start by the generic state machine (all slow paths, fast-forwards in
// place).  One warp per bitmap word, one lane per bit.  The last block to finish leaves the bitmap counters zero for the next launch
// (every set bit is cleared by the warp that handles it).
constexpr int kResumeLeanThreads = 256;
template <int ST, int ALGO, bool RENDER, class Args>
__global__ void __launch_bounds__(kResumeLeanThreads) resume_lean_kernel(const Args a, unsigned long long totalRays)
{
	__shared__ unsigned int parked;
	if (threadIdx.x == 0) parked = *reinterpret_cast<volatile unsigned int*>(a.parkCtl);
	__syncthreads();
	if (parked != 0u)
	{
		const unsigned lane = threadIdx.x & 31u;
		const unsigned long long words = (totalRays + 31ull) >> 5;
		const unsigned long long warpsTotal = (unsigned long long)gridDim.x * (kResumeLeanThreads / 32);
		RayCtx<ST, false> c;
		c.sv = a.sv;
		c.light = a.light;
		c.lw = a.lw;
		c.translation[0] = a.translation[0]; c.translation[1] = a.translation[1]; c.translation[2] = a.translation[2];
		for (unsigned long long w = (unsigned long long)blockIdx.x * (kResumeLeanThreads / 32) + (threadIdx.x >> 5); w < words; w += warpsTotal)
		{
			const uint32_t bits = a.parkBits[w];
			if (bits == 0u) continue;
			__syncwarp();
			if (lane == 0) a.parkBits[w] = 0u;
			if (!((bits >> lane) & 1u)) continue;
			const unsigned long long idx = (w << 5) | lane;
			c.reset();
			c.hitOut = nullptr;
			float o[3], d[3];
			uint32_t colour;
			int unused;
			if constexpr (RENDER)
			{
				const unsigned long long perView = (unsigned long long)a.W * a.H;
				const uint32_t view = (uint32_t)(idx / perView);
				const unsigned long long rem = idx - (unsigned long long)view * perView;
				const uint32_t y = (uint32_t)(rem / a.W), x = (uint32_t)(rem - (unsigned long long)y * a.W);
				const size_t p = (size_t)view * a.viewPixels + (size_t)y * a.W + x;
				float camv[15];
				for (int i = 0; i < 15; i++) camv[i] = __ldg(a.cams + (size_t)view * 15 + i);
				primary_ray_flat(camv, x, y, a.W, a.H, a.invW, a.invH, o, d);
				if (a.hits)
				{
					c.hitOut = a.hits + 4 * p;
					*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
				}
				colour = march_scene_flat<ST, ALGO, false, kPpInline>(c, o, d, a.scale, unused);
				a.rgb[3 * p] = (uint8_t)(colour >> 16); a.rgb[3 * p + 1] = (uint8_t)((colour >> 8) & 0xFF); a.rgb[3 * p + 2] = (uint8_t)(colour & 0xFF);
			}
			else
			{
				for (int k = 0; k < 3; k++) { o[k] = __ldg(a.rays + 6 * idx + k); d[k] = __ldg(a.rays + 6 * idx + 3 + k); }
				if (a.hits)
				{
					c.hitOut = a.hits + 4 * idx;
					*reinterpret_cast<int4*>(c.hitOut) = make_int4(0, 0, 0, 0);
				}
				colour = march_scene_flat<ST, ALGO, false, kPpInline>(c, o, d, a.scale, unused);
				a.colour[idx] = colour;
			}
		}
	}
	__syncthreads();
	if (threadIdx.x == 0)
	{
		__threadfence();
		const unsigned int done = atomicAdd(a.parkCtl + 1, 1u);
		if (done == gridDim.x - 1) { a.parkCtl[0] = 0u; a.parkCtl[1] = 0u; }
	}
}

// The storage seam on global voxel coordinates (StorageStructure.cuh:12-17).
template <int ST>
__global__ void lookup_kernel(SceneView sv, const int32_t* __restrict__ xyz, unsigned long long n, uint32_t* __restrict__ out, uint8_t* __restrict__ exists)
{
	unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
	if (i >= n) return;
	RayCtx<ST, false> c;
	c.sv = sv;
	c.reset();
	PermIdentity p;
	int v[3] = {xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]};
	int reg[3] = {v[0] >> 6, v[1] >> 6, v[2] >> 6};   // floor(c / 64), VoxelSceneCPU.cuh:19-21
	int l[3] = {v[0] & 63, v[1] & 63, v[2] & 63};     // VoxelSceneCPU.cuh:24-26
	uint32_t res = kEmpty;
	uint8_t e = 0;
	int32_t ri = region_entry(c, p, reg);
	if (ri >= 0)
	{
		RegionRef<ST> r = load_region<ST>(sv, ri);
		e = space_exists(c, r, p, l[0], l[1], l[2]) ? 1 : 0;
		if (e) res = lookup_voxel(c, r, p, reg, l[0], l[1], l[2]);
	}
	out[i] = res;
	if (exists) exists[i] = e;
}

template <class Args> void fill_common(Args& a, const vrm_scene* s, const float* translation, uint32_t scale)
{
	a.sv = s->view();
	a.light = s->light;
	a.lw = make_light_walk(s->light);  // host, IEEE fp32 without contraction (-fmad=false / -ffp-contract=off): the values the kernel would compute
	a.translation[0] = translation[0]; a.translation[1] = translation[1]; a.translation[2] = translation[2];
	a.scale = static_cast<float>(scale);  // Ray.cuh:16
	a.stats = s->statsEnabled ? s->d_stats : nullptr;
	a.defer = nullptr;
	a.parkBits = nullptr; a.parkCtl = nullptr;
	a.shadowItems = nullptr; a.shadowCtl = nullptr; a.shadowCap = 0; a.skipDead = 0;
	// the horizon map ends lit shadow rays before the reference's walk does: never with reference-comparable event counters
	a.hv = s->horizon;
	if (s->statsMode == 1) a.hv.cells = nullptr;
}

// Shadow-ray queue of the handle: room for `records` records (grow-only), counters zeroed on the stream.
template <class Args> int prepare_shadow_queue(vrm_scene* s, size_t records, Args& a)
{
	a.shadowItems = nullptr; a.shadowCtl = nullptr; a.shadowCap = 0; a.skipDead = 0;
	if (!s->light.useShadows) return VRM_OK;
	if (!s->d_shadowCtl) VRM_CUDA(s, cudaMalloc(&s->d_shadowCtl, 2 * sizeof(unsigned int)));
	if (s->shadowCap < records)
	{
		if (s->d_shadowItems) { VRM_CUDA(s, cudaStreamSynchronize(s->stream)); cudaFree(s->d_shadowItems); s->d_shadowItems = nullptr; s->shadowCap = 0; }
		VRM_CUDA(s, cudaMalloc(&s->d_shadowItems, records * 32));
		s->shadowCap = records;
	}
	VRM_CUDA(s, cudaMemsetAsync(s->d_shadowCtl, 0, 2 * sizeof(unsigned int), s->stream));
	a.shadowItems = static_cast<int4*>(s->d_shadowItems); a.shadowCtl = s->d_shadowCtl; a.shadowCap = (uint32_t)records;
	a.skipDead = s->statsMode == 1 ? 0u : 1u;  // reference-comparable event counters need every shadow ray traced, as the reference does
	return VRM_OK;
}

// form: 0 nested loops / 1 state machine, a warp claims 32 consecutive records at a time; 2 state machine with lane-level refill
template <int ST, int ALGO, class Args> void launch_shadow(vrm_scene* s, const Args& a, uint8_t* rgb, uint32_t* colour, int form)
{
	if (!a.shadowItems) return;
	ShadowArgs b;
	b.sv = a.sv; b.light = a.light; b.lw = a.lw;
	b.translation[0] = a.translation[0]; b.translation[1] = a.translation[1]; b.translation[2] = a.translation[2];
	b.items = a.shadowItems; b.ctl = a.shadowCtl; b.cap = a.shadowCap;
	b.skipDead = a.skipDead;
	b.rgb = rgb; b.colour = colour; b.stats = a.stats; b.defer = a.defer;
	static int blocksPerSm[3][2] = {};  // per instantiation (function template static)
	int& bps = blocksPerSm[form][s->statsEnabled ? 1 : 0];
	const bool st = s->statsEnabled;
	if (bps == 0)
	{
		if (form == 2) { if (st) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, shadow_refill_kernel<ST, ALGO, true>, kShadowThreads, 0); else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, shadow_refill_kernel<ST, ALGO, false>, kShadowThreads, 0); }
		else if (form == 1) { if (st) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, shadow_kernel<ST, ALGO, true, true>, kShadowThreads, 0); else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, shadow_kernel<ST, ALGO, false, true>, kShadowThreads, 0); }
		else { if (st) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, shadow_kernel<ST, ALGO, true, false>, kShadowThreads, 0); else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, shadow_kernel<ST, ALGO, false, false>, kShadowThreads, 0); }
		if (bps < 1) bps = 1;
	}
	const unsigned blocks = (unsigned)(s->numSms * bps);   // one resident wave: a multiple of the SM count
	if (form == 2) { if (st) shadow_refill_kernel<ST, ALGO, true><<<blocks, kShadowThreads, 0, s->stream>>>(b); else shadow_refill_kernel<ST, ALGO, false><<<blocks, kShadowThreads, 0, s->stream>>>(b); }
	else if (form == 1) { if (st) shadow_kernel<ST, ALGO, true, true><<<blocks, kShadowThreads, 0, s->stream>>>(b); else shadow_kernel<ST, ALGO, false, true><<<blocks, kShadowThreads, 0, s->stream>>>(b); }
	else { if (st) shadow_kernel<ST, ALGO, true, false><<<blocks, kShadowThreads, 0, s->stream>>>(b); else shadow_kernel<ST, ALGO, false, false><<<blocks, kShadowThreads, 0, s->stream>>>(b); }
}

constexpr unsigned int kDeferCapacity = 16384;  // parked rays per launch (a 4K frame of the 2048^3 orbit parks a few dozen); VRM_DEFER_CAPACITY overrides (tests)

// The queue exists only for VCS + longest axis (the one combination that can ping-pong): reset its counter before the launch.
template <int ST, int ALGO> void* prepare_defer_queue(vrm_scene* s)
{
	if constexpr (!(ST == kStorageVcs && ALGO != kAlgoOriginal)) return nullptr;
	using Rec = typename FlatRay<ST, ALGO, false>::Deferred;
	static_assert(sizeof(Rec) == sizeof(typename FlatRay<ST, ALGO, true>::Deferred), "one queue layout for both statistics modes");
	if (!s->d_defer)
	{
		unsigned int capacity = kDeferCapacity;
		if (const char* env = getenv("VRM_DEFER_CAPACITY")) { const long v = atol(env); if (v >= 1 && v <= (1l << 20)) capacity = (unsigned int)v; }
		const size_t bytes = sizeof(DeferHeader) + (size_t)capacity * sizeof(Rec);
		if (cudaMalloc(&s->d_defer, bytes) != cudaSuccess) { cudaGetLastError(); s->d_defer = nullptr; return nullptr; }  // no queue: such rays crawl like the reference
		const DeferHeader h = {0u, capacity, {0u, 0u}};
		cudaMemcpyAsync(s->d_defer, &h, sizeof(h), cudaMemcpyHostToDevice, s->stream);
		cudaStreamSynchronize(s->stream);
	}
	return s->d_defer;  // its counter is zero: resume_kernel re-arms it after every launch
}

template <int ST, int ALGO, class Args> void launch_resume(vrm_scene* s, const Args& a)
{
	if constexpr (ST == kStorageVcs && ALGO != kAlgoOriginal)
	{
		if (!a.defer) return;
		ResumeArgs r;
		r.sv = a.sv; r.light = a.light; r.lw = a.lw;
		r.translation[0] = a.translation[0]; r.translation[1] = a.translation[1]; r.translation[2] = a.translation[2];
		r.stats = a.stats; r.defer = a.defer;
		if (s->statsEnabled) resume_kernel<ST, ALGO, true><<<1, kResumeThreads, 0, s->stream>>>(r);
		else resume_kernel<ST, ALGO, false><<<1, kResumeThreads, 0, s->stream>>>(r);
	}
}

// Bitmap + counters of the lean kernels: sized for the launch (grow-only), all-zero between launches (resume_lean_kernel cleans up).
int prepare_park(vrm_scene* s, unsigned long long totalRays, uint32_t** bits, unsigned int** ctl)
{
	const size_t words = (size_t)((totalRays + 31ull) >> 5);
	if (!s->d_parkCtl)
	{
		VRM_CUDA(s, cudaMalloc(&s->d_parkCtl, 2 * sizeof(unsigned int)));
		VRM_CUDA(s, cudaMemsetAsync(s->d_parkCtl, 0, 2 * sizeof(unsigned int), s->stream));
	}
	if (s->parkWords < words)
	{
		if (s->d_parkBits) { VRM_CUDA(s, cudaStreamSynchronize(s->stream)); cudaFree(s->d_parkBits); s->d_parkBits = nullptr; s->parkWords = 0; }
		VRM_CUDA(s, cudaMalloc(&s->d_parkBits, words * 4));
		VRM_CUDA(s, cudaMemsetAsync(s->d_parkBits, 0, words * 4, s->stream));
		s->parkWords = words;
	}
	*bits = s->d_parkBits; *ctl = s->d_parkCtl;
	return VRM_OK;
}

template <int ST, int ALGO> void launch_render_t(vrm_scene* s, RenderArgs a, dim3 grid)
{
	// Which form runs is a measured choice per combination (512^3 terrain, 4K, B200; DESIGN.md 3.2, profiles/r02e_ab.json):
	//   VCS + longest axis: state machine with the shadow ray in the kernel behind a hit barrier (mode 2: 1.50 ms; with the shadow-ray
	//   queue, mode 4: 1.54 ms -- its shadow rays mix head / jump / test phases whichever way they are grouped);
	//   every other combination: nested loops for the primary rays + shadow-ray queue (mode 1: hash table 2.39 / 2.70 ms, VCS +
	//   original 0.89 ms, against 2.94 / 3.09 / 1.04 ms with the shadow ray in the kernel).
	// VRM_RENDER_MODE=0|1|2|3|4 forces one form for A/B runs.
	int mode = s->renderMode >= 0 ? s->renderMode : ((ST == kStorageVcs && ALGO != kAlgoOriginal) ? 2 : 1);
	if (mode == 3 && s->statsEnabled) mode = 2;  // the event counters live in the generic machine
	if (mode == 3)  // lean state machine (vrm_lean.cuh) + re-trace of the rays it parked
	{
		const unsigned long long totalRays = (unsigned long long)a.nViews * a.W * a.H;
		if (prepare_park(s, totalRays, &a.parkBits, &a.parkCtl) != VRM_OK) return;
		render_lean_kernel<ST, ALGO><<<grid, kRenderThreads, 0, s->stream>>>(a);
		resume_lean_kernel<ST, ALGO, true, RenderArgs><<<(unsigned)s->numSms, kResumeLeanThreads, 0, s->stream>>>(a, totalRays);
		return;
	}
	if (mode == 2)  // state machine, both phases in one kernel (hit barrier) + the rays it parked
	{
		a.defer = prepare_defer_queue<ST, ALGO>(s);
		a.skipDead = s->statsMode == 1 ? 0u : 1u;  // as in prepare_shadow_queue
		if (s->statsEnabled) render_kernel<ST, ALGO, true, 2, false><<<grid, kRenderThreads, 0, s->stream>>>(a);
		else if (a.rgbLocal && VRM_WARP_STORE) render_kernel<ST, ALGO, false, 2, true><<<grid, kRenderThreads, 0, s->stream>>>(a);
		else render_kernel<ST, ALGO, false, 2, false><<<grid, kRenderThreads, 0, s->stream>>>(a);
		launch_resume<ST, ALGO>(s, a);
		return;
	}
	if (mode == 1 || mode == 4)
	{
		// primary rays (one CTA per 32x4 pixels; mode 1: nested loops, mode 4: state machine), then the queued shadow rays, then the
		// rays either kernel parked
		if (prepare_shadow_queue(s, (size_t)grid.x * grid.y * grid.z * kRenderThreads, a) != VRM_OK) return;
		if (mode == 1)
		{
			if (s->statsEnabled) render_kernel<ST, ALGO, true, 0, false><<<grid, kRenderThreads, 0, s->stream>>>(a);
			else if (a.rgbLocal && VRM_WARP_STORE_QUEUE) render_kernel<ST, ALGO, false, 0, true><<<grid, kRenderThreads, 0, s->stream>>>(a);
			else render_kernel<ST, ALGO, false, 0, false><<<grid, kRenderThreads, 0, s->stream>>>(a);
			launch_shadow<ST, ALGO>(s, a, a.rgb, nullptr, s->shadowForm >= 0 ? s->shadowForm : 0);
		}
		else
		{
			a.defer = prepare_defer_queue<ST, ALGO>(s);
			if (s->statsEnabled) render_kernel<ST, ALGO, true, 1, false><<<grid, kRenderThreads, 0, s->stream>>>(a);
			else render_kernel<ST, ALGO, false, 1, false><<<grid, kRenderThreads, 0, s->stream>>>(a);
			launch_shadow<ST, ALGO>(s, a, a.rgb, nullptr, s->shadowForm >= 0 ? s->shadowForm : 1);
			launch_resume<ST, ALGO>(s, a);
		}
		return;
	}
	// persistent kernel: as many CTAs as fit on the device at once (a multiple of the SM count)
	static int blocksPerSm[2][2][2] = {};
	int& bps = blocksPerSm[ST][ALGO][s->statsEnabled ? 1 : 0];
	if (bps == 0)
	{
		if (s->statsEnabled) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, render_scheduled_kernel<ST, ALGO, true>, kPersistThreads, 0);
		else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, render_scheduled_kernel<ST, ALGO, false>, kPersistThreads, 0);
		if (bps < 1) bps = 1;
	}
	const unsigned blocks = (unsigned)(s->numSms * bps);
	a.skipDead = s->statsMode == 1 ? 0u : 1u;
	cudaMemsetAsync(s->d_queue, 0, sizeof(unsigned int), s->stream);
	if (s->statsEnabled) render_scheduled_kernel<ST, ALGO, true><<<blocks, kPersistThreads, 0, s->stream>>>(a);
	else render_scheduled_kernel<ST, ALGO, false><<<blocks, kPersistThreads, 0, s->stream>>>(a);
}

template <int ST, int ALGO> void launch_trace_t(vrm_scene* s, TraceArgs a, unsigned grid)
{
	// Arbitrary (incoherent) rays: the per-lane state machine measured faster than the nested loops for every combination
	// (1024^3 sparse shells, 8.3 M random rays: original 11.7 vs 21.1 ms, longest axis 28.4 vs 31.2 ms), so it is the
	// default here; VRM_RENDER_MODE=1 forces the nested form.
	int mode = s->renderMode == 1 ? 1 : (s->renderMode == 3 ? 3 : 2);
	if (mode == 3 && s->statsEnabled) mode = 2;
	if (mode == 3)
	{
		if (prepare_park(s, a.n, &a.parkBits, &a.parkCtl) != VRM_OK) return;
		trace_lean_kernel<ST, ALGO><<<(unsigned)((a.n + kLeanTraceThreads - 1) / kLeanTraceThreads), kLeanTraceThreads, 0, s->stream>>>(a);
		resume_lean_kernel<ST, ALGO, false, TraceArgs><<<(unsigned)s->numSms, kResumeLeanThreads, 0, s->stream>>>(a, a.n);
		return;
	}
	if constexpr (ST == kStorageVcs && ALGO != kAlgoOriginal)
	{
		if (mode == 2 && a.order && s->traceFused)
		{
			a.defer = prepare_defer_queue<ST, ALGO>(s);
			a.skipDead = s->statsMode == 1 ? 0u : 1u;
			const unsigned g = (unsigned)((a.n - a.first + kTraceFusedThreads - 1) / kTraceFusedThreads);
			if (s->statsEnabled) trace_fused_kernel<ST, ALGO, true><<<g, kTraceFusedThreads, 0, s->stream>>>(a);
			else trace_fused_kernel<ST, ALGO, false><<<g, kTraceFusedThreads, 0, s->stream>>>(a);
			launch_resume<ST, ALGO>(s, a);
			return;
		}
	}
	if (prepare_shadow_queue(s, (size_t)grid * 256, a) != VRM_OK) return;
	uint32_t* colour = a.colour + a.first;
	if (mode == 2)
	{
		a.defer = prepare_defer_queue<ST, ALGO>(s);
		if (s->statsEnabled) trace_kernel<ST, ALGO, true, true><<<grid, 256, 0, s->stream>>>(a);
		else trace_kernel<ST, ALGO, false, true><<<grid, 256, 0, s->stream>>>(a);
		launch_shadow<ST, ALGO>(s, a, nullptr, colour, s->shadowForm >= 0 ? s->shadowForm : 2);  // incoherent rays: lane-level refill measured best (config 5: 12.2 vs 13.4 / 14.5 ms)
		launch_resume<ST, ALGO>(s, a);
	}
	else
	{
		if (s->statsEnabled) trace_kernel<ST, ALGO, true, false><<<grid, 256, 0, s->stream>>>(a);
		else trace_kernel<ST, ALGO, false, false><<<grid, 256, 0, s->stream>>>(a);
		launch_shadow<ST, ALGO>(s, a, nullptr, colour, s->shadowForm >= 0 ? s->shadowForm : 0);
	}
}

}  // namespace

int vrm_launch_render(vrm_scene* s, const float* d_cams, uint32_t nViews, const float* translation, uint32_t scale, int algorithm,
                      uint32_t W, uint32_t H, uint8_t* d_rgb, int32_t* d_hits, uint32_t yBase, uint32_t yEnd, uint32_t viewStride, const float* h_cam)
{
	if (yEnd > H) yEnd = H;
	vrm_apply_l2_window(s);
	RenderArgs a;
	fill_common(a, s, translation, scale);
	a.cams = d_cams; a.W = W; a.H = H; a.rgb = d_rgb; a.hits = d_hits;
	a.camInline = 0u;
	for (int i = 0; i < 15; i++) a.cam0[i] = 0.0f;
	if (h_cam && nViews == 1 && vrm_camera_inline_ok(s)) { for (int i = 0; i < 15; i++) a.cam0[i] = h_cam[i]; a.camInline = 1u; }
	else if (!d_cams) { s->lastError = "no camera"; return VRM_ERR_INVALID; }
	a.invW = 1.0f / (float)W; a.invH = 1.0f / (float)H;
	a.viewPixels = (size_t)W * H * (viewStride ? viewStride : 1u);
	a.yBase = yBase; a.yEnd = yEnd;
	a.rowWordsOk = ((W * 3u) % 4u == 0 && (reinterpret_cast<uintptr_t>(d_rgb) & 3u) == 0 && (((size_t)W * H * 3) % 4 == 0 || nViews == 1)) ? 1u : 0u;
	a.queue = s->d_queue;
	a.tilesX = (W + kTileW - 1) / kTileW;
	a.tilesPerView = a.tilesX * ((yEnd - yBase + kTileH - 1) / kTileH);  // the band's tiles (persistent kernel only)
	a.nViews = nViews;
	// 32-bit pixel-slot numbers exist only in the persistent debug kernel (VRM_RENDER_MODE=0); the tiled kernels index with size_t
	if (s->renderMode == 0 && (uint64_t)a.tilesPerView * nViews * 32ull >= (1ull << 32)) { s->lastError = "too many pixels for one launch of the persistent kernel"; return VRM_ERR_INVALID; }
	if (d_hits && (reinterpret_cast<uintptr_t>(d_hits) & 15u)) { s->lastError = "hit buffer must be 16-byte aligned"; return VRM_ERR_INVALID; }
	if (s->statsEnabled && yBase == 0)
	{
		VRM_CUDA(s, cudaMemsetAsync(s->d_stats, 0, sizeof(Stats), s->stream));
		s->statsRays = (uint64_t)W * H * nViews;
	}
	// A launch covers as many views as the shadow-ray queue (one record per pixel, worst case) and 32-bit pixel numbers allow
	const uint64_t threadsPerView = (uint64_t)((W + kBlockW - 1) / kBlockW) * ((yEnd - yBase + kBlockH - 1) / kBlockH) * kRenderThreads;
	constexpr uint64_t kQueueRecords = 32ull << 20;  // 1 GiB of records at most, unless a single view needs more
	if (a.viewPixels >= (1ull << 32)) { s->lastError = "frame too large"; return VRM_ERR_INVALID; }
	uint64_t chunkViews = kQueueRecords / threadsPerView;
	if (chunkViews > ((1ull << 32) - 1) / a.viewPixels) chunkViews = ((1ull << 32) - 1) / a.viewPixels;
	if (chunkViews < 1) chunkViews = 1;
	const bool hash = s->storage == VRM_STORAGE_HASHTABLE, orig = algorithm == VRM_ALGO_ORIGINAL;
	// The shadow-ray queue pipelines (modes 1, 4) touch the frame twice -- the render kernel's coalesced rows, then shadow_kernel's
	// scattered black pixels -- which is fine in local memory but slow through PCIe / NVLink.  A frame that lives in page-locked host
	// memory or on a peer GPU is therefore rendered into a local frame first and sent in one copy behind the kernels.  (The fused form,
	// mode 2, stores every pixel once and writes remote frames directly while it computes.)
	const int mode = s->renderMode >= 0 ? s->renderMode : ((!hash && !orig) ? 2 : 1);
	bool viaLocal = false;
	{
		cudaPointerAttributes at;
		const bool local = cudaPointerGetAttributes(&at, d_rgb) == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device == s->device;
		cudaGetLastError();
		a.rgbLocal = (local || s->wstoreRemote) ? 1u : 0u;
		// frames outside this GPU's memory leave the CTA as bulk async copies when every 96-byte row segment is 16-byte aligned
		a.rowBulkOk = (!local && s->bulkStore && a.rowWordsOk && (kBlockW * 3) % 16 == 0 && ((size_t)W * 3) % 16 == 0 && (reinterpret_cast<uintptr_t>(d_rgb) & 15u) == 0 &&
		               (((size_t)W * H * 3 * (viewStride ? viewStride : 1u)) % 16 == 0 || nViews == 1)) ? 1u : 0u;
		viaLocal = !local && (mode == 1 || mode == 4) && s->light.useShadows;
	}
	const size_t frameBytes = (size_t)W * H * 3;
	if (viaLocal)
	{
		const size_t need = (size_t)(chunkViews < nViews ? chunkViews : nViews) * frameBytes;
		if (s->localFrameBytes < need)
		{
			VRM_CUDA(s, cudaStreamSynchronize(s->stream));
			if (s->d_localFrame) cudaFree(s->d_localFrame);
			s->d_localFrame = nullptr; s->localFrameBytes = 0;
			VRM_CUDA(s, cudaMalloc(&s->d_localFrame, need));
			s->localFrameBytes = need;
		}
	}
	for (uint64_t v0 = 0; v0 < nViews; v0 += chunkViews)
	{
		const uint32_t nv = (uint32_t)(nViews - v0 < chunkViews ? nViews - v0 : chunkViews);
		a.cams = d_cams + v0 * 15;
		a.rgb = d_rgb + v0 * a.viewPixels * 3;
		a.rgbViewPixels = a.viewPixels;
		if (viaLocal)
		{
			a.rgb = s->d_localFrame;
			a.rgbLocal = 1u;
			a.rowBulkOk = 0u;
			a.rgbViewPixels = (size_t)W * H;
			a.rowWordsOk = ((W * 3u) % 4u == 0 && (frameBytes % 4 == 0 || nv == 1)) ? 1u : 0u;
		}
		a.hits = d_hits ? d_hits + v0 * a.viewPixels * 4 : nullptr;
		a.nViews = nv;
		dim3 grid((W + kBlockW - 1) / kBlockW, (yEnd - yBase + kBlockH - 1) / kBlockH, nv);
		if (hash && orig) launch_render_t<kStorageHash, kAlgoOriginal>(s, a, grid);
		else if (hash) launch_render_t<kStorageHash, kAlgoLongestAxis>(s, a, grid);
		else if (orig) launch_render_t<kStorageVcs, kAlgoOriginal>(s, a, grid);
		else launch_render_t<kStorageVcs, kAlgoLongestAxis>(s, a, grid);
		VRM_CUDA(s, cudaGetLastError());
		if (viaLocal)
		{
			const size_t rowBytes = (size_t)W * 3;
			for (uint32_t v = 0; v < nv; v++)
				VRM_CUDA(s, cudaMemcpyAsync(d_rgb + (v0 + v) * a.viewPixels * 3 + yBase * rowBytes, s->d_localFrame + v * frameBytes + yBase * rowBytes,
				                            (size_t)(yEnd - yBase) * rowBytes, cudaMemcpyDefault, s->stream));
		}
	}
	if (yEnd == H) vrm_signal_completion(s, nViews);  // (a band launch signals with the frame's last band)
	return VRM_OK;
}

int vrm_launch_trace(vrm_scene* s, const float* d_rays, uint64_t n, const float* translation, uint32_t scale, int algorithm,
                     uint32_t* d_colour, int32_t* d_hits)
{
	if (n == 0) return VRM_OK;
	if (d_hits && (reinterpret_cast<uintptr_t>(d_hits) & 15u)) { s->lastError = "hit buffer must be 16-byte aligned"; return VRM_ERR_INVALID; }
	vrm_apply_l2_window(s);
	TraceArgs a;
	fill_common(a, s, translation, scale);
	a.rays = d_rays; a.n = n; a.colour = d_colour; a.hits = d_hits; a.order = nullptr;
	if (s->statsEnabled)
	{
		VRM_CUDA(s, cudaMemsetAsync(s->d_stats, 0, sizeof(Stats), s->stream));
		s->statsRays = n;
	}
	const bool hash = s->storage == VRM_STORAGE_HASHTABLE, orig = algorithm == VRM_ALGO_ORIGINAL;
	const uint64_t kChunk = s->renderMode == 3 ? n : (32ull << 20);  // rays per launch: the shadow-ray queue holds one record per ray at most (1 GiB); the lean test kernels take the list whole
	for (uint64_t first = 0; first < n; first += kChunk)
	{
		const uint64_t m = n - first < kChunk ? n - first : kChunk;
		a.first = first;
		const unsigned grid = (unsigned)((m + 255) / 256);
		a.n = first + m;
		// order the launch's rays for coherence (see ray_key_kernel); tiny batches and the lean test kernels take the caller's order
		void* sortBuf = nullptr;
		a.order = nullptr;
		if (s->traceSort && m >= 1024 && s->renderMode != 3)
		{
			const size_t mPad = (size_t)((m + 63) & ~63ull), workElems = vrm_sort_work_elems(m, kRayKeyBits);
			if (vrm_alloc_async(s, &sortBuf, (4 * mPad + workElems) * sizeof(uint32_t)) == cudaSuccess)
			{
				uint32_t* keys = static_cast<uint32_t*>(sortBuf);
				uint32_t* vals = keys + mPad; uint32_t* keysB = vals + mPad; uint32_t* valsB = keysB + mPad; uint32_t* work = valsB + mPad;
				ray_key_kernel<<<grid, 256, 0, s->stream>>>(d_rays, first, (uint32_t)m, translation[0], translation[1], translation[2], static_cast<float>(scale), keys, vals);
				vrm_sort_pairs_u32(keys, vals, keysB, valsB, m, kRayKeyBits, work, s->stream);
				a.order = vals;
			}
			else { cudaGetLastError(); sortBuf = nullptr; }  // no scratch: caller order
		}
		if (hash && orig) launch_trace_t<kStorageHash, kAlgoOriginal>(s, a, grid);
		else if (hash) launch_trace_t<kStorageHash, kAlgoLongestAxis>(s, a, grid);
		else if (orig) launch_trace_t<kStorageVcs, kAlgoOriginal>(s, a, grid);
		else launch_trace_t<kStorageVcs, kAlgoLongestAxis>(s, a, grid);
		if (sortBuf) vrm_free_async(s, sortBuf);
		VRM_CUDA(s, cudaGetLastError());
	}
	return VRM_OK;
}

int vrm_launch_lookup(vrm_scene* s, const int32_t* d_xyz, uint64_t n, uint32_t* d_out, uint8_t* d_exists)
{
	if (n == 0) return VRM_OK;
	unsigned grid = (unsigned)((n + 255) / 256);
	if (s->storage == VRM_STORAGE_HASHTABLE) lookup_kernel<kStorageHash><<<grid, 256, 0, s->stream>>>(s->view(), d_xyz, n, d_out, d_exists);
	else lookup_kernel<kStorageVcs><<<grid, 256, 0, s->stream>>>(s->view(), d_xyz, n, d_out, d_exists);
	VRM_CUDA(s, cudaGetLastError());
	return VRM_OK;
}
