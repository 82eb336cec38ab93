// vrm_internal.h -- state behind the opaque vrm_scene handle (host side).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "vrm_core.cuh"
#include "../../include/vrm_b200.h"

// Small inserts (vrm_scene_insert_voxel, short vrm_scene_add_voxels calls) are collected on the host and reach the device in
// blocks of this many voxels: a caller porting the reference's insertVoxel loop (VoxelSceneCPU.cuh:16-46) pays a vector append per
// voxel, not a device allocation and a stream synchronisation.
constexpr uint64_t kPendingFlushVoxels = 1ull << 20;
constexpr uint64_t kPendingMaxCall = 1ull << 14;  // calls with more voxels than this go to the device directly

struct vrm_scene
{
	int device = 0;
	cudaStream_t ownStream = nullptr;
	cudaStream_t stream = nullptr;
	std::string lastError;

	// staged voxels, in insertion order: ONE growable pair of device arrays (geometric growth, stream-ordered allocation) ...
	int32_t* d_stageXyz = nullptr;   // [stageCap][3]
	uint32_t* d_stageRgb = nullptr;  // [stageCap]
	uint64_t stageCap = 0;
	uint64_t nStaged = 0;            // voxels in the device arrays
	int* d_regionMinMax = nullptr;   // running {min, max} region coordinate of everything staged on the device (VoxelSceneCPU.cuh:28-35)
	// ... behind a host-side block of voxels that have not been copied yet (kPendingFlushVoxels)
	std::vector<int32_t> pendingXyz;
	std::vector<uint32_t> pendingRgb;
	bool stageLost = false;          // a failed build could not restore the staged voxels (vrm_build.cu restage): no more staging or builds

	// built structure
	int storage = -1;
	uint32_t diameter = 0;
	int32_t minCoord = 0;
	uint32_t filled = 0;
	uint64_t unique = 0;
	uint64_t bytes = 0;
	int32_t* d_regionTable = nullptr;
	vrm::HashRegionDesc* d_hashDesc = nullptr;
	unsigned long long* d_slots = nullptr;
	uint2* d_headers = nullptr;
	uint32_t* d_clusterMask = nullptr;
	uint32_t* d_values = nullptr;

	vrm::Lighting light;
	// shadow horizon map of the built scene for `light` (vrm_core.cuh HorizonView; cells null: none): rebuilt by vrm_set_lighting when
	// the direction or use_shadows changes; VRM_SHADOW_HORIZON=0 at vrm_scene_create turns it off (A/B)
	vrm::HorizonView horizon = {};
	int32_t* d_horizon = nullptr;     size_t horizonCap = 0;  // cells allocated
	bool horizonEnabled = true;

	// scratch owned by the handle for the host-buffer entry points
	int32_t* d_hits = nullptr;   size_t hitsBytes = 0;
	float* d_cams = nullptr;     size_t camsBytes = 0;
	float* h_cams = nullptr;     // pinned staging for cameras
	void* d_io = nullptr;        size_t ioBytes = 0;   // rays / lookup queries and results
	cudaEvent_t ev0 = nullptr, ev1 = nullptr;
	// vrm_render into pageable memory: page-locked staging frame written by the kernel in bands, copied out band by band
	uint8_t* h_stage = nullptr;  size_t stageBytes = 0;
	cudaEvent_t evBand[8] = {};
	// streaming multi-view renders into pageable host memory (vrm_render_views): double-buffered device batches
	cudaStream_t copyStream = nullptr;
	cudaEvent_t evRendered[2] = {nullptr, nullptr}, evCopied[2] = {nullptr, nullptr};
	uint8_t* d_batch[2] = {nullptr, nullptr};  size_t batchBytes = 0;
	size_t viewBatchBytes = size_t(256) << 20;  // device bytes per batch buffer (VRM_VIEW_BATCH_BYTES)

	unsigned int* d_queue = nullptr;  // persistent render kernel: next unclaimed pixel slot
	void* d_defer = nullptr;          // rays parked for resume_kernel (vrm_render.cu): DeferHeader + records
	// lean kernels (vrm_lean.cuh): one bit per ray of a launch for rays that need a slow path + {count, blocks done}; the resume kernel
	// re-traces the flagged rays with the generic machine and leaves both all-zero again
	uint32_t* d_parkBits = nullptr;   size_t parkWords = 0;
	unsigned int* d_parkCtl = nullptr;
	int numSms = 148;
	int renderMode = -1;              // -1 = per-combination default (vrm_render.cu); 0 = scheduled persistent kernel, 1 = nested loops, 2 = generic per-lane state machine, 3 = lean state machine (VRM_RENDER_MODE)

	// L2 access-policy window over the structure's hottest array (vrm_set_l2_persistence / VRM_L2_PERSIST=1; off by default:
	// measured no gain on the BASELINE scenes, whose touched working set already lives in L1/L2 -- DESIGN.md 3.2)
	bool l2Persist = false;
	cudaStream_t l2WindowStream = nullptr;  // stream the window is currently installed on
	bool l2WindowOn = false;

	// multi-GPU (vrm_multi.cu): word of the gatherer's memory that receives a sequence number after every render launch, and the
	// root handle's gather buffer of vrm_render_views_sharded
	uint32_t* d_doneFlag = nullptr;
	uint32_t doneSeq = 0;
	uint32_t* d_doneCounter = nullptr;  // counting form: += frames of the launch (dynamically claimed views)
	uint8_t* d_gather = nullptr;      size_t gatherBytes = 0;

	// shadow-ray queue between the render kernels (primary rays) and shadow_kernel (vrm_render.cu): 32-byte records + {queued, claimed}
	void* d_shadowItems = nullptr;    size_t shadowCap = 0;
	unsigned int* d_shadowCtl = nullptr;

	uint8_t* d_dmaFrame = nullptr;    size_t dmaFrameBytes = 0;    // vrm_render into a page-locked buffer, copy-engine form
	int pinnedDma = 0;                // bands of that form (VRM_PINNED_DMA); 0 = the kernels store into the mapped buffer themselves
	int traceSort = 1;                // trace_rays: order the rays by origin cell and direction before tracing (VRM_TRACE_SORT=0: caller order)
	int traceFused = 1;               // ordered rays, VCS + longest axis: warp-cooperative fused kernel instead of primary + shadow-ray queue (VRM_TRACE_FUSED=0)
	bool bulkStore = true;            // frames outside this GPU's memory: CTA-staged rows leave as bulk async copies (cp.async.bulk), VRM_BULK_STORE=0: ordinary stores
	bool wstoreRemote = false;        // A/B: per-warp stores for frames outside this GPU's memory too (VRM_WSTORE_REMOTE)
	uint8_t* d_localFrame = nullptr;  size_t localFrameBytes = 0;  // frames of a queue-pipeline launch whose destination is not local memory
	int shadowForm = -1;              // shadow kernel: -1 per-combination default, 0 nested loops, 1 state machine, 2 state machine with lane-level refill (VRM_SHADOW_FORM)
	int statsMode = 0;                // 0 off, 1 event counters comparable with the reference (every shadow ray traced), 2 counters of the work as executed
	bool statsEnabled = false;
	vrm::Stats* d_stats = nullptr;
	uint64_t statsRays = 0;

	vrm::SceneView view() const
	{
		vrm::SceneView v;
		v.regionTable = d_regionTable; v.diameter = diameter; v.minCoord = minCoord;
		v.hashDesc = d_hashDesc; v.slots = d_slots;
		v.headers = d_headers; v.clusterMask = d_clusterMask; v.values = d_values;
		return v;
	}
};

// status helpers -------------------------------------------------------------------------------------------------
int vrm_fail_cuda(vrm_scene* s, cudaError_t e, const char* what);
#define VRM_CUDA(s, call)                                                   \
	do {                                                                    \
		cudaError_t e__ = (call);                                           \
		if (e__ != cudaSuccess) return vrm_fail_cuda((s), e__, #call);      \
	} while (0)

// The staging calls and vrm_scene_build are legal only before a build and while the staged voxels exist.
inline int vrm_check_staging(vrm_scene* s)
{
	if (s->storage >= 0) { s->lastError = "scene already built"; return VRM_ERR_STATE; }
	if (s->stageLost) { s->lastError = "the staged voxels were lost when a build failed; create a new scene"; return VRM_ERR_STATE; }
	return VRM_OK;
}

// vrm_build.cu
int vrm_build_structure(vrm_scene* s, int storageType, float* buildMs);
void vrm_free_structure(vrm_scene* s);
int vrm_build_horizon(vrm_scene* s);  // (re)build s->horizon for s->light on s->stream, or drop it when the light gets none
// Staging (vrm_build.cu).  vrm_stage_reserve: flush the host block, make room for `extra` more voxels and return where they go;
// the caller fills them on s->stream (copy or kernel) and then calls vrm_stage_commit, which folds them into the running region
// extent.  Nothing here synchronises the stream.
int vrm_stage_reserve(vrm_scene* s, uint64_t extra, int32_t** d_xyz, uint32_t** d_rgb);
int vrm_stage_commit(vrm_scene* s, uint64_t n);
int vrm_stage_flush_pending(vrm_scene* s);
void vrm_stage_free(vrm_scene* s);
// stream-ordered allocation from the device's default memory pool (release threshold raised so that freed scratch is reused by
// the next build instead of going back to the driver)
cudaError_t vrm_alloc_async(vrm_scene* s, void** p, size_t bytes);
void vrm_free_async(vrm_scene* s, void* p);
void vrm_configure_pool(int device);
size_t vrm_scan_scratch_elems(uint64_t n);  // uint32 elements of scratch an exclusive scan of n elements needs
void vrm_exclusive_scan_u32(const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* scratch, cudaStream_t st);  // out may alias in
// the builder's stable LSD radix sort on (32- or 64-bit key, 32-bit value) pairs (vrm_build.cu)
size_t vrm_sort_work_elems(uint64_t n, int keyBits);
void vrm_sort_pairs_u32(uint32_t*& keys, uint32_t*& vals, uint32_t* keysB, uint32_t* valsB, uint64_t n, int keyBits, uint32_t* work, cudaStream_t st);
void vrm_sort_pairs_u64(unsigned long long*& keys, uint32_t*& vals, unsigned long long* keysB, uint32_t* valsB, uint64_t n, int keyBits, uint32_t* work,
                        cudaStream_t st);

// vrm_api.cu: install / remove the access-policy window on the handle's current stream (called by the launch wrappers)
void vrm_apply_l2_window(vrm_scene* s);
// vrm_api.cu: grow one of the handle's device buffers (*p, *have bytes) to at least `need` bytes (contents not kept), and stage
// nViews cameras through the pinned buffer into s->d_cams on the handle's stream
int vrm_ensure(vrm_scene* s, void** p, size_t* have, size_t need);
int vrm_upload_cameras(vrm_scene* s, const float* cameras, uint32_t nViews);

// vrm_multi.cu: publish the handle's next completion sequence number behind the launches already on its stream (no-op without a flag)
void vrm_signal_completion(vrm_scene* s, uint32_t frames);

// vrm_render.cu
int vrm_launch_render(vrm_scene* s, const float* d_cams, uint32_t nViews, const float* translation, uint32_t scale, int algorithm,
                      uint32_t W, uint32_t H, uint8_t* d_rgb, int32_t* d_hits, uint32_t yBase = 0, uint32_t yEnd = 0xFFFFFFFFu, uint32_t viewStride = 1, const float* h_cam = nullptr);
// A single-view launch of the tiled render kernels takes its camera (host pointer h_cam) in the kernel arguments: d_cams may then be null and
// nothing needs to be uploaded.  The debug forms VRM_RENDER_MODE=0 / 3 read d_cams only.
inline bool vrm_camera_inline_ok(const vrm_scene* s) { return s->renderMode != 0 && s->renderMode != 3; }
int vrm_launch_trace(vrm_scene* s, const float* d_rays, uint64_t n, const float* translation, uint32_t scale, int algorithm,
                     uint32_t* d_colour, int32_t* d_hits);
int vrm_launch_lookup(vrm_scene* s, const int32_t* d_xyz, uint64_t n, uint32_t* d_out, uint8_t* d_exists);
