// vrm_api.cu -- the extern "C" boundary declared in include/vrm_b200.h.
#include "vrm_internal.h"
#include "../../include/vrm_b200.h"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

using namespace vrm;

int vrm_fail_cuda(vrm_scene* s, cudaError_t e, const char* what)
{
	if (s) s->lastError = std::string(what) + ": " + cudaGetErrorString(e);
	cudaGetLastError();  // clear the sticky-less error state
	return e == cudaErrorMemoryAllocation ? VRM_ERR_NOMEM : VRM_ERR_CUDA;
}

// The structure's hottest array gets an L2 access-policy window on the launching stream: VCS -> the cluster headers
// (64 KB per region), hash table -> the slot array (hit ratio scaled to the persisting carve-out when it is larger).
void vrm_apply_l2_window(vrm_scene* s)
{
	const bool want = s->l2Persist && s->storage >= 0;
	if (want == s->l2WindowOn && (!want || s->l2WindowStream == s->stream)) return;
	cudaStreamAttrValue attr;
	memset(&attr, 0, sizeof(attr));
	if (s->l2WindowOn && s->l2WindowStream && s->l2WindowStream != s->stream)
	{
		attr.accessPolicyWindow.num_bytes = 0;  // remove the window from the stream it was on
		cudaStreamSetAttribute(s->l2WindowStream, cudaStreamAttributeAccessPolicyWindow, &attr);
	}
	if (want)
	{
		int maxPersist = 0, maxWindow = 0;
		cudaDeviceGetAttribute(&maxPersist, cudaDevAttrMaxPersistingL2CacheSize, s->device);
		cudaDeviceGetAttribute(&maxWindow, cudaDevAttrMaxAccessPolicyWindowSize, s->device);
		void* base = s->storage == VRM_STORAGE_VCS ? static_cast<void*>(s->d_headers) : static_cast<void*>(s->d_slots);
		size_t bytes = s->storage == VRM_STORAGE_VCS ? (size_t)s->filled * 512 * 16 * sizeof(uint2) : 0;
		if (s->storage == VRM_STORAGE_HASHTABLE) bytes = s->bytes - (size_t)s->filled * (sizeof(vrm::HashRegionDesc) + 64) - (size_t)s->diameter * s->diameter * s->diameter * 4;
		if (base && bytes && maxPersist > 0 && maxWindow > 0)
		{
			const size_t carve = (size_t)maxPersist * 3 / 4;
			cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
			const size_t window = bytes < (size_t)maxWindow ? bytes : (size_t)maxWindow;
			attr.accessPolicyWindow.base_ptr = base;
			attr.accessPolicyWindow.num_bytes = window;
			attr.accessPolicyWindow.hitRatio = window <= carve ? 1.0f : (float)((double)carve / (double)window);
			attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
			attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
			cudaStreamSetAttribute(s->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
		}
	}
	else
	{
		attr.accessPolicyWindow.num_bytes = 0;
		cudaStreamSetAttribute(s->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
		cudaCtxResetPersistingL2Cache();
	}
	cudaGetLastError();
	s->l2WindowOn = want;
	s->l2WindowStream = want ? s->stream : nullptr;
}

int vrm_ensure(vrm_scene* s, void** p, size_t* have, size_t need)
{
	if (*have >= need && *p) return VRM_OK;
	if (*p) { VRM_CUDA(s, cudaStreamSynchronize(s->stream)); cudaFree(*p); *p = nullptr; *have = 0; }
	VRM_CUDA(s, cudaMalloc(p, need));
	*have = need;
	return VRM_OK;
}

namespace
{

int check_render_args(vrm_scene* s, const float* camera, const float* translation, int algorithm, uint32_t W, uint32_t H)
{
	if (!s) return VRM_ERR_INVALID;
	if (s->storage < 0) { s->lastError = "scene not built"; return VRM_ERR_STATE; }
	if (!camera || !translation || W == 0 || H == 0 || (algorithm != VRM_ALGO_ORIGINAL && algorithm != VRM_ALGO_LONGEST_AXIS))
	{ s->lastError = "invalid render arguments"; return VRM_ERR_INVALID; }
	return VRM_OK;
}

}  // namespace

int vrm_upload_cameras(vrm_scene* s, const float* cameras, uint32_t nViews)
{
	size_t bytes = (size_t)nViews * VRM_CAMERA_FLOATS * sizeof(float);
	if (s->camsBytes < bytes || !s->h_cams || !s->d_cams)
	{
		// grow: the new pair is allocated first and swapped in only when both allocations succeeded, so a failure leaves the
		// handle as it was (status return, no half-updated state)
		float* nh = nullptr; float* nd = nullptr;
		if (cudaMallocHost(&nh, bytes) != cudaSuccess) { cudaGetLastError(); s->lastError = "camera staging allocation failed"; return VRM_ERR_NOMEM; }
		cudaError_t e = cudaMalloc(&nd, bytes);
		if (e != cudaSuccess) { cudaFreeHost(nh); return vrm_fail_cuda(s, e, "camera buffer allocation"); }
		e = cudaStreamSynchronize(s->stream);  // the old pair may still be in flight
		if (e != cudaSuccess) { cudaFreeHost(nh); cudaFree(nd); return vrm_fail_cuda(s, e, "cudaStreamSynchronize"); }
		if (s->h_cams) cudaFreeHost(s->h_cams);
		if (s->d_cams) cudaFree(s->d_cams);
		s->h_cams = nh; s->d_cams = nd; s->camsBytes = bytes;
	}
	else
	{
		// the pinned staging buffer may still be in flight from the previous asynchronous call
		VRM_CUDA(s, cudaEventSynchronize(s->ev1));
	}
	memcpy(s->h_cams, cameras, bytes);
	VRM_CUDA(s, cudaMemcpyAsync(s->d_cams, s->h_cams, bytes, cudaMemcpyHostToDevice, s->stream));
	VRM_CUDA(s, cudaEventRecord(s->ev1, s->stream));
	return VRM_OK;
}

extern "C" {

const char* vrm_error_string(int status)
{
	switch (status)
	{
	case VRM_OK: return "ok";
	case VRM_ERR_INVALID: return "invalid argument";
	case VRM_ERR_CUDA: return "CUDA error";
	case VRM_ERR_STATE: return "call not legal in this state";
	case VRM_ERR_NOMEM: return "out of memory";
	case VRM_ERR_BUILD: return "structure construction did not converge";
	default: return "unknown status";
	}
}

const char* vrm_last_error(const vrm_scene* scene) { return scene ? scene->lastError.c_str() : ""; }

int vrm_device_available(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n > 0 ? 1 : 0;
}

int vrm_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n;
}

int vrm_device_name(int device, char* out, uint64_t capacity)
{
	if (!out || capacity == 0) return VRM_ERR_INVALID;
	out[0] = 0;
	cudaDeviceProp prop;
	if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_CUDA; }
	strncpy(out, prop.name, capacity - 1);
	out[capacity - 1] = 0;
	return VRM_OK;
}

int vrm_scene_create(int device, vrm_scene** out)
{
	if (!out) return VRM_ERR_INVALID;
	*out = nullptr;
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return VRM_ERR_CUDA; }  // no CPU fallback
	if (device < 0 || device >= n) return VRM_ERR_INVALID;
	vrm_scene* s = new (std::nothrow) vrm_scene();
	if (!s) return VRM_ERR_NOMEM;
	s->device = device;
	// defaults = main/Main.cu:26-42
	float inv[3] = {1.0f, 1.0f, 1.0f};
	vrm_make_unit_vector(inv, s->light.dir);
	s->light.color[0] = s->light.color[1] = s->light.color[2] = 1.0f;
	s->light.pos[0] = 10.0f; s->light.pos[1] = 10.0f; s->light.pos[2] = -10.0f;
	s->light.usePoint = 0; s->light.useShadows = 1;
	cudaError_t e = cudaSetDevice(device);
	if (e == cudaSuccess) vrm_configure_pool(device);
	if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->ownStream, cudaStreamNonBlocking);
	if (e == cudaSuccess) e = cudaEventCreate(&s->ev0);
	if (e == cudaSuccess) e = cudaEventCreate(&s->ev1);
	if (e == cudaSuccess) e = cudaMalloc(&s->d_stats, sizeof(Stats));
	if (e == cudaSuccess) e = cudaMemset(s->d_stats, 0, sizeof(Stats));
	if (e == cudaSuccess) e = cudaMalloc(&s->d_queue, sizeof(unsigned int));

	if (e == cudaSuccess) e = cudaDeviceGetAttribute(&s->numSms, cudaDevAttrMultiProcessorCount, device);
	if (const char* mode = getenv("VRM_RENDER_MODE")) s->renderMode = atoi(mode);
	if (const char* form = getenv("VRM_SHADOW_FORM")) { const int f = atoi(form); if (f >= 0 && f <= 2) s->shadowForm = f; }
	if (const char* lp = getenv("VRM_L2_PERSIST")) s->l2Persist = atoi(lp) != 0;
	if (const char* ts = getenv("VRM_TRACE_SORT")) s->traceSort = atoi(ts);
	if (const char* tf = getenv("VRM_TRACE_FUSED")) s->traceFused = atoi(tf);
	if (const char* pd = getenv("VRM_PINNED_DMA")) s->pinnedDma = atoi(pd);
	if (const char* ws = getenv("VRM_WSTORE_REMOTE")) s->wstoreRemote = atoi(ws) != 0;
	if (const char* bs = getenv("VRM_BULK_STORE")) s->bulkStore = atoi(bs) != 0;
	if (const char* bb = getenv("VRM_VIEW_BATCH_BYTES")) { long long v = atoll(bb); if (v > 0) s->viewBatchBytes = (size_t)v; }
	if (const char* sh = getenv("VRM_SHADOW_HORIZON")) s->horizonEnabled = atoi(sh) != 0;
	if (e != cudaSuccess) { vrm_scene_destroy(s); cudaGetLastError(); return VRM_ERR_CUDA; }
	s->stream = s->ownStream;
	cudaEventRecord(s->ev1, s->stream);
	*out = s;
	return VRM_OK;
}

int vrm_scene_destroy(vrm_scene* s)
{
	if (!s) return VRM_OK;
	cudaSetDevice(s->device);
	if (s->stream) cudaStreamSynchronize(s->stream);
	vrm_stage_free(s);
	vrm_free_async(s, s->d_regionMinMax); s->d_regionMinMax = nullptr;
	vrm_free_structure(s);
	cudaStreamSynchronize(s->stream);
	cudaFree(s->d_hits); cudaFree(s->d_cams); cudaFree(s->d_io); cudaFree(s->d_stats); cudaFree(s->d_queue); cudaFree(s->d_defer); cudaFree(s->d_parkBits); cudaFree(s->d_parkCtl); cudaFree(s->d_gather); cudaFree(s->d_shadowItems); cudaFree(s->d_shadowCtl); cudaFree(s->d_localFrame); vrm_free_async(s, s->d_horizon); cudaStreamSynchronize(s->stream); if (s->h_stage) cudaFreeHost(s->h_stage); for (auto& e : s->evBand) if (e) cudaEventDestroy(e);
	if (s->h_cams) cudaFreeHost(s->h_cams);
	if (s->ev0) cudaEventDestroy(s->ev0);
	if (s->ev1) cudaEventDestroy(s->ev1);
	if (s->ownStream) cudaStreamDestroy(s->ownStream);
	if (s->copyStream) cudaStreamDestroy(s->copyStream);
	if (s->d_dmaFrame) cudaFree(s->d_dmaFrame);
	for (int i = 0; i < 2; i++)
	{
		if (s->evRendered[i]) cudaEventDestroy(s->evRendered[i]);
		if (s->evCopied[i]) cudaEventDestroy(s->evCopied[i]);
		cudaFree(s->d_batch[i]);
	}

	cudaGetLastError();
	delete s;
	return VRM_OK;
}

int vrm_scene_set_stream(vrm_scene* s, void* cuda_stream)
{
	if (!s) return VRM_ERR_INVALID;
	VRM_CUDA(s, cudaSetDevice(s->device));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	s->stream = static_cast<cudaStream_t>(cuda_stream);
	VRM_CUDA(s, cudaEventRecord(s->ev1, s->stream));
	return VRM_OK;
}

int vrm_scene_reset_stream(vrm_scene* s)
{
	if (!s) return VRM_ERR_INVALID;
	VRM_CUDA(s, cudaSetDevice(s->device));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	s->stream = s->ownStream;
	VRM_CUDA(s, cudaEventRecord(s->ev1, s->stream));
	return VRM_OK;
}

int vrm_scene_synchronize(vrm_scene* s)
{
	if (!s) return VRM_ERR_INVALID;
	VRM_CUDA(s, cudaSetDevice(s->device));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	return VRM_OK;
}

static int add_voxels(vrm_scene* s, const int32_t* xyz, const uint32_t* rgb, uint64_t n, bool fromDevice)
{
	if (!s || (n && (!xyz || !rgb))) return VRM_ERR_INVALID;
	if (int rc = vrm_check_staging(s)) return rc;
	if (n == 0) return VRM_OK;
	if (!fromDevice && n <= kPendingMaxCall)
	{
		// short host calls (down to the reference's one voxel per insertVoxel call) are collected on the host
		try
		{
			s->pendingXyz.insert(s->pendingXyz.end(), xyz, xyz + n * 3);
			s->pendingRgb.insert(s->pendingRgb.end(), rgb, rgb + n);
		}
		catch (...) { s->lastError = "host staging allocation failed"; return VRM_ERR_NOMEM; }
		if (s->pendingRgb.size() < kPendingFlushVoxels) return VRM_OK;
		VRM_CUDA(s, cudaSetDevice(s->device));
		return vrm_stage_flush_pending(s);
	}
	VRM_CUDA(s, cudaSetDevice(s->device));
	int32_t* dx = nullptr; uint32_t* dr = nullptr;
	int rc = vrm_stage_reserve(s, n, &dx, &dr);
	if (rc) return rc;
	const cudaMemcpyKind kind = fromDevice ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	VRM_CUDA(s, cudaMemcpyAsync(dx, xyz, n * 3 * sizeof(int32_t), kind, s->stream));
	VRM_CUDA(s, cudaMemcpyAsync(dr, rgb, n * sizeof(uint32_t), kind, s->stream));
	rc = vrm_stage_commit(s, n);
	if (rc) return rc;
	if (!fromDevice)
	{
		// "The caller may reuse its buffers on return": a copy from pageable memory has been staged by the driver when
		// cudaMemcpyAsync returns; only page-locked sources are read asynchronously and need the wait.
		cudaPointerAttributes at;
		const bool pinned = cudaPointerGetAttributes(&at, xyz) == cudaSuccess && at.type == cudaMemoryTypeHost;
		cudaGetLastError();
		cudaPointerAttributes at2;
		const bool pinned2 = cudaPointerGetAttributes(&at2, rgb) == cudaSuccess && at2.type == cudaMemoryTypeHost;
		cudaGetLastError();
		if (pinned || pinned2) VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	}
	return VRM_OK;
}

int vrm_scene_add_voxels(vrm_scene* s, const int32_t* xyz, const uint32_t* rgb, uint64_t n) { return add_voxels(s, xyz, rgb, n, false); }
int vrm_scene_add_voxels_device(vrm_scene* s, const int32_t* xyz, const uint32_t* rgb, uint64_t n) { return add_voxels(s, xyz, rgb, n, true); }

int vrm_scene_insert_voxel(vrm_scene* s, int32_t x, int32_t y, int32_t z, uint32_t rgb)
{
	const int32_t xyz[3] = {x, y, z};
	return add_voxels(s, xyz, &rgb, 1, false);
}

int vrm_scene_build(vrm_scene* s, int storage_type, float* build_ms)
{
	if (!s || (storage_type != VRM_STORAGE_VCS && storage_type != VRM_STORAGE_HASHTABLE)) return VRM_ERR_INVALID;
	if (int rc = vrm_check_staging(s)) return rc;
	VRM_CUDA(s, cudaSetDevice(s->device));
	int rc = vrm_build_structure(s, storage_type, build_ms);
	if (rc == VRM_OK)
	{
		// the staged copies are no longer needed (the colour array may have moved into the structure: vrm_build.cu)
		vrm_stage_free(s);
		s->nStaged = 0;
	}
	return rc;
}

int vrm_scene_info(const vrm_scene* s, uint32_t* diameter, int32_t* min_coord, uint32_t* filled, uint64_t* unique_voxels, uint64_t* bytes)
{
	if (!s) return VRM_ERR_INVALID;
	if (s->storage < 0) return VRM_ERR_STATE;
	if (diameter) *diameter = s->diameter;
	if (min_coord) *min_coord = s->minCoord;
	if (filled) *filled = s->filled;
	if (unique_voxels) *unique_voxels = s->unique;
	if (bytes) *bytes = s->bytes;
	return VRM_OK;
}

int vrm_set_lighting(vrm_scene* s, const float direction[3], const float colour[3], const float position[3], int use_point_light, int use_shadows)
{
	if (!s || !direction || !colour || !position) return VRM_ERR_INVALID;
	const bool newMap = memcmp(s->light.dir, direction, 12) != 0 || (s->light.useShadows != 0) != (use_shadows != 0);
	memcpy(s->light.dir, direction, 12); memcpy(s->light.color, colour, 12); memcpy(s->light.pos, position, 12);
	s->light.usePoint = use_point_light != 0; s->light.useShadows = use_shadows != 0;
	if (newMap && s->storage >= 0)
	{
		// the shadow horizon map belongs to the light direction: rebuilt on the handle's stream, behind the launches that still read the old one
		VRM_CUDA(s, cudaSetDevice(s->device));
		return vrm_build_horizon(s);
	}
	return VRM_OK;
}

int vrm_render_views_device_strided(vrm_scene* s, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, int algorithm,
                                    uint32_t width, uint32_t height, uint8_t* d_rgb_out, int32_t* d_hits_out, uint32_t view_stride)
{
	int rc = check_render_args(s, cameras, translation, algorithm, width, height);
	if (rc) return rc;
	if (!d_rgb_out || n_views == 0 || n_views > 65535 || view_stride == 0) { s->lastError = "invalid render arguments"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	const bool inlineCam = n_views == 1 && vrm_camera_inline_ok(s);  // the camera of a single view travels in the kernel arguments
	if (!inlineCam) { rc = vrm_upload_cameras(s, cameras, n_views); if (rc) return rc; }
	return vrm_launch_render(s, inlineCam ? nullptr : s->d_cams, n_views, translation, scale, algorithm, width, height, d_rgb_out, d_hits_out, 0, 0xFFFFFFFFu, view_stride,
	                         inlineCam ? cameras : nullptr);
}

int vrm_render_views_device(vrm_scene* s, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, int algorithm,
                            uint32_t width, uint32_t height, uint8_t* d_rgb_out, int32_t* d_hits_out)
{
	return vrm_render_views_device_strided(s, cameras, n_views, translation, scale, algorithm, width, height, d_rgb_out, d_hits_out, 1);
}

int vrm_render_device(vrm_scene* s, const float camera[VRM_CAMERA_FLOATS], const float translation[3], uint32_t scale, int algorithm,
                      uint32_t width, uint32_t height, uint8_t* d_rgb_out, int32_t* d_hits_out)
{
	return vrm_render_views_device(s, camera, 1, translation, scale, algorithm, width, height, d_rgb_out, d_hits_out);
}

int vrm_render(vrm_scene* s, const float camera[VRM_CAMERA_FLOATS], const float translation[3], uint32_t scale, int algorithm,
               uint32_t width, uint32_t height, uint8_t* rgb_out, int32_t* hits_out, float* kernel_ms)
{
	int rc = check_render_args(s, camera, translation, algorithm, width, height);
	if (rc) return rc;
	if (!rgb_out) { s->lastError = "rgb_out is NULL"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	const size_t px = (size_t)width * height;
	// Pinned (page-locked) caller buffers are mapped into the device's address space: the kernel then writes the frame
	// straight into them over PCIe (coalesced 96-byte row segments, vrm_render.cu) and no device-to-host copy is needed.
	// Pageable buffers go through the handle's device framebuffer and a copy.
	auto device_alias = [](void* host) -> void* {
		cudaPointerAttributes at;
		if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) return at.devicePointer;
		cudaGetLastError();
		return nullptr;
	};
	uint8_t* d_rgb = static_cast<uint8_t*>(device_alias(rgb_out));
	int32_t* d_hits = hits_out ? static_cast<int32_t*>(device_alias(hits_out)) : nullptr;
	if (d_hits && (reinterpret_cast<uintptr_t>(d_hits) & 15u)) d_hits = nullptr;  // hit records are 16-byte stores: an unaligned page-locked buffer takes the copy path
	const bool stageRgb = d_rgb == nullptr, copyHits = hits_out && d_hits == nullptr;
	void* p;
	if (stageRgb)
	{
		// Pageable frame: the kernel stores into a page-locked staging frame owned by the handle, in horizontal BANDS, and the host
		// copies band k into the caller's memory while band k+1 renders (a cudaMemcpy into pageable memory does the same staging
		// inside the driver, but only after the whole frame has been rendered).
		if (s->stageBytes < px * 3)
		{
			VRM_CUDA(s, cudaStreamSynchronize(s->stream));
			if (s->h_stage) cudaFreeHost(s->h_stage);
			s->h_stage = nullptr; s->stageBytes = 0;
			if (cudaHostAlloc(reinterpret_cast<void**>(&s->h_stage), px * 3, cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); s->lastError = "frame staging allocation failed"; return VRM_ERR_NOMEM; }
			s->stageBytes = px * 3;
		}
		d_rgb = static_cast<uint8_t*>(device_alias(s->h_stage));
		if (!d_rgb) { s->lastError = "page-locked staging frame is not mapped"; return VRM_ERR_CUDA; }
	}
	if (copyHits) { p = s->d_hits; rc = vrm_ensure(s, &p, &s->hitsBytes, px * 16); s->d_hits = static_cast<int32_t*>(p); if (rc) return rc; d_hits = s->d_hits; }
	// Page-locked frame, copy-engine form (s->pinnedDma bands): the kernels render horizontal bands into a frame in device memory (per-warp
	// stores, no PCIe traffic from the SMs) and the copy engine sends band k while band k+1 renders.  Full-line DMA writes instead of
	// 96-byte partial-line stores from the SMs: what keeps the end-to-end rate up when eight GPUs write frames into host memory at once.
	const bool dmaRgb = !stageRgb && s->pinnedDma > 0 && px * 3 >= (size_t(1) << 20);
	uint8_t* h_dst = rgb_out;
	if (dmaRgb)
	{
		if (s->dmaFrameBytes < px * 3)
		{
			VRM_CUDA(s, cudaStreamSynchronize(s->stream));
			if (s->d_dmaFrame) cudaFree(s->d_dmaFrame);
			s->d_dmaFrame = nullptr; s->dmaFrameBytes = 0;
			VRM_CUDA(s, cudaMalloc(reinterpret_cast<void**>(&s->d_dmaFrame), px * 3));
			s->dmaFrameBytes = px * 3;
		}
		if (!s->copyStream) VRM_CUDA(s, cudaStreamCreateWithFlags(&s->copyStream, cudaStreamNonBlocking));
		d_rgb = s->d_dmaFrame;
	}
	const bool inlineCam = vrm_camera_inline_ok(s);  // the camera travels in the kernel arguments: nothing to upload
	if (!inlineCam) { rc = vrm_upload_cameras(s, camera, 1); if (rc) return rc; }
	VRM_CUDA(s, cudaEventRecord(s->ev0, s->stream));
	constexpr int kMaxBands = 8;
	int bands = 1;
	if (stageRgb) { bands = (int)(px * 3 / (size_t(6) << 20)); if (bands < 1) bands = 1; if (bands > 4) bands = 4; }  // >= 6 MB per band, four bands at most (every band is a launch sequence of its own)
	if (dmaRgb) { bands = s->pinnedDma; if (bands > kMaxBands) bands = kMaxBands; while (bands > 1 && px * 3 / bands < (size_t(2) << 20)) bands--; }
	uint32_t bandEnd[kMaxBands];
	for (int b = 0; b < bands; b++) bandEnd[b] = b == bands - 1 ? height : (uint32_t)(((uint64_t)height * (b + 1) / bands + 7) & ~7ull);
	if (stageRgb || dmaRgb) for (int b = 0; b < bands; b++) if (!s->evBand[b]) VRM_CUDA(s, cudaEventCreateWithFlags(&s->evBand[b], cudaEventDisableTiming));
	for (int b = 0; b < bands; b++)
	{
		const uint32_t y0 = b ? bandEnd[b - 1] : 0u, y1 = bandEnd[b] < height ? bandEnd[b] : height;
		if (y1 <= y0) continue;
		rc = vrm_launch_render(s, inlineCam ? nullptr : s->d_cams, 1, translation, scale, algorithm, width, height, d_rgb, d_hits, y0, y1, 1, inlineCam ? camera : nullptr);
		if (rc) return rc;
		if (stageRgb || dmaRgb) VRM_CUDA(s, cudaEventRecord(s->evBand[b], s->stream));
		if (dmaRgb)
		{
			const size_t off = (size_t)y0 * width * 3, bytes = (size_t)(y1 - y0) * width * 3;
			VRM_CUDA(s, cudaStreamWaitEvent(s->copyStream, s->evBand[b], 0));
			VRM_CUDA(s, cudaMemcpyAsync(h_dst + off, s->d_dmaFrame + off, bytes, cudaMemcpyDeviceToHost, s->copyStream));
		}
	}
	VRM_CUDA(s, cudaEventRecord(s->ev1, s->stream));
	if (copyHits) VRM_CUDA(s, cudaMemcpyAsync(hits_out, s->d_hits, px * 16, cudaMemcpyDeviceToHost, s->stream));
	if (stageRgb)
	{
		for (int b = 0; b < bands; b++)
		{
			const uint32_t y0 = b ? bandEnd[b - 1] : 0u, y1 = bandEnd[b] < height ? bandEnd[b] : height;
			if (y1 <= y0) continue;
			VRM_CUDA(s, cudaEventSynchronize(s->evBand[b]));
			memcpy(rgb_out + (size_t)y0 * width * 3, s->h_stage + (size_t)y0 * width * 3, (size_t)(y1 - y0) * width * 3);
		}
	}
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	if (dmaRgb) VRM_CUDA(s, cudaStreamSynchronize(s->copyStream));
	if (kernel_ms) VRM_CUDA(s, cudaEventElapsedTime(kernel_ms, s->ev0, s->ev1));
	return VRM_OK;
}

int vrm_render_views(vrm_scene* s, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, int algorithm,
                     uint32_t width, uint32_t height, uint8_t* rgb_out, float* total_ms)
{
	int rc = check_render_args(s, cameras, translation, algorithm, width, height);
	if (rc) return rc;
	if (!rgb_out || n_views == 0) { s->lastError = "invalid render arguments"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	const size_t frameBytes = (size_t)width * height * 3;
	cudaPointerAttributes at;
	uint8_t* mapped = nullptr;
	if (cudaPointerGetAttributes(&at, rgb_out) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) mapped = static_cast<uint8_t*>(at.devicePointer);
	cudaGetLastError();
	const uint32_t maxViewsPerLaunch = 65535;
	VRM_CUDA(s, cudaEventRecord(s->ev0, s->stream));
	if (mapped)
	{
		// pinned frames: every view is stored straight into the caller's memory by the kernel (as in vrm_render)
		for (uint32_t v0 = 0; v0 < n_views; v0 += maxViewsPerLaunch)
		{
			const uint32_t nv = n_views - v0 < maxViewsPerLaunch ? n_views - v0 : maxViewsPerLaunch;
			rc = vrm_upload_cameras(s, cameras + (size_t)v0 * VRM_CAMERA_FLOATS, nv);
			if (rc) return rc;
			rc = vrm_launch_render(s, s->d_cams, nv, translation, scale, algorithm, width, height, mapped + (size_t)v0 * frameBytes, nullptr);
			if (rc) return rc;
		}
		VRM_CUDA(s, cudaEventRecord(s->ev1, s->stream));
		VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	}
	else
	{
		// pageable frames: batches of views rendered into two device buffers in turn; the device-to-host copy of batch k runs on a
		// second stream while batch k+1 renders
		size_t perBatch = s->viewBatchBytes / frameBytes;
		if (perBatch < 1) perBatch = 1;
		if (perBatch > n_views) perBatch = n_views;
		if (perBatch > maxViewsPerLaunch) perBatch = maxViewsPerLaunch;
		const size_t need = perBatch * frameBytes;
		if (!s->copyStream)
		{
			VRM_CUDA(s, cudaStreamCreateWithFlags(&s->copyStream, cudaStreamNonBlocking));
			for (int i = 0; i < 2; i++)
			{
				VRM_CUDA(s, cudaEventCreateWithFlags(&s->evRendered[i], cudaEventDisableTiming));
				VRM_CUDA(s, cudaEventCreateWithFlags(&s->evCopied[i], cudaEventDisableTiming));
			}
		}
		if (s->batchBytes < need)
		{
			VRM_CUDA(s, cudaStreamSynchronize(s->stream));
			VRM_CUDA(s, cudaStreamSynchronize(s->copyStream));
			for (int i = 0; i < 2; i++) { cudaFree(s->d_batch[i]); s->d_batch[i] = nullptr; }
			s->batchBytes = 0;
			for (int i = 0; i < 2; i++) VRM_CUDA(s, cudaMalloc(&s->d_batch[i], need));
			s->batchBytes = need;
		}
		uint32_t batch = 0;
		for (uint32_t v0 = 0; v0 < n_views; v0 += (uint32_t)perBatch, batch++)
		{
			const int slot = (int)(batch & 1u);
			const uint32_t nv = n_views - v0 < perBatch ? n_views - v0 : (uint32_t)perBatch;
			if (batch >= 2) VRM_CUDA(s, cudaStreamWaitEvent(s->stream, s->evCopied[slot], 0));  // the buffer's previous batch has left the device
			rc = vrm_upload_cameras(s, cameras + (size_t)v0 * VRM_CAMERA_FLOATS, nv);
			if (rc) return rc;
			rc = vrm_launch_render(s, s->d_cams, nv, translation, scale, algorithm, width, height, s->d_batch[slot], nullptr);
			if (rc) return rc;
			VRM_CUDA(s, cudaEventRecord(s->evRendered[slot], s->stream));
			VRM_CUDA(s, cudaStreamWaitEvent(s->copyStream, s->evRendered[slot], 0));
			VRM_CUDA(s, cudaMemcpyAsync(rgb_out + (size_t)v0 * frameBytes, s->d_batch[slot], (size_t)nv * frameBytes, cudaMemcpyDeviceToHost, s->copyStream));
			VRM_CUDA(s, cudaEventRecord(s->evCopied[slot], s->copyStream));
		}
		VRM_CUDA(s, cudaStreamWaitEvent(s->stream, s->evCopied[(batch - 1) & 1u], 0));
		if (batch >= 2) VRM_CUDA(s, cudaStreamWaitEvent(s->stream, s->evCopied[batch & 1u], 0));
		VRM_CUDA(s, cudaEventRecord(s->ev1, s->stream));
		VRM_CUDA(s, cudaStreamSynchronize(s->stream));
		VRM_CUDA(s, cudaStreamSynchronize(s->copyStream));
	}
	if (total_ms) VRM_CUDA(s, cudaEventElapsedTime(total_ms, s->ev0, s->ev1));
	return VRM_OK;
}

int vrm_trace_rays_device(vrm_scene* s, const float* d_rays, uint64_t n, const float translation[3], uint32_t scale, int algorithm,
                          uint32_t* d_colour_out, int32_t* d_hits_out)
{
	if (!s) return VRM_ERR_INVALID;
	if (s->storage < 0) { s->lastError = "scene not built"; return VRM_ERR_STATE; }
	if ((n && (!d_rays || !d_colour_out)) || !translation || (algorithm != VRM_ALGO_ORIGINAL && algorithm != VRM_ALGO_LONGEST_AXIS))
	{ s->lastError = "invalid trace arguments"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	return vrm_launch_trace(s, d_rays, n, translation, scale, algorithm, d_colour_out, d_hits_out);
}

int vrm_trace_rays(vrm_scene* s, const float* rays, uint64_t n, const float translation[3], uint32_t scale, int algorithm,
                   uint32_t* colour_out, int32_t* hits_out, float* kernel_ms)
{
	if (!s) return VRM_ERR_INVALID;
	if (s->storage < 0) { s->lastError = "scene not built"; return VRM_ERR_STATE; }
	if ((n && (!rays || !colour_out)) || !translation || (algorithm != VRM_ALGO_ORIGINAL && algorithm != VRM_ALGO_LONGEST_AXIS))
	{ s->lastError = "invalid trace arguments"; return VRM_ERR_INVALID; }
	if (kernel_ms) *kernel_ms = 0.0f;
	if (n == 0) return VRM_OK;
	VRM_CUDA(s, cudaSetDevice(s->device));
	const size_t rayBytes = n * 24, colBytes = n * 4, hitBytes = hits_out ? n * 16 : 0;
	int rc = vrm_ensure(s, &s->d_io, &s->ioBytes, rayBytes + colBytes + hitBytes);
	if (rc) return rc;
	char* base = static_cast<char*>(s->d_io);
	int32_t* d_hits = hits_out ? reinterpret_cast<int32_t*>(base) : nullptr;  // 16-byte aligned first
	float* d_rays = reinterpret_cast<float*>(base + hitBytes);
	uint32_t* d_col = reinterpret_cast<uint32_t*>(base + hitBytes + rayBytes);
	VRM_CUDA(s, cudaMemcpyAsync(d_rays, rays, rayBytes, cudaMemcpyHostToDevice, s->stream));
	VRM_CUDA(s, cudaEventRecord(s->ev0, s->stream));
	rc = vrm_launch_trace(s, d_rays, n, translation, scale, algorithm, d_col, d_hits);
	if (rc) return rc;
	VRM_CUDA(s, cudaEventRecord(s->ev1, s->stream));
	VRM_CUDA(s, cudaMemcpyAsync(colour_out, d_col, colBytes, cudaMemcpyDeviceToHost, s->stream));
	if (hits_out) VRM_CUDA(s, cudaMemcpyAsync(hits_out, d_hits, hitBytes, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	if (kernel_ms) VRM_CUDA(s, cudaEventElapsedTime(kernel_ms, s->ev0, s->ev1));
	return VRM_OK;
}

int vrm_lookup(vrm_scene* s, const int32_t* xyz, uint64_t n, uint32_t* out, uint8_t* exists_out)
{
	if (!s || (n && (!xyz || !out))) return VRM_ERR_INVALID;
	if (s->storage < 0) { s->lastError = "scene not built"; return VRM_ERR_STATE; }
	if (n == 0) return VRM_OK;
	VRM_CUDA(s, cudaSetDevice(s->device));
	const size_t qBytes = n * 12, oBytes = n * 4, eBytes = n;
	int rc = vrm_ensure(s, &s->d_io, &s->ioBytes, qBytes + oBytes + eBytes);
	if (rc) return rc;
	char* base = static_cast<char*>(s->d_io);
	int32_t* d_q = reinterpret_cast<int32_t*>(base);
	uint32_t* d_o = reinterpret_cast<uint32_t*>(base + qBytes);
	uint8_t* d_e = reinterpret_cast<uint8_t*>(base + qBytes + oBytes);
	VRM_CUDA(s, cudaMemcpyAsync(d_q, xyz, qBytes, cudaMemcpyHostToDevice, s->stream));
	rc = vrm_launch_lookup(s, d_q, n, d_o, d_e);
	if (rc) return rc;
	VRM_CUDA(s, cudaMemcpyAsync(out, d_o, oBytes, cudaMemcpyDeviceToHost, s->stream));
	if (exists_out) VRM_CUDA(s, cudaMemcpyAsync(exists_out, d_e, eBytes, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	return VRM_OK;
}

int vrm_peer_alloc(int device, uint64_t bytes, void** d_ptr_out, unsigned char handle_out[VRM_IPC_HANDLE_BYTES])
{
	static_assert(sizeof(cudaIpcMemHandle_t) == VRM_IPC_HANDLE_BYTES, "CUDA IPC handle size");
	if (!d_ptr_out || !handle_out || bytes == 0) return VRM_ERR_INVALID;
	*d_ptr_out = nullptr;
	if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_CUDA; }
	void* p = nullptr;
	if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_NOMEM; }
	cudaIpcMemHandle_t h;
	if (cudaMemset(p, 0, bytes) != cudaSuccess || cudaIpcGetMemHandle(&h, p) != cudaSuccess) { cudaGetLastError(); cudaFree(p); return VRM_ERR_CUDA; }
	memcpy(handle_out, &h, VRM_IPC_HANDLE_BYTES);
	*d_ptr_out = p;
	return VRM_OK;
}

int vrm_peer_open(int device, const unsigned char handle[VRM_IPC_HANDLE_BYTES], void** d_ptr_out)
{
	if (!d_ptr_out || !handle) return VRM_ERR_INVALID;
	*d_ptr_out = nullptr;
	if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_CUDA; }
	cudaIpcMemHandle_t h;
	memcpy(&h, handle, VRM_IPC_HANDLE_BYTES);
	void* p = nullptr;
	if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_CUDA; }
	*d_ptr_out = p;
	return VRM_OK;
}

int vrm_peer_close(int device, void* d_ptr)
{
	if (!d_ptr) return VRM_OK;
	if (cudaSetDevice(device) != cudaSuccess || cudaIpcCloseMemHandle(d_ptr) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_CUDA; }
	return VRM_OK;
}

int vrm_peer_free(int device, void* d_ptr)
{
	if (!d_ptr) return VRM_OK;
	if (cudaSetDevice(device) != cudaSuccess || cudaFree(d_ptr) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_CUDA; }
	return VRM_OK;
}

int vrm_copy_device(int device, void* d_dst, const void* d_src, uint64_t bytes)
{
	if (!d_dst || !d_src) return VRM_ERR_INVALID;
	if (cudaSetDevice(device) != cudaSuccess || cudaMemcpy(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice) != cudaSuccess) { cudaGetLastError(); return VRM_ERR_CUDA; }
	return VRM_OK;
}

int vrm_set_l2_persistence(vrm_scene* s, int enabled)
{
	if (!s) return VRM_ERR_INVALID;
	VRM_CUDA(s, cudaSetDevice(s->device));
	s->l2Persist = enabled != 0;
	vrm_apply_l2_window(s);
	return VRM_OK;
}

int vrm_set_statistics(vrm_scene* s, int enabled)
{
	if (!s) return VRM_ERR_INVALID;
	s->statsEnabled = enabled != 0;
	s->statsMode = enabled == 2 ? 2 : (enabled ? 1 : 0);
	return VRM_OK;
}

int vrm_get_statistics(vrm_scene* s, uint64_t out[8])
{
	if (!s || !out) return VRM_ERR_INVALID;
	VRM_CUDA(s, cudaSetDevice(s->device));
	Stats h;
	VRM_CUDA(s, cudaMemcpyAsync(&h, s->d_stats, sizeof(Stats), cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	out[0] = h.nExist; out[1] = h.nExistFalse; out[2] = h.nLookup; out[3] = h.nLookupHit; out[4] = h.nProbe2; out[5] = h.nRegionReads;
	out[6] = s->statsRays; out[7] = h.nCrawlSkipped;
	return VRM_OK;
}

}  // extern "C"
