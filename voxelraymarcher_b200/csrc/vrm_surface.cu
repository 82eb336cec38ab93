// vrm_surface.cu -- depth and face maps of reported hits (include/vrm_b200.h, "hit surfaces"; DESIGN.md §3.6).
//
// A streaming pass over a hit map the render / trace kernels already wrote, so that no traversal kernel changes.  Each thread takes
// kPer consecutive records (128-bit ld.global.nc loads), rebuilds the ray only where the flag is set (primary_ray for a pixel, the
// caller's 24-byte ray for a trace) and evaluates vrm_core.cuh hit_surface, the one definition the CPU tests also compile.  Depth leaves
// as one 16-byte store and the faces as one packed 4-byte store per thread when the outputs are aligned for it, else element by element.
#include "vrm_internal.h"
#include "../../include/vrm_b200.h"

using namespace vrm;

namespace
{

constexpr int kThreads = 256;
constexpr int kPer = 4;                          // records per thread
constexpr uint64_t kMaxRecords = 1ull << 40;     // 16 TiB of hit records: far beyond any device, keeps the index arithmetic in 64 bits

struct SurfaceArgs
{
	const int4* hits;                // n records {x, y, z, flag}
	const float* rays;               // trace: n x 6 floats (origin, direction); views: null
	const float* cams;               // views: n_views x 15 floats in device memory; null when `cam` holds the only view
	float cam[VRM_CAMERA_FLOATS];
	float tr[3];
	float scale;
	uint32_t W, H;
	uint64_t n;                      // records of the launch (views: n_views * H * W, view-major)
	float* depth;                    // nullable
	uint8_t* face;                   // nullable
	bool depthVec, faceVec;          // depth 16-byte aligned / face 4-byte aligned: one vector store per thread
};

template <bool VIEWS>
__global__ void __launch_bounds__(kThreads) hit_surface_kernel(const __grid_constant__ SurfaceArgs a)
{
	const uint64_t i0 = (blockIdx.x * (uint64_t)kThreads + threadIdx.x) * kPer;
	if (i0 >= a.n) return;
	const int m = a.n - i0 < (uint64_t)kPer ? (int)(a.n - i0) : kPer;
	int4 h[kPer];
#pragma unroll
	for (int k = 0; k < kPer; k++) h[k] = k < m ? __ldg(a.hits + i0 + k) : make_int4(0, 0, 0, 0);
	// pixel (x, y) of view v of the first record; the others follow in row-major order
	uint32_t x = 0, y = 0, v = 0;
	if (VIEWS && (h[0].w | h[1].w | h[2].w | h[3].w))
	{
		const uint64_t px = (uint64_t)a.W * a.H;
		v = (uint32_t)(i0 / px);
		const uint64_t p = i0 - (uint64_t)v * px;
		y = (uint32_t)(p / a.W);
		x = (uint32_t)(p - (uint64_t)y * a.W);
	}
	float dep[kPer];
	uint32_t fc[kPer];
#pragma unroll
	for (int k = 0; k < kPer; k++)
	{
		float P[3] = {0.0f, 0.0f, 0.0f}, D[3] = {0.0f, 0.0f, 0.0f}, len = 0.0f;
		if (h[k].w != 0)
		{
			if constexpr (VIEWS)
				primary_ray(a.cams ? a.cams + (size_t)v * VRM_CAMERA_FLOATS : a.cam, x, y, a.W, a.H, P, D, len);
			else
			{
				const float* r = a.rays + 6 * (i0 + k);
				for (int c = 0; c < 3; c++) { P[c] = __ldg(r + c); D[c] = __ldg(r + 3 + c); }
			}
		}
		const int32_t rec[4] = {h[k].x, h[k].y, h[k].z, h[k].w};
		dep[k] = hit_surface(rec, P, D, a.tr, a.scale, len, VIEWS, fc[k]);
		if (VIEWS && ++x == a.W) { x = 0; if (++y == a.H) { y = 0; v++; } }
	}
	if (a.depth)
	{
		if (m == kPer && a.depthVec) *reinterpret_cast<float4*>(a.depth + i0) = make_float4(dep[0], dep[1], dep[2], dep[3]);
		else for (int k = 0; k < m; k++) a.depth[i0 + k] = dep[k];
	}
	if (a.face)
	{
		if (m == kPer && a.faceVec) *reinterpret_cast<uint32_t*>(a.face + i0) = fc[0] | fc[1] << 8 | fc[2] << 16 | fc[3] << 24;
		else for (int k = 0; k < m; k++) a.face[i0 + k] = (uint8_t)fc[k];
	}
}

// One launch over n records on the handle's stream.  Views: d_cams (device) or h_cam (one view, travels in the kernel arguments).
int launch_surface(vrm_scene* s, uint64_t n, const int32_t* d_hits, const float* d_rays, const float* d_cams, const float* h_cam, uint32_t W, uint32_t H,
                   const float* translation, uint32_t scale, float* d_depth, uint8_t* d_face)
{
	SurfaceArgs a = {};
	a.hits = reinterpret_cast<const int4*>(d_hits);
	a.rays = d_rays;
	a.cams = d_cams;
	if (h_cam) for (int i = 0; i < VRM_CAMERA_FLOATS; i++) a.cam[i] = h_cam[i];
	for (int i = 0; i < 3; i++) a.tr[i] = translation[i];
	a.scale = (float)scale;
	a.W = W; a.H = H; a.n = n;
	a.depth = d_depth; a.face = d_face;
	a.depthVec = (reinterpret_cast<uintptr_t>(d_depth) & 15u) == 0;
	a.faceVec = (reinterpret_cast<uintptr_t>(d_face) & 3u) == 0;
	const uint64_t blocks = (n + (uint64_t)kThreads * kPer - 1) / ((uint64_t)kThreads * kPer);  // <= 2^30 (kMaxRecords)
	if (d_rays) hit_surface_kernel<false><<<(unsigned)blocks, kThreads, 0, s->stream>>>(a);
	else hit_surface_kernel<true><<<(unsigned)blocks, kThreads, 0, s->stream>>>(a);
	VRM_CUDA(s, cudaGetLastError());
	return VRM_OK;
}

// Checks shared by the four entry points.  Returns -1 when the call goes on, else the status to return (VRM_OK for zero records).
int check_surface(vrm_scene* s, uint64_t n, const void* hits, const void* src, const float* translation, const float* depth, const uint8_t* face, bool device)
{
	if (!s) return VRM_ERR_INVALID;
	if (!translation) { s->lastError = "hit_surface: translation is NULL"; return VRM_ERR_INVALID; }
	if (!depth && !face) { s->lastError = "hit_surface: depth_out and face_out are both NULL"; return VRM_ERR_INVALID; }
	if (n == 0) return VRM_OK;
	if (!hits || !src) { s->lastError = "hit_surface: hits, rays or cameras is NULL"; return VRM_ERR_INVALID; }
	if (n > kMaxRecords) { s->lastError = "hit_surface: more than 2^40 records"; return VRM_ERR_INVALID; }
	if (device && ((reinterpret_cast<uintptr_t>(hits) & 15u) || (reinterpret_cast<uintptr_t>(depth) & 3u)))
	{ s->lastError = "hit_surface: device hits must be 16-byte aligned and device depth 4-byte aligned"; return VRM_ERR_INVALID; }
	return -1;
}

// records of a view batch, 0 when a factor is 0; kMaxRecords + 1 when the product exceeds kMaxRecords
uint64_t view_records(uint32_t nViews, uint32_t W, uint32_t H)
{
	const uint64_t px = (uint64_t)W * H;
	if (px == 0 || nViews == 0) return 0;
	return px > kMaxRecords / nViews ? kMaxRecords + 1 : px * nViews;
}

int surface_views(vrm_scene* s, const float* cameras, uint32_t nViews, const float* translation, uint32_t scale, uint32_t W, uint32_t H,
                  const int32_t* hits, float* depthOut, uint8_t* faceOut, bool device)
{
	const uint64_t n = view_records(nViews, W, H);
	int rc = check_surface(s, n, hits, cameras, translation, depthOut, faceOut, device);
	if (rc >= 0) return rc;
	VRM_CUDA(s, cudaSetDevice(s->device));
	const int32_t* d_hits = hits;
	float* d_depth = depthOut;
	uint8_t* d_face = faceOut;
	if (!device)
	{
		void* p = s->d_hits;
		rc = vrm_ensure(s, &p, &s->hitsBytes, n * 16);
		s->d_hits = static_cast<int32_t*>(p);
		if (rc) return rc;
		const size_t depthBytes = depthOut ? (n * 4 + 15) & ~size_t(15) : 0;
		rc = vrm_ensure(s, &s->d_io, &s->ioBytes, depthBytes + (faceOut ? n : 0));
		if (rc) return rc;
		d_depth = depthOut ? static_cast<float*>(s->d_io) : nullptr;
		d_face = faceOut ? static_cast<uint8_t*>(s->d_io) + depthBytes : nullptr;
		VRM_CUDA(s, cudaMemcpyAsync(s->d_hits, hits, n * 16, cudaMemcpyHostToDevice, s->stream));
		d_hits = s->d_hits;
	}
	const bool inlineCam = nViews == 1;  // a single view travels in the kernel arguments
	if (!inlineCam) { rc = vrm_upload_cameras(s, cameras, nViews); if (rc) return rc; }
	rc = launch_surface(s, n, d_hits, nullptr, inlineCam ? nullptr : s->d_cams, inlineCam ? cameras : nullptr, W, H, translation, scale, d_depth, d_face);
	if (rc || device) return rc;
	if (depthOut) VRM_CUDA(s, cudaMemcpyAsync(depthOut, d_depth, n * 4, cudaMemcpyDeviceToHost, s->stream));
	if (faceOut) VRM_CUDA(s, cudaMemcpyAsync(faceOut, d_face, n, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	return VRM_OK;
}

int surface_rays(vrm_scene* s, const float* rays, uint64_t n, const float* translation, uint32_t scale, const int32_t* hits, float* depthOut,
                 uint8_t* faceOut, bool device)
{
	int rc = check_surface(s, n, hits, rays, translation, depthOut, faceOut, device);
	if (rc >= 0) return rc;
	if (device && (reinterpret_cast<uintptr_t>(rays) & 3u)) { s->lastError = "hit_surface: device rays must be 4-byte aligned"; return VRM_ERR_INVALID; }
	VRM_CUDA(s, cudaSetDevice(s->device));
	if (device) return launch_surface(s, n, hits, rays, nullptr, nullptr, 0, 0, translation, scale, depthOut, faceOut);
	// [hits 16n][rays 24n][depth 4n][face n]: every part aligned for its loads and stores
	const size_t hitBytes = n * 16, rayBytes = n * 24, depthBytes = depthOut ? n * 4 : 0;
	rc = vrm_ensure(s, &s->d_io, &s->ioBytes, hitBytes + rayBytes + depthBytes + (faceOut ? n : 0));
	if (rc) return rc;
	char* base = static_cast<char*>(s->d_io);
	int32_t* d_hits = reinterpret_cast<int32_t*>(base);
	float* d_rays = reinterpret_cast<float*>(base + hitBytes);
	float* d_depth = depthOut ? reinterpret_cast<float*>(base + hitBytes + rayBytes) : nullptr;
	uint8_t* d_face = faceOut ? reinterpret_cast<uint8_t*>(base + hitBytes + rayBytes + depthBytes) : nullptr;
	VRM_CUDA(s, cudaMemcpyAsync(d_hits, hits, hitBytes, cudaMemcpyHostToDevice, s->stream));
	VRM_CUDA(s, cudaMemcpyAsync(d_rays, rays, rayBytes, cudaMemcpyHostToDevice, s->stream));
	rc = launch_surface(s, n, d_hits, d_rays, nullptr, nullptr, 0, 0, translation, scale, d_depth, d_face);
	if (rc) return rc;
	if (depthOut) VRM_CUDA(s, cudaMemcpyAsync(depthOut, d_depth, n * 4, cudaMemcpyDeviceToHost, s->stream));
	if (faceOut) VRM_CUDA(s, cudaMemcpyAsync(faceOut, d_face, n, cudaMemcpyDeviceToHost, s->stream));
	VRM_CUDA(s, cudaStreamSynchronize(s->stream));
	return VRM_OK;
}

}  // namespace

extern "C" {

int vrm_hit_surface_views(vrm_scene* s, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, uint32_t width,
                          uint32_t height, const int32_t* hits, float* depth_out, uint8_t* face_out)
{
	return surface_views(s, cameras, n_views, translation, scale, width, height, hits, depth_out, face_out, false);
}

int vrm_hit_surface_views_device(vrm_scene* s, const float* cameras, uint32_t n_views, const float translation[3], uint32_t scale, uint32_t width,
                                 uint32_t height, const int32_t* d_hits, float* d_depth_out, uint8_t* d_face_out)
{
	return surface_views(s, cameras, n_views, translation, scale, width, height, d_hits, d_depth_out, d_face_out, true);
}

int vrm_hit_surface_rays(vrm_scene* s, const float* rays, uint64_t n, const float translation[3], uint32_t scale, const int32_t* hits,
                         float* depth_out, uint8_t* face_out)
{
	return surface_rays(s, rays, n, translation, scale, hits, depth_out, face_out, false);
}

int vrm_hit_surface_rays_device(vrm_scene* s, const float* d_rays, uint64_t n, const float translation[3], uint32_t scale, const int32_t* d_hits,
                                float* d_depth_out, uint8_t* d_face_out)
{
	return surface_rays(s, d_rays, n, translation, scale, d_hits, d_depth_out, d_face_out, true);
}

}  // extern "C"
